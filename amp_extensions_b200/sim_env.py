"""gym-simenv's learned-dynamics environment, batched and device-resident.

`VecSimEnv` steps E independent environments per call on one GPU (one grouped tensor-core pass over all
ensemble members, fused next-state / discrepancy / termination kernel, optional MILO cost).  `SimEnv`
keeps the reference's single-environment plugin surface (reference
gym-simenv/gym_simenv/envs/sim_env.py:13-288: reset/step/is_done/seed_env, float64 numpy observations,
member round-robin on reset) on top of a 1-row VecSimEnv so existing samplers run unchanged.

Initial states: the reference draws them from DeepMimicCore (sim_env.py:270-285).  That simulator is not
part of this package; pass `reset_fn(n, rng) -> float[n, S]` (or a fixed array `reset_states`), or, when
the reference's `deepmimic` package is importable, `deepmimic_args=...` to get the original behaviour.
"""
import copy
import json

import numpy as np
import torch

from .engine import HumanoidTermination


class VecSimEnv:
    """E learned-dynamics envs on one device.  All arrays are CUDA tensors; nothing syncs unless asked."""

    def __init__(self, dynamic_ensemble, num_envs, termination=None, horizon=300, enable_velocity_check=False,
                 reset_fn=None, reset_states=None, cost=None, seed=None):
        self.dynamic_ensemble = dynamic_ensemble
        self.num_envs = int(num_envs)
        self.state_size = dynamic_ensemble.state_dim
        self.action_size = dynamic_ensemble.action_dim
        self.termination = termination or HumanoidTermination(horizon=horizon,
                                                              enable_velocity_check=enable_velocity_check)
        self.horizon = self.termination.horizon
        self.reset_fn = reset_fn
        self.reset_states = reset_states
        self.rng = np.random.default_rng(seed)
        self.cost = cost
        eng = dynamic_ensemble.engine()
        eng.set_termination(self.termination)
        self.device = eng.device
        E, S = self.num_envs, self.state_size
        self.ob = torch.zeros((E, S), device=self.device, dtype=torch.float32)
        self._ob_next = torch.zeros((E, S), device=self.device, dtype=torch.float32)
        self.num_steps = torch.zeros((E,), device=self.device, dtype=torch.int32)
        # sim_env.py:118-119: the first episode uses member 0, every reset advances round-robin (:282-283)
        self.member = torch.zeros((E,), device=self.device, dtype=torch.int32)
        self.disc = torch.zeros((E,), device=self.device, dtype=torch.float32)
        self.done = torch.zeros((E,), device=self.device, dtype=torch.uint8)
        self.cost_out = torch.zeros((E,), device=self.device, dtype=torch.float32)
        self.ipm_out = torch.zeros((E,), device=self.device, dtype=torch.float32)
        self.bonus_out = torch.zeros((E,), device=self.device, dtype=torch.float32)
        self._w_dev = None
        if cost is not None:
            self.attach_cost(cost)

    # -- cost -------------------------------------------------------------------------------
    def attach_cost(self, cost):
        """Fuse an RBFLinearCost into the step: loads its rff layer into the ensemble's handle."""
        self.cost = cost
        eng = self.dynamic_ensemble.engine()
        eng.load_rff(cost.rff.weight.data, cost.rff.bias.data, split=bool(cost._split), input_type=cost.input_type)
        self.set_cost_weights(cost.w)

    def set_cost_weights(self, w):
        """Device copy of the cost weights, refreshed IN PLACE (captured CUDA graphs keep pointing at it), and the
        cost's current hi/lo decision (RBFLinearCost.fit_cost measures it)."""
        if w is None:
            self._w_dev = None
            return
        w = w.detach().to(self.device, torch.float32).contiguous()
        if self._w_dev is not None and self._w_dev.shape == w.shape:
            self._w_dev.copy_(w)
        else:
            self._w_dev = w.clone()
        eng = self.dynamic_ensemble.engine()
        active = getattr(self.cost, "split_active", None)
        if active is not None and getattr(eng, "rff_split_loaded", False) and eng.rff_split != bool(active):
            eng.set_rff_split(bool(active))

    # -- gym-like surface -------------------------------------------------------------------
    @staticmethod
    def clip_reset_fn(imitation, device=None, reset_args=None, **record_flags):
        """reset_fn that starts envs on the reference motion at t ~ U(0, duration) - or U(time_min, time_max) with
        reset_args['custom_time'] (sim_env.py:76-77) - as SimEnv.reset() does through the simulator (sim_env.py:270-285:
        reset_time(time, **reset_dict) then record_state) — here without the simulator: the clip is sampled on the
        device, the pose / velocity noise of `reset_args` (the plugin's dict, sim_env.py:28-31) is applied there too
        (reset_noise.add_reset_noise = cKinCharacter::AddNoise, KinCharacter.cpp:340-532) and the state features are
        built kinematically (ImitationReward.reset_states).  `resolve` (ground intersection of the simulated character)
        needs the simulator and is not applied."""
        t_lo, t_hi = 0.0, float(imitation.clip.duration)
        if reset_args and reset_args.get("custom_time", False):
            t_lo, t_hi = float(reset_args["time_min"]), float(reset_args["time_max"])
        gen = [None]

        def fn(n, rng):
            t = torch.as_tensor(rng.uniform(t_lo, t_hi, size=n), dtype=torch.float32)
            dev = imitation.engine.device
            if reset_args and gen[0] is None:      # the noise stream is seeded from the env's own generator
                gen[0] = torch.Generator(device=dev)
                gen[0].manual_seed(int(rng.integers(0, 2 ** 31 - 1)) if hasattr(rng, "integers")
                                   else int(rng.randint(0, 2 ** 31 - 1)))
            return imitation.reset_states(t.to(dev), reset_args=reset_args, generator=gen[0], **record_flags)
        return fn

    def _draw_initial(self, n):
        if self.reset_fn is not None:
            s = self.reset_fn(n, self.rng)
        elif self.reset_states is not None:
            pool = self.reset_states
            idx = self.rng.integers(0, pool.shape[0], size=n)
            s = pool[idx] if not torch.is_tensor(pool) else pool[torch.as_tensor(idx, device=pool.device)]
        else:
            raise RuntimeError("VecSimEnv needs reset_fn or reset_states to draw initial states")
        return torch.as_tensor(s).to(self.device, torch.float32)

    def reset(self, mask=None, initial_states=None):
        """Reset all envs (mask None) or those where mask is True.  Advances each reset env's member index."""
        N = self.dynamic_ensemble.num_models
        if mask is None:
            s = initial_states if initial_states is not None else self._draw_initial(self.num_envs)
            self.ob.copy_(torch.as_tensor(s).to(self.device, torch.float32))
            self.num_steps.zero_()
            self.member.add_(1).remainder_(N)
        else:
            mask = torch.as_tensor(mask, device=self.device, dtype=torch.bool)
            idx = mask.nonzero(as_tuple=False).squeeze(1)
            if idx.numel():
                s = initial_states if initial_states is not None else self._draw_initial(int(idx.numel()))
                self.ob[idx] = torch.as_tensor(s).to(self.device, torch.float32)
                self.num_steps[idx] = 0
                self.member[idx] = (self.member[idx] + 1) % N
        return self.ob

    def step(self, actions, with_cost=None):
        """One env step for every env.  Returns (ob, reward, done, info) as CUDA tensors; reward is 0 as in
        sim_env.py:160 unless a cost is attached, in which case reward = -cost (batch_reinforce.py:144)."""
        eng = self.dynamic_ensemble.engine()
        a = torch.as_tensor(actions).to(self.device, torch.float32).contiguous()
        use_cost = (self.cost is not None and self._w_dev is not None) if with_cost is None else with_cost
        if use_cost:
            c = self.cost
            clamp = c.cost_range is not None
            eng.step_cost(self.ob, a, self.member, self.num_steps, self._w_dev, c.lambda_b,
                          self.dynamic_ensemble.threshold if clamp else 1.0, c.c_min if clamp else 0.0,
                          c.c_max if clamp else 0.0, clamp, next_state=self._ob_next, disc=self.disc, done=self.done,
                          cost=self.cost_out, ipm=self.ipm_out, bonus=self.bonus_out)
            reward = -self.cost_out
            info = {"valid": True, "disc": self.disc, "cost": self.cost_out, "ipm": self.ipm_out,
                    "bonus": self.bonus_out}
        else:
            eng.step(self.ob, a, self.member, self.num_steps, next_state=self._ob_next, disc=self.disc,
                     done=self.done)
            reward = torch.zeros((self.num_envs,), device=self.device, dtype=torch.float32)
            info = {"valid": True, "disc": self.disc}
        self.ob, self._ob_next = self._ob_next, self.ob
        return self.ob, reward, self.done, info


class _Box:
    """Minimal stand-in for gym.spaces.Box when gym is not installed."""

    def __init__(self, low, high, dtype):
        self.low, self.high, self.dtype, self.shape = low, high, dtype, low.shape


def _make_box(dim):
    low, high = np.array([-np.inf] * dim), np.array([np.inf] * dim)
    try:  # pragma: no cover - gym is optional
        from gym import spaces
        return spaces.Box(low=low, high=high, dtype=np.float64)
    except Exception:
        return _Box(low, high, np.float64)


def _env_base():
    """gym.Env (or gymnasium.Env) when one of them is importable, so that gym.make / wrappers accept the class;
    a plain object otherwise.  The reference subclasses gym.Env and EzPickle (sim_env.py:13)."""
    for mod in ("gym", "gymnasium"):
        try:  # pragma: no cover - optional dependency
            return __import__(mod).Env
        except Exception:
            continue
    return object


class _SingleStep:
    """SimEnv.step's device side for ONE env: a packed pinned record in (ob | action | step counter | member), the
    step's launches, a packed pinned record out (next state | disc | done) - one host->device copy, one
    device->host copy, one synchronisation, and the three replayed from a CUDA graph."""

    def __init__(self, ensemble, termination, use_graph=True):
        self.eng = eng = ensemble.engine()
        eng.set_termination(termination)
        S, A, dev = eng.S, eng.A, eng.device
        self.S, self.A = S, A
        self.h_in = torch.zeros(S + A + 2, dtype=torch.float32, pin_memory=True)
        self.d_in = torch.zeros(S + A + 2, device=dev, dtype=torch.float32)
        self.h_out = torch.zeros((S + 2) * 4, dtype=torch.uint8, pin_memory=True)
        self.d_out = torch.zeros((S + 2) * 4, device=dev, dtype=torch.uint8)
        self.np_in = self.h_in.numpy()
        self.np_in_i = self.h_in.view(torch.int32).numpy()
        self.np_out_f = self.h_out.view(torch.float32).numpy()
        self.np_out_b = self.h_out.numpy()
        self.v_ob = self.d_in[:S].view(1, S)
        self.v_act = self.d_in[S:S + A].view(1, A)
        ints = self.d_in[S + A:].view(torch.int32)
        self.v_steps, self.v_member = ints[0:1], ints[1:2]
        outf = self.d_out.view(torch.float32)
        self.v_next = outf[:S].view(1, S)
        self.v_disc = outf[S:S + 1]
        self.v_done = self.d_out[(S + 1) * 4:(S + 1) * 4 + 1]
        self.stream = torch.cuda.Stream(dev)
        self.use_graph = use_graph
        self.graph, self.graph_gen = None, -1

    def _enqueue(self):
        self.d_in.copy_(self.h_in, non_blocking=True)
        self.eng.step(self.v_ob, self.v_act, self.v_member, self.v_steps, next_state=self.v_next, disc=self.v_disc,
                      done=self.v_done)
        self.h_out.copy_(self.d_out, non_blocking=True)

    def step(self, ob, action, num_steps, member):
        S, A = self.S, self.A
        self.np_in[:S] = ob
        self.np_in[S:S + A] = action
        self.np_in_i[S + A] = num_steps
        self.np_in_i[S + A + 1] = member
        with torch.cuda.stream(self.stream):
            if self.use_graph and (self.graph is None or self.graph_gen != self.eng.generation):
                self._enqueue()                      # eager once: workspace allocation, kernel attributes
                self.stream.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self.stream):
                    self._enqueue()
                self.graph, self.graph_gen = g, self.eng.generation
            if self.graph is not None:
                self.graph.replay()
            else:
                self._enqueue()
        self.stream.synchronize()
        return (self.np_out_f[:S].astype(np.float64), float(self.np_out_f[S]), bool(self.np_out_b[(S + 1) * 4]))


class SimEnv(_env_base()):
    """Single-environment surface of the reference SimEnv (sim_env.py:13-288), same kwargs."""

    metadata = {"render.modes": ["human"], "render_modes": ["human"]}

    def __init__(self, dynamic_ensemble, deepmimic_args=None, enable_velocity_check=False, horizon=300,
                 device=torch.device("cpu"), seed=None,
                 reset_args={"custom_time": False, "time_min": 0, "time_max": 0, "resolve": True,
                             "noise_bef_rot": False, "noise_min": 0, "noise_max": 0, "radian": 0,
                             "rot_vel_w_pose": False, "vel_noise": False, "interp": False, "knee_rot": False},
                 reset_fn=None, reset_states=None, termination=None):
        self._ctor = dict(dynamic_ensemble=dynamic_ensemble, deepmimic_args=deepmimic_args,
                          enable_velocity_check=enable_velocity_check, horizon=horizon, device=device, seed=seed,
                          reset_args=reset_args, reset_fn=reset_fn, reset_states=reset_states, termination=termination)
        self.dynamic_ensemble = dynamic_ensemble
        self.device = device
        self.enable_velocity_check = enable_velocity_check
        self.horizon = horizon
        self.ob = None
        self.num_steps = 0
        self.agentID = 0
        self.state_size = dynamic_ensemble.state_dim
        self.action_size = dynamic_ensemble.action_dim
        self.observation_space = _make_box(self.state_size)
        self.action_space = _make_box(self.action_size)
        self.deepmimic = None
        self._reset_fn = reset_fn
        self._reset_states = reset_states
        self._termination = termination
        self.reset_dict = None
        self.time_max = 0.0
        if deepmimic_args is not None and reset_fn is None and reset_states is None:
            self._init_deepmimic(deepmimic_args, reset_args)
        self.seed_env(seed)
        self.reset_counter = 0
        self.dynamics = dynamic_ensemble.models[0]
        self.dynamics.model.eval()
        self._vec = None
        self._fast = None

    # The reference builds its termination tables from the DeepMimic arg/character/controller files
    # (sim_env.py:84-116); do the same when they are available.
    def _init_deepmimic(self, deepmimic_args, reset_args):
        from deepmimic.env.deepmimic_env import DeepMimicEnv  # reference simulator, optional
        from deepmimic.util.arg_parser import ArgParser
        self.deepmimic = DeepMimicEnv(["--arg_file", deepmimic_args], False)
        self.deepmimic.set_mode(1)
        self.time_max = reset_args["time_max"] if reset_args["custom_time"] else self.deepmimic.get_motion_length()
        self.reset_dict = dict(time=0, resolve=reset_args["resolve"], noise_bef_rot=reset_args["noise_bef_rot"],
                               low=reset_args["noise_min"], high=reset_args["noise_max"], radian=reset_args["radian"],
                               rot_vel_w_pose=reset_args["rot_vel_w_pose"], vel_noise=reset_args["vel_noise"],
                               interp=reset_args["interp"], knee_rot=reset_args["knee_rot"])
        parser = ArgParser()
        parser.load_file(deepmimic_args)
        with open(parser.parse_string("char_ctrl_files")) as f:
            ctrl = json.load(f)
        with open(parser.parse_string("character_files")) as f:
            char = json.load(f)
        self._termination = HumanoidTermination(
            horizon=self.horizon, enable_velocity_check=self.enable_velocity_check, body_defs=char["BodyDefs"],
            pos_dim=self.deepmimic.get_pos_feature_dim(), rot_dim=self.deepmimic.get_rot_feature_dim(),
            vel_offset=self.deepmimic.get_vel_offset(),
            vel_divisor=(1.0 / self.deepmimic.get_agent_update_rate()) if ctrl.get("RecordVelAsPos", False) else 1.0,
            record_all_world=bool(ctrl.get("RecordAllWorld", False)),
            record_world_root_pos=bool(ctrl.get("RecordWorldRootPos", False)))

    def _vec_env(self):
        if self._vec is None:
            self._vec = VecSimEnv(self.dynamic_ensemble, 1, termination=self._termination, horizon=self.horizon,
                                  enable_velocity_check=self.enable_velocity_check)
        return self._vec

    def seed_env(self, seed=None):
        """sim_env.py:122-132."""
        if seed and self.deepmimic is not None:
            self.deepmimic.seed(seed)
        self.np_random = np.random.RandomState(seed)
        return seed

    def get_observation(self):
        return self.ob

    def set_observation(self, value):
        self.ob = value

    def step(self, action):
        """sim_env.py:140-162: ob += member forward; reward 0; done from is_done(); info tolerates ['valid']."""
        assert self.ob is not None
        if self._fast is None:
            term = self._termination or HumanoidTermination(horizon=self.horizon,
                                                            enable_velocity_check=self.enable_velocity_check)
            self._fast = _SingleStep(self.dynamic_ensemble, term)
        # device state is fp32; the observation handed back is its exact float64 widening (the reference keeps a
        # float64 accumulator, sim_env.py:158, but feeds the model the fp32 cast of it, sim_env.py:155)
        ob, disc, done = self._fast.step(np.asarray(self.ob, dtype=np.float64), np.asarray(action, dtype=np.float64),
                                         self.num_steps, self.reset_counter)
        self.num_steps += 1
        self.ob = ob
        self._last_done = done
        self._last_disc = disc
        return copy.deepcopy(self.ob), 0, self._last_done, {"valid": True, "disc": self._last_disc}

    def is_done(self):
        """sim_env.py:164-173 evaluated on the state produced by the last step."""
        return bool(getattr(self, "_last_done", False)) or self.num_steps >= self.horizon

    def reset(self):
        """sim_env.py:270-285."""
        self.num_steps = 0
        if self.deepmimic is not None:
            time = self.np_random.uniform(low=0, high=self.time_max)
            self.reset_dict["time"] = time
            self.deepmimic.reset_time(**self.reset_dict)
            self.ob = np.asarray(self.deepmimic.record_state(0), dtype=np.float64)
        elif self._reset_fn is not None:
            s0 = self._reset_fn(1, self.np_random)   # may be a CUDA tensor (VecSimEnv.clip_reset_fn)
            s0 = s0.detach().cpu().numpy() if torch.is_tensor(s0) else np.asarray(s0)
            self.ob = np.asarray(s0, dtype=np.float64).reshape(-1).copy()
        elif self._reset_states is not None:
            i = self.np_random.randint(0, len(self._reset_states))
            self.ob = np.asarray(self._reset_states[i], dtype=np.float64).copy()
        else:
            raise RuntimeError("SimEnv needs deepmimic_args, reset_fn or reset_states to draw initial states")
        self.reset_counter = (self.reset_counter + 1) % len(self.dynamic_ensemble.models)
        self.dynamics = self.dynamic_ensemble.models[self.reset_counter]
        self.dynamics.model.eval()
        self._last_done = False
        return copy.deepcopy(self.ob)

    def render(self, mode="human", close=False):
        pass

    def close(self):
        self._fast = None
        self._vec = None

    # EzPickle-equivalent: re-create from ctor args, dropping device state (sim_env.py:48)
    def __getstate__(self):
        return self._ctor  # the device handle, streams and graphs are re-created lazily in the new process

    def __setstate__(self, d):
        self.__init__(**d)
