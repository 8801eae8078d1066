"""Thin object wrapper over a libsimstep handle: device tensors in, device tensors out.

torch is used for device memory and streams only; every computation is a call into the C ABI
(include/simstep.h).  A missing library or GPU raises — nothing here computes on the CPU.
"""
import ctypes as C
import math

import torch

from . import _lib

DEFAULT_PRECISION = "fp16"


def _ptr(t):
    if t is None:
        return C.c_void_p(0)
    return C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check_i32(t, name, n):
    """member / step-counter vectors cross the ABI as raw int32 pointers: refuse anything else instead of
    reinterpreting it."""
    if t is None:
        return
    if not (torch.is_tensor(t) and t.dtype == torch.int32 and t.is_cuda and t.is_contiguous() and t.numel() == n):
        raise TypeError(f"{name} must be a contiguous CUDA int32 tensor with {n} elements, got "
                        f"{getattr(t, 'dtype', type(t))} {tuple(getattr(t, 'shape', ()))}")


def _check_f32(t, name, shape):
    if not (torch.is_tensor(t) and t.dtype == torch.float32 and t.is_cuda and t.is_contiguous()
            and tuple(t.shape) == tuple(shape)):
        raise TypeError(f"{name} must be a contiguous CUDA float32 tensor of shape {tuple(shape)}, got "
                        f"{getattr(t, 'dtype', type(t))} {tuple(getattr(t, 'shape', ()))}")


def _dev_f32(x, device):
    """Contiguous fp32 CUDA tensor (no copy when it already is one)."""
    if not torch.is_tensor(x):
        x = torch.as_tensor(x)
    return x.to(device=device, dtype=torch.float32, non_blocking=True).contiguous()


class HumanoidTermination:
    """Fall-contact model of SimEnv (reference gym-simenv/gym_simenv/envs/sim_env.py:100-116, 164-268).

    body_defs: list of dicts with 'Shape', 'Param0', 'Param1' (humanoid3d.txt BodyDefs) indexed by body id.
    """

    # humanoid3d.txt BodyDefs (shape, Param0, Param1), see SURVEY.md appendix B
    HUMANOID3D = [
        ("sphere", 0.18, 0.18), ("sphere", 0.22, 0.22), ("sphere", 0.205, 0.205), ("capsule", 0.11, 0.30),
        ("capsule", 0.10, 0.31), ("box", 0.177, 0.055), ("capsule", 0.09, 0.18), ("capsule", 0.08, 0.135),
        ("sphere", 0.08, 0.08), ("capsule", 0.11, 0.30), ("capsule", 0.10, 0.31), ("box", 0.177, 0.055),
        ("capsule", 0.09, 0.18), ("capsule", 0.08, 0.135), ("sphere", 0.08, 0.08),
    ]
    FALL_CONTACT_BODIES = (0, 1, 2, 3, 4, 6, 7, 8, 9, 10, 12, 13, 14)

    def __init__(self, horizon=300, enable_velocity_check=False, body_defs=None, fall_contact_bodies=None,
                 pos_dim=3, rot_dim=6, vel_offset=136, vel_threshold=100.0, vel_divisor=1.0,
                 record_all_world=False, record_world_root_pos=False):
        self.horizon = int(horizon)
        self.enable_velocity_check = bool(enable_velocity_check)
        self.body_defs = list(body_defs) if body_defs is not None else list(self.HUMANOID3D)
        self.fall_contact_bodies = tuple(fall_contact_bodies if fall_contact_bodies is not None
                                         else self.FALL_CONTACT_BODIES)
        self.pos_dim, self.rot_dim = int(pos_dim), int(rot_dim)
        self.vel_offset = int(vel_offset)
        self.vel_threshold = float(vel_threshold)
        self.vel_divisor = float(vel_divisor)
        self.record_all_world = bool(record_all_world)
        self.record_world_root_pos = bool(record_world_root_pos)

    def to_struct(self):
        t = _lib.SimstepTermination()
        t.horizon = self.horizon
        t.enable_velocity_check = int(self.enable_velocity_check)
        t.vel_offset = self.vel_offset
        t.vel_threshold = self.vel_threshold
        t.vel_divisor = self.vel_divisor
        t.record_all_world = int(self.record_all_world)
        t.record_world_root_pos = int(self.record_world_root_pos)
        t.n_bodies = len(self.fall_contact_bodies)
        t.pos_dim = self.pos_dim
        for i, b in enumerate(self.fall_contact_bodies):
            d = self.body_defs[b]
            if isinstance(d, dict):
                shape, p0, p1 = d["Shape"], d["Param0"], d["Param1"]
            else:
                shape, p0, p1 = d
            t.body_offset[i] = (self.pos_dim + self.rot_dim) * b + 1
            t.body_shape[i] = _lib.SHAPE.get(shape, _lib.SHAPE["box"])
            t.body_param0[i] = float(p0)
            t.body_param1[i] = float(p1)
        return t


class Engine:
    """One libsimstep handle on one CUDA device."""

    def __init__(self, state_dim, action_dim, num_models, hidden_sizes, dense_connect=True, activation="relu",
                 transform=True, precision=None, device=None, max_chunk_envs=0):
        if not torch.cuda.is_available():
            raise _lib.SimstepError("amp_extensions_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise _lib.SimstepError(f"device must be a CUDA device, got {self.device}")
        self.S, self.A, self.N = int(state_dim), int(action_dim), int(num_models)
        self.hidden = [int(h) for h in hidden_sizes]
        self.precision = precision or DEFAULT_PRECISION
        cfg = _lib.SimstepConfig()
        cfg.abi_version = _lib.ABI_VERSION
        cfg.state_dim, cfg.action_dim, cfg.n_models, cfg.n_hidden = self.S, self.A, self.N, len(self.hidden)
        for i, h in enumerate(self.hidden):
            cfg.hidden[i] = h
        cfg.dense_connect = int(bool(dense_connect))
        cfg.activation = _lib.ACT[activation if activation in _lib.ACT else "tanh"]
        cfg.transform = int(bool(transform))
        cfg.precision = _lib.PREC[self.precision]
        cfg.max_chunk_envs = int(max_chunk_envs)
        self.transform = bool(transform)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.simstep_create(C.byref(cfg), C.byref(self._h)))
        self.rff_dim = 0
        self.rff_in = 0
        # bumped by every call that re-allocates device parameters or changes what the step's launches bake in
        # (load_* / set_*): captured CUDA graphs of an older generation must not be replayed
        self.generation = 0
        # bumped by load_policy only: it replaces the policy's device parameters and discards the NPG state
        self.policy_generation = 0

    # -- lifetime -----------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.simstep_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        _lib.check(rc, self._h)

    # -- parameters ---------------------------------------------------------------------
    def load_ensemble(self, weights, biases, transforms=None):
        """weights[m][l], biases[m][l]: CPU fp32 tensors in nn.Linear layout; transforms: 6 vectors or None."""
        nl = len(self.hidden) + 1
        keep = []
        wp = (C.c_void_p * (self.N * nl))()
        bp = (C.c_void_p * (self.N * nl))()
        for m in range(self.N):
            for l in range(nl):
                w = weights[m][l].detach().to("cpu", torch.float32).contiguous()
                b = biases[m][l].detach().to("cpu", torch.float32).contiguous()
                keep += [w, b]
                wp[m * nl + l] = w.data_ptr()
                bp[m * nl + l] = b.data_ptr()
        tp = None
        if self.transform:
            if transforms is None:
                raise ValueError("transform=True needs the six transformation vectors")
            tfs = [t.detach().to("cpu", torch.float32).contiguous() for t in transforms]
            keep += tfs
            tp = (C.c_void_p * 6)(*[t.data_ptr() for t in tfs])
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_load_ensemble(self._h, wp, bp, tp))
            self.generation += 1

    def set_termination(self, term):
        t = term.to_struct()
        self._check(self.lib.simstep_set_termination(self._h, C.byref(t)))
        self.generation += 1

    def load_rff(self, weight, bias, split=True):
        w = weight.detach().to("cpu", torch.float32).contiguous()
        b = bias.detach().to("cpu", torch.float32).contiguous()
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_load_rff(self._h, w.shape[0], w.shape[1], _ptr(w), _ptr(b), int(bool(split))))
            self.generation += 1
        self.rff_dim, self.rff_in = int(w.shape[0]), int(w.shape[1])
        self.rff_split_loaded = bool(split)
        self.rff_split = bool(split)

    def saturation_count(self, reset=False):
        """Normalised inputs beyond the fp16 range seen by this (fp16) handle so far; 0 for tf32 / bf16 handles.
        Synchronises."""
        n = C.c_int64(0)
        self._check(self.lib.simstep_saturation_count(self._h, C.byref(n), int(bool(reset))))
        return int(n.value)

    def forward_launches(self, n_envs):
        """Launches the ensemble forward pass takes for n_envs rows: 1 = the column-fused kernel (csrc/gemm_chain.cuh),
        n_hidden + 1 = one grouped launch per layer (simstep_forward_launches)."""
        n = C.c_int32(0)
        self._check(self.lib.simstep_forward_launches(self._h, int(n_envs), C.byref(n)))
        return int(n.value)

    def check_guards(self):
        """(guarded buffers, overwritten guard bytes) of the handle's workspaces; buffers are only guarded when
        SIMSTEP_DEBUG_GUARDS=1 was set when the engine was created (simstep_debug_check_guards).  Synchronises."""
        n, bad = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.simstep_debug_check_guards(self._h, C.byref(n), C.byref(bad)))
        return int(n.value), int(bad.value)

    def round_rows(self, n_envs):
        """Row granule at which a pass of the column-fused forward kernel ends on a whole round of its CTA pairs: the
        kernel's units are (256-row env tile, member) pairs taken round-robin by sm_count / 2 CTA pairs, so a chunk of
        lcm(pairs, N) / N env tiles leaves no partial round.  256 when every layer is a launch of its own.  Callers that
        split a batch into chunks (HostEnvPipeline) cut at multiples of it."""
        if self.forward_launches(n_envs) != 1:
            return 256
        import math
        pairs = torch.cuda.get_device_properties(self.device).multi_processor_count // 2
        return 256 * (math.lcm(pairs, self.N) // self.N)

    def set_rff_split(self, split):
        """Turn the hi/lo (three-product) evaluation of the random-feature layer on or off (simstep_set_rff_split)."""
        self._check(self.lib.simstep_set_rff_split(self._h, int(bool(split))))
        self.generation += 1
        self.rff_split = bool(split)

    HEAD_TANH_COS, HEAD_LINEAR = 1, 2
    COST_IDENTITY, COST_GAIL_LS, COST_GAIL_LL = 0, 1, 2

    def set_cost_transform(self, transform):
        """What rff_dot / bonus_cost apply to phi(x).w before the bonus combine (COST_*: identity, or GAILCost's
        least-squares / log-likelihood costs of a discriminator output, gail_cost.py:232-246)."""
        self._check(self.lib.simstep_set_cost_transform(self._h, int(transform)))
        self.generation += 1

    def load_feature_net(self, weights, biases, head_weight, head_bias, head_tanh=True, head_mode=None):
        """MLPCost's feature map (linear_cost.py:200-236): hidden nn.Linear layers + the last nn.Linear whose
        output goes through tanh and cos.  The handle must have been created with num_models=1, action_dim=0,
        dense_connect=False, transform=False and hidden_sizes = the hidden layers' widths."""
        nl = len(weights)
        ws = [w.detach().to("cpu", torch.float32).contiguous() for w in weights]
        bs = [b.detach().to("cpu", torch.float32).contiguous() for b in biases]
        hw = head_weight.detach().to("cpu", torch.float32).contiguous()
        hb = head_bias.detach().to("cpu", torch.float32).contiguous()
        wp = (C.c_void_p * max(nl, 1))(*[w.data_ptr() for w in ws])
        bp = (C.c_void_p * max(nl, 1))(*[b.data_ptr() for b in bs])
        with torch.cuda.device(self.device):
            mode = head_mode if head_mode is not None else (self.HEAD_TANH_COS if head_tanh else self.HEAD_LINEAR)
            self._check(self.lib.simstep_load_feature_net(self._h, wp, bp, int(hw.shape[0]), _ptr(hw), _ptr(hb),
                                                          int(mode)))
            self.generation += 1
        self.rff_dim, self.rff_in = int(hw.shape[0]), self.S

    # -- ensemble -----------------------------------------------------------------------
    def forward(self, state, action):
        """All members' un-normalised predictions, CUDA tensor [N, E, S]."""
        s, a = _dev_f32(state, self.device), _dev_f32(action, self.device)
        E = s.shape[0]
        out = torch.empty((self.N, E, self.S), device=self.device, dtype=torch.float32)
        self._check(self.lib.simstep_forward(self._h, _ptr(s), _ptr(a), E, _ptr(out), _stream(self.device)))
        return out

    def discrepancy(self, state, action):
        s, a = _dev_f32(state, self.device), _dev_f32(action, self.device)
        E = s.shape[0]
        out = torch.empty((E,), device=self.device, dtype=torch.float32)
        self._check(self.lib.simstep_discrepancy(self._h, _ptr(s), _ptr(a), E, _ptr(out), _stream(self.device)))
        return out

    def step(self, state, action, member, num_steps, next_state=None, disc=None, done=None, want_disc=True,
             want_done=True):
        """In-place batched env step on device tensors. Returns (next_state, disc, done)."""
        E = state.shape[0]
        _check_f32(state, "state", (E, self.S)); _check_f32(action, "action", (E, self.A))
        _check_i32(member, "member", E); _check_i32(num_steps, "num_steps", E)
        if next_state is None:
            next_state = torch.empty_like(state)
        if disc is None and want_disc:
            disc = torch.empty((E,), device=self.device, dtype=torch.float32)
        if done is None and want_done:
            done = torch.empty((E,), device=self.device, dtype=torch.uint8)
        self._check(self.lib.simstep_step(self._h, _ptr(state), _ptr(action), _ptr(member), _ptr(num_steps), E,
                                          _ptr(next_state), _ptr(disc), _ptr(done), _stream(self.device)))
        return next_state, disc, done

    def step_cost(self, state, action, member, num_steps, w, lambda_b, threshold, c_min=-1.0, c_max=0.0,
                  clamp_cost=True, next_state=None, disc=None, done=None, cost=None, ipm=None, bonus=None):
        E = state.shape[0]
        _check_f32(state, "state", (E, self.S)); _check_f32(action, "action", (E, self.A))
        _check_i32(member, "member", E); _check_i32(num_steps, "num_steps", E)
        f32 = dict(device=self.device, dtype=torch.float32)
        next_state = torch.empty_like(state) if next_state is None else next_state
        disc = torch.empty((E,), **f32) if disc is None else disc
        done = torch.empty((E,), device=self.device, dtype=torch.uint8) if done is None else done
        cost = torch.empty((E,), **f32) if cost is None else cost
        ipm = torch.empty((E,), **f32) if ipm is None else ipm
        bonus = torch.empty((E,), **f32) if bonus is None else bonus
        self._check(self.lib.simstep_step_cost(
            self._h, _ptr(state), _ptr(action), _ptr(member), _ptr(num_steps), E, _ptr(next_state), _ptr(disc),
            _ptr(done), _ptr(w), float(lambda_b), float(threshold), float(c_min), float(c_max), int(bool(clamp_cost)),
            _ptr(cost), _ptr(ipm), _ptr(bonus), _stream(self.device)))
        return next_state, disc, done, cost, ipm, bonus

    # -- cost ---------------------------------------------------------------------------
    def rff_features(self, x, want_sum=False):
        x = _dev_f32(x, self.device)
        n = x.shape[0]
        phi = torch.empty((n, self.rff_dim), device=self.device, dtype=torch.float32)
        psum = torch.empty((self.rff_dim,), device=self.device, dtype=torch.float64) if want_sum else None
        self._check(self.lib.simstep_rff_features(self._h, _ptr(x), n, _ptr(phi), _ptr(psum), _stream(self.device)))
        return (phi, psum) if want_sum else phi

    def rff_dot(self, x, w):
        x, w = _dev_f32(x, self.device), _dev_f32(w, self.device)
        n = x.shape[0]
        out = torch.empty((n,), device=self.device, dtype=torch.float32)
        self._check(self.lib.simstep_rff_dot(self._h, _ptr(x), n, _ptr(w), _ptr(out), _stream(self.device)))
        return out

    def bonus_cost(self, x, disc, w, lambda_b, threshold, c_min=-1.0, c_max=0.0, clamp_cost=True):
        x, w, disc = _dev_f32(x, self.device), _dev_f32(w, self.device), _dev_f32(disc, self.device)
        n = x.shape[0]
        cost, ipm, bonus = (torch.empty((n,), device=self.device, dtype=torch.float32) for _ in range(3))
        self._check(self.lib.simstep_bonus_cost(self._h, _ptr(x), _ptr(disc), n, _ptr(w), float(lambda_b),
                                                float(threshold), float(c_min), float(c_max), int(bool(clamp_cost)),
                                                _ptr(cost), _ptr(ipm), _ptr(bonus), _stream(self.device)))
        return cost, ipm, bonus

    def histogram(self, x, lo, hi, bins):
        """int64 [bins] counts of a device fp32 vector over [lo, hi] (see simstep_histogram)."""
        x = _dev_f32(x, self.device).reshape(-1)
        out = torch.empty((int(bins),), device=self.device, dtype=torch.int64)
        self._check(self.lib.simstep_histogram(self._h, _ptr(x), x.numel(), float(lo), float(hi), int(bins), _ptr(out),
                                               _stream(self.device)))
        return out

    QOP_MINMAX, QOP_HIST, QOP_SELECT, QOP_WINMIN = 0, 1, 2, 3

    def quantile_op(self, op, x=None, bins=0, qstate=None, counts=None, out=None):
        """One device-side step of the distributed quantile (simstep_quantile_op); x: contiguous fp32 CUDA vector."""
        n = 0 if x is None else x.numel()
        self._check(self.lib.simstep_quantile_op(self._h, int(op), _ptr(x), n, int(bins), _ptr(qstate), _ptr(counts),
                                                 _ptr(out), _stream(self.device)))

    def reduce_max_sum(self, x, out=None):
        """[max, sum] of a device vector as fp64 (written into `out` when given)."""
        x = _dev_f32(x, self.device)
        if out is None:
            out = torch.empty((2,), device=self.device, dtype=torch.float64)
        self._check(self.lib.simstep_reduce_max_sum(self._h, _ptr(x), x.numel(), _ptr(out), _stream(self.device)))
        return out

    # -- measurement --------------------------------------------------------------------
    def profile_enable(self, on=True):
        self._check(self.lib.simstep_profile_enable(self._h, int(bool(on))))

    def profile_read(self, reset=True):
        """{category: (milliseconds, regions)} of device time measured with CUDA events inside the library."""
        n = len(_lib.PROF_CATEGORIES)
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        self._check(self.lib.simstep_profile_read(self._h, ms, cnt, int(bool(reset))))
        return {name: (ms[i], cnt[i]) for i, name in enumerate(_lib.PROF_CATEGORIES)}

    # -- imitation reward ---------------------------------------------------------------
    def load_clip(self, character, clip):
        ch = character.to_struct()
        fr = torch.as_tensor(clip.frames, dtype=torch.float32).contiguous()
        fv = torch.as_tensor(clip.frame_vels, dtype=torch.float32).contiguous()
        ft = torch.as_tensor(clip.frame_times, dtype=torch.float32).contiguous()
        cd = torch.as_tensor(clip.cycle_delta, dtype=torch.float32).contiguous()
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_load_clip(self._h, C.byref(ch), fr.shape[0], _ptr(fr), _ptr(fv), _ptr(ft),
                                                   float(clip.duration), int(bool(clip.loop_wrap)), _ptr(cd)))
            self.generation += 1
        self.dof = int(fr.shape[1])
        self.n_joints = int(ch.n_joints)

    def imitation_reward(self, pose, vel, kin_time, kin_origin=None, want_terms=False, out=None):
        pose, vel = _dev_f32(pose, self.device), _dev_f32(vel, self.device)
        kin_time = _dev_f32(kin_time, self.device)
        kin_origin = _dev_f32(kin_origin, self.device) if kin_origin is not None else None
        E = pose.shape[0]
        reward = out if out is not None else torch.empty((E,), device=self.device, dtype=torch.float32)
        terms = torch.empty((E, 5), device=self.device, dtype=torch.float32) if want_terms else None
        self._check(self.lib.simstep_imitation_reward(self._h, _ptr(pose), _ptr(vel), _ptr(kin_time),
                                                      _ptr(kin_origin), E, _ptr(reward), _ptr(terms),
                                                      _stream(self.device)))
        return (reward, terms) if want_terms else reward

    def record_state(self, pose, vel, record_all_world=False, record_world_root_pos=False,
                     record_world_root_rot=True, vel_scale=1.0):
        """Env state features [E, 1 + 15 * n_joints] of generalized poses / velocities (CtController.cpp:378-495);
        the flag defaults are data/controllers/humanoid3d_rot_ctrl.txt's."""
        pose, vel = _dev_f32(pose, self.device), _dev_f32(vel, self.device)
        E = pose.shape[0]
        out = torch.empty((E, 1 + 15 * self.n_joints), device=self.device, dtype=torch.float32)
        self._check(self.lib.simstep_record_state(self._h, _ptr(pose), _ptr(vel), E, int(record_all_world),
                                                  int(record_world_root_pos), int(record_world_root_rot),
                                                  float(vel_scale), _ptr(out), _stream(self.device)))
        return out

    def clip_sample(self, kin_time, kin_origin=None):
        kin_time = _dev_f32(kin_time, self.device)
        kin_origin = _dev_f32(kin_origin, self.device) if kin_origin is not None else None
        E = kin_time.shape[0]
        pose = torch.empty((E, self.dof), device=self.device, dtype=torch.float32)
        vel = torch.empty((E, self.dof), device=self.device, dtype=torch.float32)
        self._check(self.lib.simstep_clip_sample(self._h, _ptr(kin_time), _ptr(kin_origin), E, _ptr(pose), _ptr(vel),
                                                 _stream(self.device)))
        return pose, vel

    # -- rollout helpers ----------------------------------------------------------------
    def load_policy(self, weights, biases, nonlinearity="tanh", in_shift=None, in_scale=None, out_shift=None,
                    out_scale=None, log_std=None):
        """mjrl's Gaussian MLP policy (mjrl/mjrl/policies/gaussian_mlp.py:6-104): nn.Linear weights/biases of
        FCNetwork.fc_layers, its four transformations and the policy's log_std (CPU tensors / arrays)."""
        nl = len(weights)
        ws = [torch.as_tensor(w).detach().to("cpu", torch.float32).contiguous() for w in weights]
        bs = [torch.as_tensor(b).detach().to("cpu", torch.float32).contiguous() for b in biases]
        lin = (C.c_int32 * nl)(*[int(w.shape[1]) for w in ws])
        lout = (C.c_int32 * nl)(*[int(w.shape[0]) for w in ws])
        wp = (C.c_void_p * nl)(*[w.data_ptr() for w in ws])
        bp = (C.c_void_p * nl)(*[b.data_ptr() for b in bs])

        def vec(x):
            return None if x is None else torch.as_tensor(x).detach().to("cpu", torch.float32).contiguous()

        extra = [vec(in_shift), vec(in_scale), vec(out_shift), vec(out_scale), vec(log_std)]
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_load_policy(self._h, nl, lin, lout, wp, bp, int(nonlinearity == "tanh"),
                                                     *[_ptr(x) for x in extra]))
            self.generation += 1
            self.policy_generation += 1
        self.policy_obs_dim, self.policy_act_dim = int(ws[0].shape[1]), int(ws[-1].shape[0])

    def policy_act(self, obs, noise=None, action=None, mean=None, want_mean=True):
        """(action, mean) of the loaded policy for a batch of observations; noise [E, act] standard normal draws or
        None for the evaluation action."""
        E = obs.shape[0]
        f32 = dict(device=self.device, dtype=torch.float32)
        if action is None:
            action = torch.empty((E, self.policy_act_dim), **f32)
        if mean is None and want_mean:
            mean = torch.empty((E, self.policy_act_dim), **f32)
        self._check(self.lib.simstep_policy_act(self._h, _ptr(obs), _ptr(noise), E, _ptr(action), _ptr(mean),
                                                _stream(self.device)))
        return action, mean

    def discount(self, reward, gamma, baseline=None, gae_lambda=1.0, seg_end=None, lengths=None, terminated=None,
                 want_returns=True, want_advantages=None):
        """Time-major [T, E] discounted returns and GAE advantages (mjrl/mjrl/utils/process_samples.py:3-45)."""
        T, E = reward.shape
        want_advantages = (baseline is not None) if want_advantages is None else want_advantages
        ret = torch.empty_like(reward) if want_returns else None
        adv = torch.empty_like(reward) if want_advantages else None
        self._check(self.lib.simstep_discount(self._h, _ptr(reward), _ptr(baseline), _ptr(seg_end), _ptr(lengths),
                                              _ptr(terminated), T, E, float(gamma), float(gae_lambda), _ptr(ret),
                                              _ptr(adv), _stream(self.device)))
        return ret, adv

    def auto_reset(self, next_state, done, pool, pick, state_out, member=None, num_steps=None):
        E = next_state.shape[0]
        self._check(self.lib.simstep_auto_reset(self._h, _ptr(next_state), _ptr(done), _ptr(pool), _ptr(pick),
                                                int(pool.shape[0]), E, _ptr(state_out), _ptr(member), _ptr(num_steps),
                                                _stream(self.device)))
        return state_out

    def moments(self, x, valid=None):
        """{count, sum, sum of squares} of a device tensor as a CUDA fp64 [3] tensor."""
        out = torch.empty((3,), device=self.device, dtype=torch.float64)
        self._check(self.lib.simstep_moments(self._h, _ptr(x), _ptr(valid), x.numel(), _ptr(out), _stream(self.device)))
        return out

    def whiten(self, x, stats, valid=None, eps=1e-8, out=None):
        """(x - mean) / (std + eps) with mean/std from `stats` (see moments)."""
        out = torch.empty_like(x) if out is None else out
        self._check(self.lib.simstep_whiten(self._h, _ptr(x), _ptr(valid), x.numel(), _ptr(stats), float(eps), _ptr(out),
                                            _stream(self.device)))
        return out

    # -- natural policy gradient step of the loaded policy (simstep_npg_*) ----------------
    NPG_CG_START, NPG_CG_STEP = 0, 1

    def npg_init(self, min_log_std=-3.0):
        """Allocate the NPG state of the loaded policy; returns P, the length of its parameter vector."""
        n = C.c_int64(0)
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_npg_init(self._h, float(min_log_std), C.byref(n)))
        self.npg_n_params = int(n.value)
        return self.npg_n_params

    def _npg_rows(self, t, name, dtype=torch.float32):
        """Row tensors of the simstep_npg_* calls cross the ABI as raw device pointers: refuse anything else."""
        if t is None:
            return
        if not (torch.is_tensor(t) and t.dtype == dtype and t.device == self.device and t.is_contiguous()):
            raise TypeError(f"{name} must be a contiguous {dtype} tensor on {self.device}, got "
                            f"{getattr(t, 'dtype', type(t))} on {getattr(t, 'device', '?')}")

    def npg_params(self, theta=None):
        """Set the parameters from a CUDA fp32 [P] tensor (mjrl's flat order), or return a copy of them."""
        if theta is not None:
            theta = theta.to(self.device, torch.float32).contiguous()
            self._check(self.lib.simstep_npg_params(self._h, 1, _ptr(theta), _stream(self.device)))
            return theta
        out = torch.empty((self.npg_n_params,), device=self.device, dtype=torch.float32)
        self._check(self.lib.simstep_npg_params(self._h, 0, _ptr(out), _stream(self.device)))
        return out

    def npg_grad(self, obs, act, adv, valid=None, out=None):
        n = obs.shape[0]
        for t, nm in ((obs, "obs"), (act, "act"), (adv, "adv")):
            self._npg_rows(t, nm)
        self._npg_rows(valid, "valid", torch.uint8)
        out = torch.empty((self.npg_n_params + 2,), device=self.device, dtype=torch.float64) if out is None else out
        self._check(self.lib.simstep_npg_grad(self._h, _ptr(obs), _ptr(act), _ptr(adv), _ptr(valid), n, _ptr(out),
                                              _stream(self.device)))
        return out

    def npg_prepare(self, obs, idx=None):
        n = obs.shape[0]
        self._npg_rows(obs, "obs")
        self._npg_rows(idx, "idx", torch.int64)
        self._check(self.lib.simstep_npg_prepare(self._h, _ptr(obs), n, _ptr(idx), 0 if idx is None else idx.numel(),
                                                 _stream(self.device)))

    def npg_fvp(self, obs, valid=None, idx=None, v=None, out=None):
        n = obs.shape[0]
        self._npg_rows(obs, "obs")
        self._npg_rows(valid, "valid", torch.uint8)
        self._npg_rows(idx, "idx", torch.int64)
        self._npg_rows(v, "v", torch.float64)
        out = torch.empty((self.npg_n_params + 2,), device=self.device, dtype=torch.float64) if out is None else out
        self._check(self.lib.simstep_npg_fvp(self._h, _ptr(obs), _ptr(valid), n, _ptr(idx),
                                             0 if idx is None else idx.numel(), _ptr(v), _ptr(out), _stream(self.device)))
        return out

    def npg_cg(self, op, sums, damping=0.0):
        self._check(self.lib.simstep_npg_cg(self._h, int(op), _ptr(sums), float(damping), _stream(self.device)))

    def npg_apply(self, step, const_lr=False):
        self._check(self.lib.simstep_npg_apply(self._h, float(step), int(bool(const_lr)), _stream(self.device)))

    def npg_diag(self, obs, act, adv, valid=None):
        for t, nm in ((obs, "obs"), (act, "act"), (adv, "adv")):
            self._npg_rows(t, nm)
        self._npg_rows(valid, "valid", torch.uint8)
        out = torch.empty((3,), device=self.device, dtype=torch.float64)
        self._check(self.lib.simstep_npg_diag(self._h, _ptr(obs), _ptr(act), _ptr(adv), _ptr(valid), obs.shape[0],
                                              _ptr(out), _stream(self.device)))
        return out

    def npg_scalars(self):
        """{r.r, g.x, alpha, gradient rows, mean advantage, CG iterations run} as a CUDA fp64 [6] tensor."""
        out = torch.empty((6,), device=self.device, dtype=torch.float64)
        self._check(self.lib.simstep_npg_scalars(self._h, _ptr(out), _stream(self.device)))
        return out

    # -- training (tf32 handles only) ---------------------------------------------------
    TRAIN_PARAMS, TRAIN_GRADS, TRAIN_MOMENTS = 0, 1, 2

    def train_init(self, max_batch_rows, optim="sgd", lr=1e-4, momentum=0.9, beta2=0.999, eps=1e-8):
        """Prepare the handle for DynamicsModel.train_step on device (dynamics.py:236-250).  optim: "sgd"
        (torch.optim.SGD, nesterov=True, as dynamics.py:199) or "adam" (momentum = beta1).  Call before
        load_ensemble: parameters loaded afterwards keep all their fp32 bits."""
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_train_init(self._h, int(max_batch_rows), 0 if optim == "sgd" else 1, float(lr),
                                                    float(momentum), float(beta2), float(eps)))

    def _train_call(self, fn, state, action, next_state, *extra):
        s, a, s2 = _dev_f32(state, self.device), _dev_f32(action, self.device), _dev_f32(next_state, self.device)
        assert s.dim() == 3 and s.shape[0] == self.N, "training batches are [n_models, batch_rows, dim]"
        loss = torch.zeros((self.N,), device=self.device, dtype=torch.float64)
        self._check(fn(self._h, _ptr(s), _ptr(a), _ptr(s2), int(s.shape[1]), *extra, _ptr(loss), _stream(self.device)))
        return loss

    def train_step(self, state, action, next_state, grad_clip=0.0):
        """One optimisation step of every member on its own batch; returns the members' losses (CUDA fp64 [N])."""
        return self._train_call(self.lib.simstep_train_step, state, action, next_state, C.c_float(float(grad_clip)))

    def train_step_graph(self, state, action, next_state, grad_clip=0.0):
        """train_step replayed from a CUDA graph (the step is ~45 small launches at the reference's 256-row batches,
        launch-latency bound when issued one by one).  The first call for a batch size runs eagerly (it also warms
        the kernels up), the second captures, later ones replay; inputs are copied into the graph's static
        buffers.  The returned loss tensor is overwritten by the next replay."""
        cache = self.__dict__.setdefault("_train_graphs", {})
        key = (int(state.shape[1]), float(grad_clip))
        ent = cache.get(key)
        if ent is None:
            cache[key] = "warm"
            return self.train_step(state, action, next_state, grad_clip)
        if ent == "warm":
            f32 = dict(device=self.device, dtype=torch.float32)
            sb = torch.empty(tuple(state.shape), **f32)
            ab = torch.empty(tuple(action.shape), **f32)
            nb = torch.empty(tuple(next_state.shape), **f32)
            loss = torch.zeros((self.N,), device=self.device, dtype=torch.float64)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._check(self.lib.simstep_train_step(self._h, _ptr(sb), _ptr(ab), _ptr(nb), int(sb.shape[1]),
                                                        C.c_float(float(grad_clip)), _ptr(loss), _stream(self.device)))
            ent = cache[key] = (g, sb, ab, nb, loss)
        g, sb, ab, nb, loss = ent
        sb.copy_(state, non_blocking=True)
        ab.copy_(action, non_blocking=True)
        nb.copy_(next_state, non_blocking=True)
        g.replay()
        return loss

    def train_loss(self, state, action, next_state):
        """DynamicsModel.validate_step (dynamics.py:252-262) for every member."""
        return self._train_call(self.lib.simstep_train_loss, state, action, next_state)

    def train_grads(self, state, action, next_state):
        """Forward + backward without an update; read the gradients with train_export(TRAIN_GRADS)."""
        return self._train_call(self.lib.simstep_train_grads, state, action, next_state)

    def train_export(self, what=0):
        """(weights[m][l], biases[m][l]) CPU tensors in nn.Linear layout: parameters, last gradients or the first
        optimiser moment."""
        n_layers = C.c_int32()
        lin = (C.c_int32 * 16)()
        lout = (C.c_int32 * 16)()
        self._check(self.lib.simstep_query(self._h, C.byref(n_layers), lin, lout, None, None))
        nl = n_layers.value
        ws = [[torch.empty((lout[l], lin[l]), dtype=torch.float32) for l in range(nl)] for _ in range(self.N)]
        bs = [[torch.empty((lout[l],), dtype=torch.float32) for l in range(nl)] for _ in range(self.N)]
        wp = (C.c_void_p * (self.N * nl))(*[ws[m][l].data_ptr() for m in range(self.N) for l in range(nl)])
        bp = (C.c_void_p * (self.N * nl))(*[bs[m][l].data_ptr() for m in range(self.N) for l in range(nl)])
        with torch.cuda.device(self.device):
            self._check(self.lib.simstep_train_export(self._h, int(what), wp, bp))
        return ws, bs
