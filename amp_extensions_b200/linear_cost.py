"""MILO's IPM / random-Fourier-feature cost with the reference's surface, evaluated on B200.

Mirrors reference milo/milo/linear_cost.py:6-152 (RBFLinearCost): same constructor arguments, the same
host-side RNG consumption (so bandwidth, rff weights and bias are bit-identical to the reference's for a
given seed and torch build), same return shapes (CPU tensors [B,1], info dict keys).  Feature
evaluation, the cost dot product and the bonus combine run through libsimstep's tcgen05 GEMM.
"""
import numpy as np
import torch
import torch.nn as nn

from . import engine as _engine


class RBFLinearCost:
    def __init__(self, expert_data, feature_dim=1024, input_type="ss", cost_range=[-1.0, 0.0], bw_quantile=0.1,
                 bw_samples=100000, lambda_b=1.0, lr=0.0, seed=100, precision=None, device=None, split="auto",
                 split_tol=3e-4):
        torch.manual_seed(seed)  # linear_cost.py:33-35
        np.random.seed(seed)
        self.expert_data = expert_data
        input_dim = expert_data.size(1)
        self.input_type = input_type
        self.feature_dim = feature_dim
        self.cost_range = cost_range
        if cost_range is not None:
            self.c_min, self.c_max = cost_range
        self.lambda_b = lambda_b
        self.lr = lr
        self.quantile = bw_quantile
        self.bw_samples = bw_samples
        self._precision = precision
        self._device = device
        # hi/lo operand pairs for the feature GEMM (three products, ~21 mantissa bits into the cosine): True / False, or
        # "auto": loaded, and switched off by fit_cost when plain operands measurably meet the budget (split_decision)
        self._split = split
        self._split_tol = float(split_tol)
        self.split_active = bool(split)  # "auto" starts with the split on
        self.split_report = None
        self._eng = None
        self.bw = self.fit_bandwidth(expert_data)
        # linear_cost.py:53-55 (the nn.Linear default init consumes RNG before rand_like, as in the reference)
        self.rff = nn.Linear(input_dim, feature_dim)
        self.rff.bias.data = (torch.rand_like(self.rff.bias.data) - 0.5) * 2.0 * np.pi
        self.rff.weight.data = torch.rand_like(self.rff.weight.data) / (self.bw + 1e-8)
        self.w = None
        self.expert_rep, self.phi_e = self._expert_features(expert_data)  # linear_cost.py:61-62

    # -- host-side fitting (same arithmetic and RNG stream as the reference) --------------------
    def fit_bandwidth(self, data):
        """linear_cost.py:73-82: quantile of the distance between random pairs."""
        num_data = data.shape[0]
        idxs_0 = torch.randint(low=0, high=num_data, size=(self.bw_samples,))
        idxs_1 = torch.randint(low=0, high=num_data, size=(self.bw_samples,))
        norm = torch.norm(data[idxs_0, :] - data[idxs_1, :], dim=1)
        return torch.quantile(norm, q=self.quantile).item()

    # -- device side --------------------------------------------------------------------------
    def engine(self):
        if self._eng is None:
            d = self.rff.weight.shape[1]
            self._eng = _engine.Engine(state_dim=d, action_dim=0, num_models=1, hidden_sizes=[], dense_connect=True,
                                       transform=False, precision=self._precision, device=self._device)
            self._rff_stamp = None
        # (storage address, in-place version) per parameter: `.data` hands out a fresh wrapper on every access, so
        # its id() is not a stamp; an assignment to `.data` changes data_ptr()
        stamp = tuple((p.data_ptr(), p._version) for p in (self.rff.weight, self.rff.bias))
        if stamp != self._rff_stamp:
            # this engine's "state" is the whole cost input row, whatever input_type built it
            self._eng.load_rff(self.rff.weight.data, self.rff.bias.data, split=bool(self._split), input_type="s")
            self._rff_stamp = stamp
        if self._eng.rff_split_loaded and self._eng.rff_split != self.split_active:
            self._eng.set_rff_split(self.split_active)
        return self._eng

    def _precise_engine(self):
        """The engine with the hi/lo split forced on when it was loaded with that capability: feature MEANS (phi_e,
        fit_cost's w, get_expert_cost) are differences of nearly equal averages, where a rounding bias that is
        harmless per row is not; they are computed once per iteration on a few thousand rows."""
        eng = self.engine()
        if getattr(eng, "rff_split_loaded", False) and not eng.rff_split:
            eng.set_rff_split(True)
        return eng

    def mark_dirty(self):
        """Force a re-upload of the rff layer on the next use (after replacing a parameter in a way the
        (data_ptr, version) stamp cannot see)."""
        self._rff_stamp = None

    @staticmethod
    def _round_operand(t, precision):
        """float64 copy of `t` rounded to the tensor-core operand format of `precision`."""
        t = t.detach().to(torch.float32)
        if precision == "bf16":
            return t.to(torch.bfloat16).to(torch.float64)
        if precision == "tf32":  # 10 explicit mantissa bits, round to nearest (cvt.rna.tf32)
            bits = t.contiguous().view(torch.int32)
            bits = (bits + 0x1000) & ~0x1FFF
            return bits.view(torch.float32).to(torch.float64)
        return t.clamp(-65504.0, 65504.0).to(torch.float16).to(torch.float64)

    def split_decision(self, x, w=None, max_rows=512):
        """Measured error of the PLAIN (single-product) operand format on rows `x`: the cost phi(x).w evaluated in
        float64 from exact operands and from operands rounded to the engine's format.  The split stays on where the
        worst row error exceeds split_tol * max|cost| (3e-4: a third of the north star's 1e-3, the rest is left to
        the ensemble's own rounding).  Returns {"err", "scale", "split"}."""
        w = self.w if w is None else w
        prec = self._precision or _engine.DEFAULT_PRECISION
        x = torch.as_tensor(x)[:max_rows].detach().cpu()
        W, b = self.rff.weight.data.cpu(), self.rff.bias.data.cpu().double()
        scale_phi = float(np.sqrt(2.0 / self.feature_dim))
        wd = w.detach().cpu().double()
        exact = (torch.cos(x.double() @ W.double().t() + b) * scale_phi) @ wd
        plain = (torch.cos(self._round_operand(x, prec) @ self._round_operand(W, prec).t() + b) * scale_phi) @ wd
        err = float((plain - exact).abs().max())
        scale = float(exact.abs().max())
        return {"err": err, "scale": scale, "split": bool(err > self._split_tol * max(scale, 1e-30)),
                "rows": int(x.shape[0]), "precision": prec, "tol": self._split_tol}

    def _expert_features(self, expert_data):
        """(phi(expert) as a CPU tensor, its mean): the mean comes from the device's fp64 column sums."""
        phi, psum = self._precise_engine().rff_features(expert_data, want_sum=True)
        return phi.cpu(), (psum / max(int(expert_data.shape[0]), 1)).float().cpu()

    def get_rep(self, x):
        """linear_cost.py:64-71: cos(rff(x)) * sqrt(2/D), returned on the CPU like the reference."""
        with torch.no_grad():
            return self.engine().rff_features(x).cpu()

    def fit_cost(self, data_pi):
        """linear_cost.py:84-94: w = mean phi(pi) - mean phi(expert); returns w.w."""
        _, psum = self._precise_engine().rff_features(data_pi, want_sum=True)
        phi = (psum / max(int(data_pi.shape[0]), 1)).float().cpu()
        feat_diff = phi - self.phi_e
        self.w = feat_diff
        if self._split == "auto":
            sample = torch.cat([torch.as_tensor(data_pi)[:384].cpu().float(), self.expert_data[:128].cpu().float()])
            self.split_report = self.split_decision(sample)
            self.split_active = self.split_report["split"]
        return torch.dot(self.w, feat_diff).item()

    def get_costs(self, x):
        """linear_cost.py:96-103."""
        dot = self.engine().rff_dot(x, self.w).cpu().unsqueeze(1)
        if self.cost_range is not None:
            return torch.clamp(dot, self.c_min, self.c_max)
        return dot

    def get_expert_cost(self):
        """linear_cost.py:105-109: (1 - lambda_b) * mean(clamp(phi(expert) . w)), evaluated on the device: the combine
        kernel's `ipm` output is (1 - lambda_b) * clamp(.), its mean comes from the fp64 moments kernel."""
        eng = self._precise_engine()
        x = self.expert_data.float()
        zeros = torch.zeros(x.shape[0], device=eng.device, dtype=torch.float32)
        clamp = self.cost_range is not None
        c_min, c_max = (self.c_min, self.c_max) if clamp else (0.0, 0.0)
        _, ipm, _ = eng.bonus_cost(x, zeros, self.w, self.lambda_b, 1.0, c_min, c_max, clamp)
        stats = eng.moments(ipm)
        return (stats[1] / stats[0]).float().cpu()

    def rff_input(self, states, actions, next_states=None):
        """linear_cost.py:115-126."""
        if self.input_type == "sa":
            return torch.cat([states, actions], dim=1)
        if self.input_type == "ss":
            assert next_states is not None
            return torch.cat([states, next_states], dim=1)
        if self.input_type == "sas":
            return torch.cat([states, actions, next_states], dim=1)
        if self.input_type == "s":
            return states
        raise NotImplementedError("Input type not implemented")

    def get_bonus_costs(self, states, actions, ensemble, next_states=None):
        """linear_cost.py:111-152. `ensemble` needs get_action_discrepancy(states, actions) and .threshold."""
        eng = self.engine()
        rff_in = self.rff_input(states.float(), actions.float(), None if next_states is None else next_states.float())
        disc = ensemble.get_action_discrepancy(states, actions)
        clamp = self.cost_range is not None
        c_min, c_max = (self.c_min, self.c_max) if clamp else (0.0, 0.0)
        cost, ipm, bonus = eng.bonus_cost(rff_in, disc, self.w, self.lambda_b, ensemble.threshold if clamp else 1.0,
                                          c_min, c_max, clamp)
        cost, ipm, bonus = cost.cpu().unsqueeze(1), ipm.cpu().unsqueeze(1), bonus.cpu().unsqueeze(1)
        v_targ = ipm / (1 - self.lambda_b) if self.lambda_b != 1 else self.get_costs(rff_in)
        info = {"bonus": bonus, "ipm": ipm, "v_targ": v_targ, "cost": cost}
        return cost, info

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_eng"] = None
        return d


class MLPCost(RBFLinearCost):
    """MILO's MMD cost over MLP features with the reference's surface (milo/milo/linear_cost.py:154-301): the
    feature map is `net(x)` = Linear/activation stack ending in Tanh, then cos(.) * sqrt(2/feature_dim).  Same
    constructor arguments, same torch RNG consumption (the nn.Linear layers are built in the reference's order
    before the bandwidth draw), so `net` is bit-identical to the reference's for a given seed and torch build.
    The hidden layers and the cos-feature head run through libsimstep's grouped tcgen05 GEMM
    (simstep_load_feature_net); fit_cost / get_costs / get_expert_cost / get_bonus_costs are inherited."""

    def __init__(self, expert_data, hidden_dims=[2048, 2048], activation="relu", feature_dim=1024, input_type="ss",
                 cost_range=[-1.0, 0.0], bw_quantile=0.1, bw_samples=100000, lambda_b=1.0, lr=0.0, seed=100,
                 precision=None, device=None):
        torch.manual_seed(seed)  # linear_cost.py:187-188
        np.random.seed(seed)
        self.expert_data = expert_data
        input_dim = expert_data.size(1)
        self.input_type = input_type
        self.feature_dim = feature_dim
        self.cost_range = cost_range
        if cost_range is not None:
            self.c_min, self.c_max = cost_range
        self.lambda_b = lambda_b
        self.lr = lr
        self._precision = precision
        self._device = device
        self._eng = None
        self._split, self.split_active, self.split_report = False, False, None  # no hi/lo pairs for MLP features
        # linear_cost.py:200-216, layer for layer
        self.activation_name = "relu" if activation == "relu" else "tanh"
        self.activation = nn.ReLU() if activation == "relu" else nn.Tanh()
        dim = feature_dim if not hidden_dims else hidden_dims[0]
        layers = [nn.Linear(input_dim, dim)]
        if hidden_dims[1:]:
            for size in hidden_dims[1:]:
                layers.append(self.activation)
                layers.append(nn.Linear(dim, size))
                dim = size
            layers.append(self.activation)
            layers.append(nn.Linear(dim, feature_dim))
        layers.append(nn.Tanh())
        self.net = nn.Sequential(*layers)
        self.quantile = bw_quantile
        self.bw_samples = bw_samples
        self.bw = self.fit_bandwidth(expert_data)  # linear_cost.py:219-221
        self.w = None
        self.expert_rep, self.phi_e = self._expert_features(expert_data)

    def _linears(self):
        return [m for m in self.net if isinstance(m, nn.Linear)]

    def engine(self):
        lin = self._linears()
        if self._eng is None:
            self._eng = _engine.Engine(state_dim=lin[0].in_features, action_dim=0, num_models=1,
                                       hidden_sizes=[l.out_features for l in lin[:-1]], dense_connect=False,
                                       activation=self.activation_name, transform=False, precision=self._precision,
                                       device=self._device)
            self._net_stamp = None
        stamp = tuple((l.weight._version, l.bias._version, id(l.weight.data), id(l.bias.data)) for l in lin)
        if stamp != self._net_stamp:
            self._eng.load_feature_net([l.weight.data for l in lin[:-1]], [l.bias.data for l in lin[:-1]],
                                       lin[-1].weight.data, lin[-1].bias.data, head_tanh=True)
            self._net_stamp = stamp
        return self._eng
