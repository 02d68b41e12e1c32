"""Shared parity-check machinery: runs a library implementing include/lqgk.h (the CUDA product library on a GPU,
or the host emulation of the same step functions on CPU) against the float64 oracle."""
from __future__ import annotations

import os

import numpy as np
import torch

from lqg_b200 import abi
from oracle import adjoint_np as AD
from oracle import lqg_np as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_PATH = os.path.join(ROOT, "tests", "emul", "liblqgk_emul.so")

PM = O.point_mass_mats


def model_mats(name, **kw):
    return {"bounded": O.bounded_actor_mats, "bounded2": lambda **k: O.bounded_actor_mats(dim=2, **k),
            "subjective": O.subjective_actor_mats, "subjective2": lambda **k: O.subjective_actor_mats(dim=2, **k),
            "relobs": O.relative_observation_mats, "relobs2": lambda **k: O.relative_observation_mats(dim=2, **k),
            "pointmass": O.point_mass_mats,
            "hand": lambda **k: O.hand_model_mats(position_noise=0.3, **k),
            "delay2": lambda **k: tuple(O.delay_mats(m, 2) for m in O.bounded_actor_mats(**k)),
            # BASELINE config c4: TemporalDelayModel(PointMassBoundedActor, delay=2), 12-dim state (joint dim 24)
            "pmdelay2": lambda **k: tuple(O.delay_mats(m, 2) for m in O.point_mass_mats(**k))}[name](**kw)


MODEL_DIMS = {"bounded": (2, 2, 1, 2), "bounded2": (4, 4, 2, 4), "subjective": (2, 3, 1, 2), "subjective2": (4, 6, 2, 4),
              "relobs": (2, 2, 1, 1), "relobs2": (4, 4, 2, 2), "pointmass": (4, 4, 1, 3), "hand": (5, 5, 1, 2), "delay2": (6, 6, 1, 2), "pmdelay2": (12, 12, 1, 3)}
MODEL_PARAMS = {"bounded": ("action_variability", "sigma_target", "sigma_cursor", "action_cost"),
                "subjective": ("action_variability", "sigma_target", "sigma_cursor", "action_cost", "subj_noise",
                               "subj_vel_noise"),
                "relobs": ("action_variability", "sigma", "action_cost"),
                "pointmass": ("action_variability", "sigma_target", "sigma_cursor", "action_cost"),
                "hand": ("action_variability", "sigma_target", "sigma_cursor", "action_cost"),
                "delay": ("action_variability", "sigma_target", "sigma_cursor", "action_cost"),
                "pmdelay": ("action_variability", "sigma_target", "sigma_cursor", "action_cost")}
DEFAULTS = dict(action_variability=0.5, sigma_target=6.0, sigma_cursor=6.0, action_cost=1.0, subj_noise=1.0,
                subj_vel_noise=0.5, sigma=6.0)


def jittered_params(name, S, seed, scale=0.25):
    base = name.rstrip("2")
    
    rng = np.random.default_rng(seed)
    out = []
    for s in range(S):
        kw = {}
        for k in MODEL_PARAMS[base]:
            v0 = DEFAULTS[k] if base not in ("pointmass", "pmdelay") else dict(action_variability=1e-3, sigma_target=6.0,
                                                              sigma_cursor=6.0, action_cost=0.01)[k]
            kw[k] = v0 * (1.0 if s == 0 else float(np.exp(scale * rng.standard_normal())))
        out.append(kw)
    return out


class Case:
    """S jittered parameter samples of one model, N simulated trials, oracle results in float64.

    The trials are simulated from sample 0 and shared by all samples, or with `per_sample_data` one data set per sample,
    simulated from that sample's own parameters (X[S, N, T+1, d]; the library then sees x_sample_stride != 0).  The
    cotangents of the per-trial log-likelihoods are 1 (default), uniform(0.5, 1.5) (`weights`) or given explicitly (`w`,
    [S, N]); the oracle's gradient is that of sum_i w[s, i] ll[s, i] for every sample s."""

    def __init__(self, name, S, T, N, d=None, seed=0, weights=False, want_grad=True, per_sample_data=False, w=None):
        self.name, self.S, self.T, self.N = name, S, T, N
        x, b, u, y = MODEL_DIMS[name]
        self.d = d if d is not None else x
        self.dims = (x, b, u, y, self.d)
        self.per_sample_data = per_sample_data
        self.params = jittered_params(name, S, seed)
        self.mats = [model_mats(name, **kw) for kw in self.params]
        rng = np.random.default_rng(seed + 1)
        if per_sample_data:
            X = np.stack([O.simulate(*O.make_system(m, T), N, rng) for m in self.mats])[..., :self.d]
        else:
            sa, sd = O.make_system(self.mats[0], T)
            X = O.simulate(sa, sd, N, rng)[..., :self.d]
        self.X = X.astype(np.float32)                       # what the library sees
        X64 = self.X.astype(np.float64)
        if w is not None:
            self.w = np.asarray(w, dtype=np.float64)
            assert self.w.shape == (S, N), self.w.shape
        else:
            self.w = rng.uniform(0.5, 1.5, (S, N)) if weights else None
        self.ll = np.zeros((S, N))
        self.ga, self.gd = [], []
        for s, m in enumerate(self.mats):
            Xs = X64[s] if per_sample_data else X64
            if want_grad:
                ll, (ga, gd) = AD.value_and_grad(m[0], m[1], Xs, w=None if self.w is None else self.w[s])
                self.ga.append(ga); self.gd.append(gd)
            else:
                ll, _ = AD.forward(m[0], m[1], Xs)
            self.ll[s] = ll

    def tensors(self, device, dtype):
        act = {k: torch.tensor(np.stack([np.ascontiguousarray(m[0][k]) for m in self.mats]), dtype=dtype, device=device)
               for k in abi.ACTOR_KEYS}
        dyn = {k: torch.tensor(np.stack([np.ascontiguousarray(m[1][k]) for m in self.mats]), dtype=dtype, device=device)
               for k in abi.DYN_KEYS}
        return act, dyn

    def x_tm(self, lib, device):
        """The observations in the library's time-major layout: [T+1, N, d], or [S, T+1, N, d] with one set per sample."""
        st = stream_of(device)
        if not self.per_sample_data:
            return lib.pack_obs(torch.tensor(self.X, device=device), stream=st)
        return torch.stack([lib.pack_obs(torch.tensor(X, device=device), stream=st) for X in self.X])

    def lqgk_dims(self, S=None):
        """The call's dims (S systems, default the case's samples); with per-sample data, the stride between the data sets
        of x_tm(), which the workspace size depends on."""
        stride = (self.T + 1) * self.N * self.d if self.per_sample_data else 0
        return abi.LqgkDims(self.S if S is None else S, self.N, self.T, *self.dims, stride)


def workspace(lib, dims, mode, device, max_chunk=0):
    nbytes = lib.workspace_bytes(dims, mode, max_chunk)
    if nbytes == 0:
        return None
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def stream_of(device):
    return torch.cuda.current_stream(device).cuda_stream if device.type == "cuda" else 0


def rel_err(a, ref):
    return float(np.abs(a - ref).max() / (np.abs(ref).max() + 1e-300))


def check_vjp(lib, device, case: Case, dtype=torch.float32, max_chunk=0, ll_rtol=1e-4, g_rtol=1e-3):
    """Runs lqgk_loglik_vjp on `case` and compares ll and all 12 base-matrix gradients with the oracle.
    Gradient criterion: max-abs error <= g_rtol * max-abs of that matrix' oracle gradient (per sample)."""
    dims = case.lqgk_dims()
    act, dyn = case.tensors(device, dtype)
    x_tm = case.x_tm(lib, device)
    ws = workspace(lib, dims, abi.MODE_VJP, device, max_chunk)
    ll_bar = None if case.w is None else torch.tensor(case.w, dtype=dtype, device=device)
    ll, oa, od, _ = lib.loglik_vjp(dims, act, dyn, x_tm, ll_bar=ll_bar, ws=ws, stream=stream_of(device))
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    ll = ll.double().cpu().numpy()
    assert np.isfinite(ll).all()
    assert np.allclose(ll, case.ll, rtol=ll_rtol), rel_err(ll, case.ll)
    worst = 0.0
    for s in range(case.S):
        # matrices whose whole gradient is numerically zero (e.g. 1e-26) are compared on the scale of the largest gradient
        floor = 1e-9 * max(max(np.abs(case.ga[s][k]).max() for k in abi.ACTOR_KEYS), max(np.abs(case.gd[s][k]).max() for k in abi.DYN_KEYS))
        for who, keys, out, ref in (("actor", abi.ACTOR_KEYS, oa, case.ga), ("dyn", abi.DYN_KEYS, od, case.gd)):
            for k in keys:
                err = np.abs(out[k][s].double().cpu().numpy() - ref[s][k]).max()
                scale = np.abs(ref[s][k]).max()
                assert err <= g_rtol * scale + floor, (who, k, s, err, scale)
                worst = max(worst, err / (scale + floor))
    return worst


def check_vjp_tiled(lib, device, case: Case, reps: int = 1, dtype=torch.float32, ll_rtol=1e-4, g_rtol=1e-3, total=None, max_chunk=0):
    """check_vjp on `total` systems in one call (default S * reps), system k being sample k mod S of the case, with that
    sample's data set when the case has one per sample: reaches sample counts whose kernels differ from the small-batch ones
    (thread-per-sample covariance kernels above 1,024 samples; several chunks with `max_chunk`) at the oracle cost of S.
    Every system is compared with the oracle."""
    S = case.S
    total = S * reps if total is None else total
    idx = torch.arange(total, device=device) % S
    dims = case.lqgk_dims(total)
    act, dyn = case.tensors(device, dtype)
    act = {k: v[idx].contiguous() for k, v in act.items()}
    dyn = {k: v[idx].contiguous() for k, v in dyn.items()}
    x_tm = case.x_tm(lib, device)
    if case.per_sample_data:
        x_tm = x_tm[idx].contiguous()
    ws = workspace(lib, dims, abi.MODE_VJP, device, max_chunk)
    ll_bar = None if case.w is None else torch.tensor(case.w, dtype=dtype, device=device)[idx].contiguous()
    ll, oa, od, _ = lib.loglik_vjp(dims, act, dyn, x_tm, ll_bar=ll_bar, ws=ws, stream=stream_of(device))
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    ll = ll.double().cpu().numpy()
    oa = {k: v.double().cpu().numpy() for k, v in oa.items()}
    od = {k: v.double().cpu().numpy() for k, v in od.items()}
    floor = [1e-9 * max(max(np.abs(case.ga[s][k]).max() for k in abi.ACTOR_KEYS), max(np.abs(case.gd[s][k]).max() for k in abi.DYN_KEYS))
             for s in range(S)]
    for j in range(total):
        s = j % S
        assert np.allclose(ll[j], case.ll[s], rtol=ll_rtol), (j, rel_err(ll[j], case.ll[s]))
        for keys, out, ref in ((abi.ACTOR_KEYS, oa, case.ga), (abi.DYN_KEYS, od, case.gd)):
            for k in keys:
                err = np.abs(out[k][j] - ref[s][k]).max()
                assert err <= g_rtol * np.abs(ref[s][k]).max() + floor[s], (k, j, s, err)


def check_param_vjp(lib, device, case: Case, dtype=torch.float32, ll_rtol=1e-4, g_rtol=1e-3):
    """lqgk_loglik_vjp on `case`, compared with the oracle at the level BASELINE.json's tolerance is stated for: the
    gradient w.r.t. the model PARAMETERS (base-matrix cotangents chained through the constructor's Jacobian, central
    differences of the oracle's constructor).  Criterion per sample: |g - g_ref| <= g_rtol * |g_ref| + 1e-4 * max|g_ref|."""
    dims = case.lqgk_dims()
    act, dyn = case.tensors(device, dtype)
    x_tm = case.x_tm(lib, device)
    ws = workspace(lib, dims, abi.MODE_VJP, device)
    ll, oa, od, _ = lib.loglik_vjp(dims, act, dyn, x_tm, ws=ws, stream=stream_of(device))
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    assert np.allclose(ll.double().cpu().numpy(), case.ll, rtol=ll_rtol)
    names = MODEL_PARAMS[case.name.rstrip("2")]
    worst = 0.0
    for s in range(case.S):
        kw = case.params[s]
        g, g_ref = np.zeros(len(names)), np.zeros(len(names))
        for i, k in enumerate(names):
            h = 1e-6 * kw[k]
            mp, mm = model_mats(case.name, **dict(kw, **{k: kw[k] + h})), model_mats(case.name, **dict(kw, **{k: kw[k] - h}))
            for who, keys, out, ref in ((0, abi.ACTOR_KEYS, oa, case.ga), (1, abi.DYN_KEYS, od, case.gd)):
                for kk in keys:
                    J = (mp[who][kk] - mm[who][kk]) / (2 * h)
                    g[i] += float((J * out[kk][s].double().cpu().numpy()).sum())
                    g_ref[i] += float((J * ref[s][kk]).sum())
        assert np.allclose(g, g_ref, rtol=g_rtol, atol=1e-4 * np.abs(g_ref).max()), (s, g, g_ref)
        worst = max(worst, float(np.abs(g - g_ref).max() / np.abs(g_ref).max()))
    return worst


def check_fwd(lib, device, case: Case, dtype=torch.float32, max_chunk=0, ll_rtol=1e-4):
    dims = case.lqgk_dims()
    act, dyn = case.tensors(device, dtype)
    x_tm = case.x_tm(lib, device)
    ws = workspace(lib, dims, abi.MODE_FWD, device, max_chunk)
    ll = lib.loglik_fwd(dims, act, dyn, x_tm, ws=ws, stream=stream_of(device))
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    ll = ll.double().cpu().numpy()
    assert np.allclose(ll, case.ll, rtol=ll_rtol), rel_err(ll, case.ll)
    return rel_err(ll, case.ll)


def check_gains(lib, device, case: Case, dtype=torch.float64, rtol=1e-4):
    dims = case.lqgk_dims()
    act, _ = case.tensors(device, dtype)
    ws = workspace(lib, dims, abi.MODE_GAINS, device)
    L, l, H = lib.lqr_backward(dims, act, ws=ws, stream=stream_of(device))
    K = lib.kf_forward(dims, act, ws=ws, stream=stream_of(device))
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    for s, m in enumerate(case.mats):
        sa, _ = O.make_system(m, case.T)
        Lo, lo, Ho = O.lqr_backward(sa)
        Ko = O.kf_forward(sa, sa["V"][0] @ sa["V"][0].T)
        assert np.allclose(L[s].double().cpu().numpy(), Lo, rtol=rtol, atol=rtol * np.abs(Lo).max() * 1e-3)
        assert np.allclose(K[s].double().cpu().numpy(), Ko, rtol=rtol, atol=rtol * np.abs(Ko).max() * 1e-3)
        assert np.allclose(H[s].double().cpu().numpy(), Ho, rtol=rtol)
        assert np.abs(l[s].double().cpu().numpy()).max() == 0.0
