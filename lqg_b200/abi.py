"""ctypes binding of the C ABI declared in ``include/lqgk.h``.

Thin and mechanical: builds the ``LqgkDims / LqgkSpec / LqgkMat`` structs from torch tensors (pointer +
strides, no copies) and calls the entry points.  The product path loads ``liblqgk.so`` (CUDA, sm_100a) through
:func:`load_library`; there is no CPU fallback -- a missing library raises.  ``tests/`` additionally point
:class:`Library` at ``tests/emul/liblqgk_emul.so`` (the kernels' step functions compiled for the host) to check
the math without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LQGK_LIB_PATH") or os.path.join(HERE, "csrc", "liblqgk.so")   # override: tuning experiments (tools/)

MODE_GAINS, MODE_FWD, MODE_VJP, MODE_MOMENTS, MODE_GAINS_VJP = 0, 1, 2, 3, 4
ACTOR_KEYS = ("A", "B", "F", "V", "W", "Q", "R")
DYN_KEYS = ("A", "B", "F", "V", "W")


class LqgkDims(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("S", "N", "T", "x", "b", "u", "y", "d")] + [("x_sample_stride", C.c_int64)]


class LqgkMat(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("sample_stride", C.c_int64), ("time_stride", C.c_int64)]


class LqgkSpec(C.Structure):
    _fields_ = [(k, LqgkMat) for k in ("A", "B", "F", "V", "W", "Q", "R", "Qf", "q", "r", "P", "qf")]


class LqgkMatGrad(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("sample_stride", C.c_int64)]


class LqgkSpecGrad(C.Structure):
    _fields_ = [(k, LqgkMatGrad) for k in ("A", "B", "F", "V", "W", "Q", "R", "Qf")]


class LqgkError(RuntimeError):
    pass


def _mat(t: Optional[torch.Tensor], S: int, T: int, trailing: int = 2) -> LqgkMat:
    """Describe ``t`` of shape ``([S|1], [T|1], *trailing dims)`` (leading dims optional) without copying."""
    if t is None:
        return LqgkMat(None, 0, 0)
    lead = t.dim() - trailing
    if lead < 0 or lead > 2:
        raise ValueError(f"matrix with shape {tuple(t.shape)} has too many/few leading dims")
    core = t.shape[lead:]
    exp_stride, n = [], 1
    for sz in reversed(core):
        exp_stride.append(n)
        n *= sz
    if list(t.stride()[lead:]) != list(reversed(exp_stride)) and n > 1:
        raise ValueError("trailing matrix dims must be row-major contiguous")
    ss = ts = 0
    if lead == 2:
        if t.shape[0] not in (1, S) or t.shape[1] not in (1, T):
            raise ValueError(f"leading dims {tuple(t.shape[:2])} do not match (S={S}, T={T})")
        ss = t.stride(0) if t.shape[0] == S and S > 1 else 0
        ts = t.stride(1) if t.shape[1] == T and T > 1 else 0
    elif lead == 1:
        # a single leading dim is the sample axis (time-invariant per-sample matrices)
        if t.shape[0] not in (1, S):
            raise ValueError(f"leading dim {t.shape[0]} does not match S={S}")
        ss = t.stride(0) if t.shape[0] == S and S > 1 else 0
    return LqgkMat(t.data_ptr(), ss, ts)


class LqgkSdnDims(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("S", "T", "b", "u", "y", "nc", "nd", "sweeps")]


class LqgkSdnSpec(C.Structure):
    _fields_ = [(k, LqgkMat) for k in ("A", "B", "H", "C", "D", "Q", "R", "Qf", "Om_xi", "Om_omega", "Sigma1", "xhat1")]


class LqgkSdnNoise(C.Structure):
    _fields_ = [("C", LqgkMat), ("D", LqgkMat), ("nc", C.c_int32), ("nd", C.c_int32)]


class Library:
    """One loaded implementation of the C ABI."""

    def __init__(self, path: str):
        if not os.path.exists(path):
            raise LqgkError(
                f"{path} not found: the CUDA library is not built (run `python -c 'import __graft_entry__ as g; "
                f"g.build()'`).  lqg_b200 has no CPU fallback.")
        self.path = path
        self.lib = C.CDLL(path)
        self.lib.lqgk_version.restype = C.c_char_p
        if hasattr(self.lib, "lqgk_workspace_bytes"):
            self.lib.lqgk_workspace_bytes.restype = C.c_size_t
            self.lib.lqgk_workspace_bytes.argtypes = [C.POINTER(LqgkDims), C.c_int, C.c_int32]
            self.lib.lqgk_strerror.restype = C.c_char_p

    # -- helpers
    def version(self) -> str:
        return self.lib.lqgk_version().decode()

    def strerror(self, code: int) -> str:
        if hasattr(self.lib, "lqgk_strerror"):
            return self.lib.lqgk_strerror(code).decode()
        return {-1: "invalid argument", -2: "unsupported dims / time-varying VJP", -3: "workspace too small",
                -4: "CUDA error", -5: "not initialised"}.get(code, f"error {code}")

    def _check(self, code: int, what: str):
        if code != 0:
            detail = ""
            if code == -4 and hasattr(self.lib, "lqgk_last_cuda_error"):
                self.lib.lqgk_last_cuda_error.restype = C.c_char_p
                detail = ": " + self.lib.lqgk_last_cuda_error().decode()
            raise LqgkError(f"{what} failed: {self.strerror(code)} ({code}){detail}")

    def workspace_bytes(self, dims: LqgkDims, mode: int, max_chunk: int = 0) -> int:
        if not hasattr(self.lib, "lqgk_workspace_bytes"):
            return 0
        n = int(self.lib.lqgk_workspace_bytes(C.byref(dims), mode, max_chunk))
        # slack for the per-slice alignment of the internal concurrent slices (lqgk_set_streams)
        return n + n // 64 + (1 << 20) if n else 0

    @staticmethod
    def _suffix(dtype) -> str:
        return {torch.float32: "f32", torch.float64: "f64"}[dtype]

    @staticmethod
    def _spec(mats: Dict[str, torch.Tensor], S: int, T: int, keys) -> LqgkSpec:
        sp = LqgkSpec()
        for k in keys:
            setattr(sp, k, _mat(mats.get(k), S, T))
        for k in ("Qf",):
            setattr(sp, k, _mat(mats.get(k), S, 1))
        for k, tr in (("q", 1), ("r", 1), ("P", 2), ("qf", 1)):
            setattr(sp, k, _mat(mats.get(k), S, T if k != "qf" else 1, trailing=tr))
        return sp

    @staticmethod
    def _check_obs(dims, x_tm):
        """x_tm: float32 contiguous, [T+1, N, d] shared by all samples or [S, T+1, N, d] with one data set per sample;
        sets dims.x_sample_stride accordingly."""
        assert x_tm.dtype == torch.float32 and x_tm.is_contiguous()
        if x_tm.dim() == 3:
            assert tuple(x_tm.shape) == (dims.T + 1, dims.N, dims.d), tuple(x_tm.shape)
            dims.x_sample_stride = 0
        else:
            assert tuple(x_tm.shape) == (dims.S, dims.T + 1, dims.N, dims.d), tuple(x_tm.shape)
            dims.x_sample_stride = x_tm.stride(0)

    @staticmethod
    def _ws(ws: Optional[torch.Tensor]):
        return (ws.data_ptr(), ws.numel() * ws.element_size()) if ws is not None else (None, 0)

    # -- entry points
    def lqr_backward(self, dims, actor, eps=1e-8, want_l=True, want_H=True, ws=None, stream=0):
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T = dims.S, dims.T
        L = torch.empty((S, T, dims.u, dims.b), dtype=dt, device=dev)
        l = torch.empty((S, T, dims.u), dtype=dt, device=dev) if want_l else None
        H = torch.empty((S, T, dims.u, dims.u), dtype=dt, device=dev) if want_H else None
        sp = self._spec(actor, S, T, ACTOR_KEYS)
        p, n = self._ws(ws)
        fn = getattr(self.lib, "lqgk_lqr_backward_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sp), C.c_double(eps), C.c_void_p(L.data_ptr()),
                       C.c_void_p(l.data_ptr() if want_l else None), C.c_void_p(H.data_ptr() if want_H else None),
                       C.c_void_p(p), C.c_size_t(n), C.c_void_p(stream)), "lqgk_lqr_backward")
        return L, l, H

    def kf_forward(self, dims, actor, sigma0=None, ws=None, stream=0):
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T = dims.S, dims.T
        K = torch.empty((S, T, dims.b, dims.y), dtype=dt, device=dev)
        sp = self._spec(actor, S, T, ACTOR_KEYS)
        s0 = _mat(sigma0, S, 1) if sigma0 is not None else None
        p, n = self._ws(ws)
        fn = getattr(self.lib, "lqgk_kf_forward_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sp), C.byref(s0) if s0 is not None else None,
                       C.c_void_p(K.data_ptr()), C.c_void_p(p), C.c_size_t(n), C.c_void_p(stream)), "lqgk_kf_forward")
        return K

    def gains_vjp(self, dims, actor, sigma0=None, eps=1e-8, L_bar=None, K_bar=None, want=ACTOR_KEYS, ws=None, stream=0):
        """Gradients of <L_bar, L> + <K_bar, K> (lqr_backward's L, kf_forward's K; either cotangent may be None, not both)
        with respect to the actor's base matrices: ({name: [S, r, c]} for the names in `want` -- ACTOR_KEYS and "Qf" --, the
        gradient of sigma0 [S, b, b] or None).  actor: time-invariant base matrices as for loglik_vjp."""
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T = dims.S, dims.T
        sp = self._spec(actor, S, T, ACTOR_KEYS)
        s0 = _mat(sigma0, S, 1) if sigma0 is not None else None
        shp = dict(A=(dims.b, dims.b), B=(dims.b, dims.u), F=(dims.y, dims.b), V=(dims.b, dims.b), W=(dims.y, dims.y),
                   Q=(dims.b, dims.b), R=(dims.u, dims.u), Qf=(dims.b, dims.b))
        ga, out = LqgkSpecGrad(), {}
        for k in want:
            out[k] = torch.empty((S,) + shp[k], dtype=dt, device=dev)
            setattr(ga, k, LqgkMatGrad(out[k].data_ptr(), out[k].stride(0)))
        gs0, out_s0 = None, None
        if sigma0 is not None:
            out_s0 = torch.empty((S, dims.b, dims.b), dtype=dt, device=dev)
            gs0 = LqgkMatGrad(out_s0.data_ptr(), out_s0.stride(0))
        keep = [None if v is None else v.to(dt).contiguous() for v in (L_bar, K_bar)]
        for v, shape in zip(keep, ((S, T, dims.u, dims.b), (S, T, dims.b, dims.y))):
            assert v is None or tuple(v.shape) == shape, (tuple(v.shape), shape)
        p, n = self._ws(ws)
        fn = getattr(self.lib, "lqgk_gains_vjp_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sp), C.byref(s0) if s0 is not None else None, C.c_double(eps),
                       C.c_void_p(keep[0].data_ptr() if keep[0] is not None else None),
                       C.c_void_p(keep[1].data_ptr() if keep[1] is not None else None), C.byref(ga),
                       C.byref(gs0) if gs0 is not None else None, C.c_void_p(p), C.c_size_t(n), C.c_void_p(stream)),
                    "lqgk_gains_vjp")
        return out, out_s0

    def loglik_fwd(self, dims, actor, dyn, x_tm, sigma0=None, ws=None, stream=0):
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T = dims.S, dims.T
        self._check_obs(dims, x_tm)
        ll = torch.empty((S, dims.N), dtype=dt, device=dev)
        sa, sd = self._spec(actor, S, T, ACTOR_KEYS), self._spec(dyn, S, T, DYN_KEYS)
        s0 = _mat(sigma0, S, 1) if sigma0 is not None else None
        p, n = self._ws(ws)
        fn = getattr(self.lib, "lqgk_loglik_fwd_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sa), C.byref(sd), C.byref(s0) if s0 is not None else None,
                       C.c_void_p(x_tm.data_ptr()), C.c_void_p(ll.data_ptr()), C.c_void_p(p), C.c_size_t(n),
                       C.c_void_p(stream)), "lqgk_loglik_fwd")
        return ll

    def loglik_vjp(self, dims, actor, dyn, x_tm, ll_bar=None, sigma0=None, want_actor=ACTOR_KEYS, want_dyn=DYN_KEYS,
                   want_qf=False, ws=None, stream=0):
        """Returns ll[S,N], grads_actor{name: [S,r,c]}, grads_dyn{...}, grad_sigma0 or None."""
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T = dims.S, dims.T
        self._check_obs(dims, x_tm)
        ll = torch.empty((S, dims.N), dtype=dt, device=dev)
        sa, sd = self._spec(actor, S, T, ACTOR_KEYS), self._spec(dyn, S, T, DYN_KEYS)
        s0 = _mat(sigma0, S, 1) if sigma0 is not None else None
        shp_a = dict(A=(dims.b, dims.b), B=(dims.b, dims.u), F=(dims.y, dims.b), V=(dims.b, dims.b),
                     W=(dims.y, dims.y), Q=(dims.b, dims.b), R=(dims.u, dims.u), Qf=(dims.b, dims.b))
        shp_d = dict(A=(dims.x, dims.x), B=(dims.x, dims.u), F=(dims.y, dims.x), V=(dims.x, dims.x), W=(dims.y, dims.y))
        ga, gd = LqgkSpecGrad(), LqgkSpecGrad()
        out_a, out_d = {}, {}
        for k in list(want_actor) + (["Qf"] if want_qf else []):
            out_a[k] = torch.empty((S,) + shp_a[k], dtype=dt, device=dev)
            setattr(ga, k, LqgkMatGrad(out_a[k].data_ptr(), out_a[k].stride(0)))
        for k in want_dyn:
            out_d[k] = torch.empty((S,) + shp_d[k], dtype=dt, device=dev)
            setattr(gd, k, LqgkMatGrad(out_d[k].data_ptr(), out_d[k].stride(0)))
        gs0, out_s0 = None, None
        if sigma0 is not None:
            out_s0 = torch.empty((S, dims.b, dims.b), dtype=dt, device=dev)
            gs0 = LqgkMatGrad(out_s0.data_ptr(), out_s0.stride(0))
        if ll_bar is not None:
            ll_bar = ll_bar.to(dt).expand(S, dims.N).contiguous()
        p, n = self._ws(ws)
        fn = getattr(self.lib, "lqgk_loglik_vjp_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sa), C.byref(sd), C.byref(s0) if s0 is not None else None,
                       C.c_void_p(x_tm.data_ptr()), C.c_void_p(ll_bar.data_ptr() if ll_bar is not None else None),
                       C.c_void_p(ll.data_ptr()), C.byref(ga), C.byref(gd), C.byref(gs0) if gs0 is not None else None,
                       C.c_void_p(p), C.c_size_t(n), C.c_void_p(stream)), "lqgk_loglik_vjp")
        return ll, out_a, out_d, out_s0

    def moments(self, dims, actor, dyn, x_tm, sigma0=None, want_mu=True, want_sigma=True, ws=None, stream=0):
        """Predictive moments of the joint state (x, xhat): mu[S, N, T, n], Sigma[S, T, n, n] (None when not wanted)."""
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T, n = dims.S, dims.T, dims.x + dims.b
        self._check_obs(dims, x_tm)
        mu = torch.empty((S, dims.N, T, n), dtype=dt, device=dev) if want_mu else None
        Sig = torch.empty((S, T, n, n), dtype=dt, device=dev) if want_sigma else None
        sa, sd = self._spec(actor, S, T, ACTOR_KEYS), self._spec(dyn, S, T, DYN_KEYS)
        s0 = _mat(sigma0, S, 1) if sigma0 is not None else None
        p, nb = self._ws(ws)
        fn = getattr(self.lib, "lqgk_moments_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sa), C.byref(sd), C.byref(s0) if s0 is not None else None,
                       C.c_void_p(x_tm.data_ptr()), C.c_void_p(mu.data_ptr() if want_mu else None),
                       C.c_void_p(Sig.data_ptr() if want_sigma else None), C.c_void_p(p), C.c_size_t(nb), C.c_void_p(stream)),
                    "lqgk_moments")
        return mu, Sig

    def _noise(self, dims, dt, C_noise, D_noise, keep):
        """LqgkSdnNoise from C_noise[S?, nc, x, u], D_noise[S?, nd, y, x] (None = none); tensors kept alive in `keep`."""
        nz = LqgkSdnNoise()
        for name, v, shp in (("C", C_noise, (dims.x, dims.u)), ("D", D_noise, (dims.y, dims.x))):
            if v is None or v.numel() == 0:   # (a fresh structure is zero: no matrix, no terms)
                continue
            v = v.to(dt).contiguous()
            keep.append(v)
            assert tuple(v.shape[-2:]) == shp and v.dim() in (3, 4), (name, tuple(v.shape))
            setattr(nz, name, _mat(v, dims.S, 1, trailing=3))
            setattr(nz, "n" + name.lower(), v.shape[-3])
        return nz

    def simulate(self, dims, actor, dyn, L, l, K, seed, x0=None, xhat0=None, return_all=False, stream=0, C_noise=None, D_noise=None):
        """Batched System.simulate: x[S, N, T+1, x] (and xhat, y, u when return_all) for the given gains.  C_noise / D_noise:
        multiplicative-noise matrices of the signal-dependent-noise extension (lqgk_sdn_simulate_*)."""
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T, N = dims.S, dims.T, dims.N
        x = torch.empty((S, N, T + 1, dims.x), dtype=dt, device=dev)
        xh = torch.empty((S, N, T + 1, dims.b), dtype=dt, device=dev) if return_all else None
        y = torch.empty((S, N, T, dims.y), dtype=dt, device=dev) if return_all else None
        u = torch.empty((S, N, T, dims.u), dtype=dt, device=dev) if return_all else None
        sa, sd = self._spec(actor, S, T, ACTOR_KEYS), self._spec(dyn, S, T, DYN_KEYS)
        keep = [t.to(dt).contiguous() if t is not None else None for t in (L, l, K, x0, xhat0)]
        ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else None)
        tail = (ptr(keep[0]), ptr(keep[1]), ptr(keep[2]), ptr(keep[3]), ptr(keep[4]), C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF),
                ptr(x), ptr(xh), ptr(y), ptr(u), C.c_void_p(stream))
        if C_noise is None and D_noise is None:
            fn = getattr(self.lib, "lqgk_simulate_" + self._suffix(dt))
            self._check(fn(C.byref(dims), C.byref(sa), C.byref(sd), *tail), "lqgk_simulate")
        else:
            nz = self._noise(dims, dt, C_noise, D_noise, keep)
            fn = getattr(self.lib, "lqgk_sdn_simulate_" + self._suffix(dt))
            self._check(fn(C.byref(dims), C.byref(sa), C.byref(sd), C.byref(nz), *tail), "lqgk_sdn_simulate")
        return (x, xh, y, u) if return_all else x

    def pack_obs(self, x: torch.Tensor, stream=0) -> torch.Tensor:
        """x[N, T+1, d] (f32/f64) -> time-major float32 x_tm[T+1, N, d] on the same device."""
        N, T1, d = x.shape
        x = x.contiguous()
        out = torch.empty((T1, N, d), dtype=torch.float32, device=x.device)
        fn = getattr(self.lib, "lqgk_pack_obs_" + self._suffix(x.dtype))
        self._check(fn(C.c_int32(N), C.c_int32(T1), C.c_int32(d), C.c_void_p(x.data_ptr()),
                       C.c_void_p(out.data_ptr()), C.c_void_p(stream)), "lqgk_pack_obs")
        return out

    def last_launch_count(self) -> int:
        return int(self.lib.lqgk_last_launch_count())

    PROFILE_KINDS = ("pack", "lqr_fwd", "kf_fwd", "cov_fwd", "trial_fwd", "misc", "trial_rev", "cov_rev", "kf_rev",
                     "lqr_rev", "unpack", "cov_contrib", "reduce")

    def sdn_gains(self, mats: Dict[str, torch.Tensor], T: int, sweeps: int = 10, stream=0, filter_form: bool = False):
        """Signal-dependent-noise gains (extension, include/lqgk.h).  mats: float64 CUDA tensors A[S?,b,b], B[S?,b,u],
        H[S?,y,b], C[S?,nc,b,u], D[S?,nd,y,b], Q, R, (Qf), Om_xi, Om_omega, Sigma1, xhat1[S?,b]; a leading sample axis is
        optional per tensor (absent / size 1 = shared).  Returns L[S,T,u,b], K[S,T,b,y], cost[S]."""
        A, Bm, H = mats["A"], mats["B"], mats["H"]
        b, u, y = A.shape[-1], Bm.shape[-1], H.shape[-2]
        base_nd = dict(A=2, B=2, H=2, C=3, D=3, Q=2, R=2, Qf=2, Om_xi=2, Om_omega=2, Sigma1=2, xhat1=1)
        S = 1
        for k, v in mats.items():
            if v is not None and v.dim() == base_nd[k] + 1:
                S = max(S, v.shape[0])
        sp = LqgkSdnSpec()
        keep = []
        for k in base_nd:
            v = mats.get(k)
            if v is None or v.numel() == 0:
                continue
            assert v.dtype == torch.float64 and (v.is_cuda or not hasattr(self.lib, "lqgk_init")), k   # (host tensors: test harness only)
            v = v.contiguous()
            keep.append(v)
            setattr(sp, k, _mat(v, S, 1, trailing=base_nd[k]))
        nc = 0 if mats.get("C") is None else mats["C"].shape[-3]
        nd = 0 if mats.get("D") is None else mats["D"].shape[-3]
        dims = LqgkSdnDims(S, T, b, u, y, nc, nd, sweeps)
        dev = A.device
        L = torch.empty((S, T, u, b), dtype=torch.float64, device=dev)
        K = torch.zeros((S, T, b, y), dtype=torch.float64, device=dev)   # sweeps = 0 leaves K = 0 (the iterations' starting point)
        cost = torch.empty((S,), dtype=torch.float64, device=dev)
        fn = self.lib.lqgk_sdn_gains_filter_f64 if filter_form else self.lib.lqgk_sdn_gains_f64
        rc = fn(C.byref(dims), C.byref(sp), C.c_void_p(L.data_ptr()), C.c_void_p(K.data_ptr()), C.c_void_p(cost.data_ptr()),
                C.c_void_p(stream))
        self._check(rc, "lqgk_sdn_gains" + ("_filter" if filter_form else "") + "_f64")
        return L, K, cost

    def sdn_loglik(self, dims, actor, dyn, L, K, x_tm, C_noise=None, D_noise=None, stream=0):
        """Log-likelihood under signal-dependent noise (extension, include/lqgk.h: lqgk_sdn_loglik_*).  actor / dyn: base
        matrices as for loglik_fwd (time-invariant), L[S,T,u,b], K[S,T,b,y]: gains, C_noise[S?,nc,x,u], D_noise[S?,nd,y,x]:
        multiplicative-noise matrices (None = none; a leading sample axis is optional).  Returns ll[S,N]."""
        dt, dev = actor["A"].dtype, actor["A"].device
        S, T = dims.S, dims.T
        self._check_obs(dims, x_tm)
        sa, sd = self._spec(actor, S, T, ACTOR_KEYS), self._spec(dyn, S, T, DYN_KEYS)
        keep = [L.to(dt).contiguous(), K.to(dt).contiguous()]
        assert tuple(keep[0].shape) == (S, T, dims.u, dims.b) and tuple(keep[1].shape) == (S, T, dims.b, dims.y)
        nz = self._noise(dims, dt, C_noise, D_noise, keep)
        ll = torch.empty((S, dims.N), dtype=dt, device=dev)
        fn = getattr(self.lib, "lqgk_sdn_loglik_" + self._suffix(dt))
        self._check(fn(C.byref(dims), C.byref(sa), C.byref(sd), C.byref(nz), C.c_void_p(keep[0].data_ptr()),
                       C.c_void_p(keep[1].data_ptr()), C.c_void_p(x_tm.data_ptr()), C.c_void_p(ll.data_ptr()),
                       C.c_void_p(stream)), "lqgk_sdn_loglik")
        return ll

    def init(self, max_sample_slices: int = 1):
        """Pre-create the library's internal streams / events (needed before capturing calls into a CUDA graph)."""
        self._check(self.lib.lqgk_init(C.c_int(int(max_sample_slices))), "lqgk_init")

    def set_streams(self, n: int):
        self._check(self.lib.lqgk_set_streams(C.c_int(n)), "lqgk_set_streams")

    def set_warp_cov_max_samples(self, n: int):
        self._check(self.lib.lqgk_set_warp_cov_max_samples(C.c_int(int(n))), "lqgk_set_warp_cov_max_samples")

    def set_pipeline(self, max_samples: int, segments: int = 6):
        self._check(self.lib.lqgk_set_pipeline(C.c_int(int(max_samples)), C.c_int(int(segments))), "lqgk_set_pipeline")

    def set_kernel_overlap(self, mask: int):
        self._check(self.lib.lqgk_set_kernel_overlap(C.c_int(int(mask))), "lqgk_set_kernel_overlap")

    def profile_enable(self, on: bool):
        self._check(self.lib.lqgk_profile_enable(C.c_int(1 if on else 0)), "lqgk_profile_enable")

    def profile_read(self):
        """{kind: (milliseconds, launches)} accumulated since the last read (synchronises on the recorded events)."""
        n = len(self.PROFILE_KINDS)
        ms = (C.c_float * n)()
        cnt = (C.c_int32 * n)()
        rc = self.lib.lqgk_profile_read(ms, cnt, C.c_int(n))
        if rc < 0:
            self._check(rc, "lqgk_profile_read")
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROFILE_KINDS)}

    def profile_timeline(self, max_entries=4096):
        """[(kind, start_ms, end_ms)] of every launch recorded since the last profile_read."""
        st = (C.c_float * max_entries)()
        en = (C.c_float * max_entries)()
        kd = (C.c_int32 * max_entries)()
        n = self.lib.lqgk_profile_timeline(st, en, kd, C.c_int(max_entries))
        if n < 0:
            self._check(n, "lqgk_profile_timeline")
        return [(self.PROFILE_KINDS[kd[i]], float(st[i]), float(en[i])) for i in range(n)]

    def peak_fma(self, fp64: bool, device, iters=4096, reps=5) -> float:
        """Measured CUDA-core FMA peak in TFLOP/s (best of `reps`), CUDA events on the current stream."""
        sink = torch.zeros(8, dtype=torch.float64, device=device)
        st = torch.cuda.current_stream(device).cuda_stream
        flop = C.c_double(0.0)
        best = 0.0
        for r in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self._check(self.lib.lqgk_peak_fma(C.c_int(1 if fp64 else 0), C.c_int(iters), C.c_void_p(sink.data_ptr()),
                                               C.c_void_p(st), C.byref(flop)), "lqgk_peak_fma")
            e1.record()
            e1.synchronize()
            if r > 0:
                best = max(best, flop.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        return best


_LIB: Optional[Library] = None


def load_library() -> Library:
    """The product library (CUDA).  Raises if it has not been built -- there is no fallback."""
    global _LIB
    if _LIB is None:
        _LIB = Library(LIB_PATH)
    return _LIB
