"""Host-side glue between the torch-facing API (``lqg_b200.system`` etc.) and the C ABI (``lqg_b200.abi``).

* canonicalises ``LQGSpec`` tensors to the ``(S, T, r, c)`` views the ABI describes by strides (no copies for
  stride-0 time axes / shared samples);
* owns one cached device workspace per GPU, sized by :data:`WORKSPACE_FRACTION` of free memory (the library
  chunks over parameter samples inside that budget);
* wraps the fused forward+adjoint entry point in a ``torch.autograd.Function`` (the reference gets its
  gradient from ``jax.value_and_grad``; here the CUDA adjoint is the ``backward``).

There is no CPU path: every function raises if the tensors are not on a CUDA device or the library is missing.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from lqg_b200 import abi
from lqg_b200.dims import FP64_ONLY_DIMS, SUPPORTED_DIMS
from lqg_b200.spec import LQGSpec

WORKSPACE_FRACTION = 0.85         # of currently free device memory, upper bound for the cached workspace
WORKSPACE_MAX_BYTES = 150 << 30   # B200: 180 GB HBM3e; more samples in flight = better latency hiding in the per-sample kernels
_WS: Dict[int, torch.Tensor] = {}

ACT_KEYS = abi.ACTOR_KEYS
DYN_KEYS = abi.DYN_KEYS


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"lqg_b200: {what} must live on a CUDA device (got {t.device}); there is no CPU fallback. "
                           f"Move the model/data to 'cuda' (B200, sm_100a).")


def workspace(device: torch.device, need: int) -> torch.Tensor:
    """Cached uint8 workspace on `device`, at least min(need, budget) bytes."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    cur = _WS.get(idx)
    if cur is not None and cur.numel() >= need:
        return cur
    free, _total = torch.cuda.mem_get_info(idx)
    have = cur.numel() if cur is not None else 0
    budget = min(int((free + have) * WORKSPACE_FRACTION), WORKSPACE_MAX_BYTES)
    size = min(need, budget)
    if cur is not None and cur.numel() >= size:
        return cur
    _WS.pop(idx, None)
    del cur
    _WS[idx] = torch.empty(size, dtype=torch.uint8, device=torch.device("cuda", idx))
    return _WS[idx]


def release_workspace():
    _WS.clear()


def spec_batch(spec: LQGSpec) -> Tuple[int, int]:
    """(S, T) of a spec whose arrays are (T, r, c) or (S, T, r, c)."""
    A = spec.A
    if A.dim() == 3:
        return 1, A.shape[0]
    if A.dim() == 4:
        return A.shape[0], A.shape[1]
    raise ValueError(f"spec arrays must be (T, r, c) or (S, T, r, c); got {tuple(A.shape)}")


def _as4(M: torch.Tensor) -> torch.Tensor:
    return M if M.dim() == 4 else M.unsqueeze(0)


def _row_major(M: torch.Tensor) -> torch.Tensor:
    """Make the trailing matrix dims row-major contiguous without materialising stride-0 leading axes."""
    r, c = M.shape[-2:]
    if M.stride(-1) == 1 and (M.stride(-2) == c or r == 1):
        return M
    lead = M.shape[:-2]
    # collapse expanded (stride-0) leading dims before copying, then expand again
    idx = tuple(slice(0, 1) if (M.stride(i) == 0 and M.shape[i] > 1) else slice(None) for i in range(len(lead)))
    return M[idx].contiguous().expand(*lead, r, c)


def _vec_rows(v: torch.Tensor) -> torch.Tensor:
    """(S|1, T, k) vectors with a contiguous last axis, keeping stride-0 leading axes un-materialised."""
    if v.stride(-1) == 1 or v.shape[-1] == 1:
        return v
    idx = tuple(slice(0, 1) if (v.stride(i) == 0 and v.shape[i] > 1) else slice(None) for i in range(v.dim() - 1))
    return v[idx].contiguous().expand(*v.shape)


def spec_mats(spec: LQGSpec, keys) -> Dict[str, torch.Tensor]:
    return {k: _row_major(_as4(getattr(spec, k))) for k in keys}


def _untimed(M: torch.Tensor, dt) -> torch.Tensor:
    """(S|1, r, c) row-major in dtype dt from a matrix without time axis (Qf, Sigma0) shaped (r, c) or (S, r, c)."""
    return _row_major(M if M.dim() == 3 else M.unsqueeze(0)).to(dt)


def _per_sample(t: Optional[torch.Tensor], nd: int, S: int, dt) -> Optional[torch.Tensor]:
    """Gains with an optional leading sample axis (nd dims without it) -> (S, ...) contiguous."""
    if t is None:
        return None
    t = t if t.dim() == nd + 1 else t.unsqueeze(0)
    return t.expand(S, *t.shape[1:]).to(dt).contiguous()


def _unbatch(actor: LQGSpec, dynamics: LQGSpec, out):
    """Drops the sample axis of a call's output(s) (a tensor, or a tuple of tensors and Nones) for an un-batched model."""
    if not (actor.A.dim() == 3 and dynamics.A.dim() == 3):
        return out
    return tuple(o[0] if o is not None else None for o in out) if isinstance(out, tuple) else out[0]


def is_time_invariant(M4: torch.Tensor) -> bool:
    return M4.shape[1] == 1 or M4.stride(1) == 0


def dims_of(actor: LQGSpec, dynamics: LQGSpec, N: int, d: int) -> abi.LqgkDims:
    Sa, T = spec_batch(actor)
    Sd, Td = spec_batch(dynamics)
    if T != Td:
        raise ValueError("actor and dynamics specs have different numbers of time steps")
    if Sa != Sd and 1 not in (Sa, Sd):
        raise ValueError("actor and dynamics specs have incompatible sample axes")
    S = max(Sa, Sd)
    x, b = dynamics.A.shape[-1], actor.A.shape[-1]
    u, y = dynamics.B.shape[-1], dynamics.F.shape[-2]
    return abi.LqgkDims(S, N, T, x, b, u, y, d)


def check_supported(dims: abi.LqgkDims, gains_only=False):
    tup = (dims.x, dims.b, dims.u, dims.y, dims.d)
    if gains_only:
        if not any(t[:4] == tup[:4] for t in SUPPORTED_DIMS):
            raise NotImplementedError(f"lqg_b200: no kernels compiled for (x,b,u,y)={tup[:4]}; add a line to csrc/lqgk_dims.h")
    elif tup not in SUPPORTED_DIMS:
        raise NotImplementedError(f"lqg_b200: no kernels compiled for (x,b,u,y,d)={tup}; supported: {SUPPORTED_DIMS}. "
                                  f"Add a line to lqg_b200/csrc/lqgk_dims.h and rebuild.")


def _stream(device):
    return torch.cuda.current_stream(device).cuda_stream


def _gains_dims(spec: LQGSpec) -> abi.LqgkDims:
    """Dimensions of a gains-only call.  The sweeps read the actor's (b, u, y) only: x and d are those of the first compiled
    tuple with that (b, u, y), or (b, 1) when there is none (check_supported then refuses the call)."""
    S, T = spec_batch(spec)
    b, u, y = spec.A.shape[-1], spec.B.shape[-1], spec.F.shape[-2]
    x, d = next(((t[0], t[4]) for t in SUPPORTED_DIMS if t[1:4] == (b, u, y)), (b, 1))
    return abi.LqgkDims(S, 1, T, x, b, u, y, d)


def _gains_call(spec: LQGSpec):
    """What lqr_backward and kf_forward share: the library, the dimensions, the actor's matrices and the workspace."""
    _require_cuda(spec.A, "spec")
    lib = abi.load_library()
    dims = _gains_dims(spec)
    check_supported(dims, gains_only=True)
    ws = workspace(spec.A.device, lib.workspace_bytes(dims, abi.MODE_GAINS, 0))
    return lib, dims, spec_mats(spec, ACT_KEYS), ws


def _grad_wanted(*ts) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)


def _gains_bases(spec: LQGSpec, mats: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """``mats`` with the actor's seven matrices replaced by their (S|1, r, c) base matrices, taken from the spec through
    differentiable views.  The library sees the same pointers and strides (a time-invariant array has a stride-0 time axis),
    so the gains call is the same; the gradient of a base matrix flows back to the spec's array by autograd."""
    out = dict(mats)
    for k in ACT_KEYS:
        M4 = _as4(getattr(spec, k))
        if not is_time_invariant(M4):
            raise NotImplementedError(
                "lqg_b200: gradients of lqr.backward / kf.forward are implemented for time-invariant specs (stride-0 time "
                "axis, as built by lqg_b200.utils.time_stack); materialised time-varying arrays only support the forward pass.")
        out[k] = _row_major(M4[:, 0])
    return out


class _GainsFn(torch.autograd.Function):
    """The gains of one sweep with the CUDA adjoint (lqgk_gains_vjp_*) as backward: ``kind`` "lqr" returns lqr_backward's
    (L, l, H), "kf" kf_forward's K.  The forward is the gains call itself.

    ``fixed``: what the call reads that is not differentiated; ``names``: the keys of the differentiable inputs ``mats`` --
    (S|1, r, c) base matrices: A, B, Q, R and Qf for the Riccati sweep, A, F, V, W and Sigma0 for the Kalman sweep.  ``l`` and
    ``H`` are not differentiable: ``l`` is zero in every reference model (no affine cost terms) and ``H`` is a by-product."""

    @staticmethod
    def forward(ctx, kind, dims, eps, fixed, names, *mats):
        lib = abi.load_library()
        act = {**fixed, **dict(zip(names, mats))}
        sigma0 = act.pop("Sigma0", None)
        dev = act["A"].device
        ws = workspace(dev, lib.workspace_bytes(dims, abi.MODE_GAINS, 0))
        ctx.kind, ctx.dims, ctx.eps, ctx.names = kind, dims, eps, names
        ctx.act, ctx.sigma0 = act, sigma0
        ctx.shapes = [m.shape for m in mats]
        if kind == "kf":
            return lib.kf_forward(dims, act, sigma0=sigma0, ws=ws, stream=_stream(dev))
        L, l, H = lib.lqr_backward(dims, act, eps=eps, ws=ws, stream=_stream(dev))
        ctx.mark_non_differentiable(l, H)
        return L, l, H

    @staticmethod
    def backward(ctx, bar, *_l_H_bar):
        if bar is None:
            return (None,) * (5 + len(ctx.shapes))
        lib = abi.load_library()
        dev = bar.device
        ws = workspace(dev, lib.workspace_bytes(ctx.dims, abi.MODE_GAINS_VJP, 0))
        act = {k: ctx.act[k] for k in ACT_KEYS + ("Qf",) if k in ctx.act}   # (the adjoint reads no affine terms)
        g, gs = lib.gains_vjp(ctx.dims, act, sigma0=ctx.sigma0, eps=ctx.eps, L_bar=bar if ctx.kind == "lqr" else None,
                              K_bar=bar if ctx.kind == "kf" else None, want=[k for k in ctx.names if k != "Sigma0"], ws=ws,
                              stream=_stream(dev))
        g["Sigma0"] = gs
        # the kernels sum over time; an input shared by the samples (leading 1) gets the sum over samples
        out = [g[k].sum(0, keepdim=True) if (shp[0] == 1 and g[k].shape[0] != 1) else g[k] for k, shp in zip(ctx.names, ctx.shapes)]
        return (None,) * 5 + tuple(out)


def lqr_backward(spec: LQGSpec, eps: float = 1e-8):
    """CUDA backward Riccati sweep.  Returns L, l, H shaped like the reference ((T,u,b) or (S,T,u,b)).

    L is differentiable with respect to the spec's A, B, Q, R and Qf (time-invariant specs without a cross cost P); l and H
    are not."""
    lib, dims, mats, ws = _gains_call(spec)
    # affine terms are always handed to the kernel (zeros in every reference model): no host-side "is it zero?" sync
    for k, tr in (("q", 1), ("r", 1), ("P", 2)):
        v = getattr(spec, k)
        if v is not None:
            v = v if v.dim() == tr + 2 else v.unsqueeze(0)
            mats[k] = _row_major(v) if tr == 2 else _vec_rows(v)
    if spec.qf is not None:
        mats["qf"] = (spec.qf if spec.qf.dim() == 2 else spec.qf.unsqueeze(0)).contiguous()
    if spec.Qf is not None:
        mats["Qf"] = _untimed(spec.Qf, spec.A.dtype)
    if _grad_wanted(spec.A, spec.B, spec.Q, spec.R, spec.Qf):
        _check_no_cross_cost(spec)
        mats = _gains_bases(spec, mats)
        names = ("A", "B", "Q", "R") + (("Qf",) if "Qf" in mats else ())
        fixed = {k: v for k, v in mats.items() if k not in names}
        L, l, H = _GainsFn.apply("lqr", dims, eps, fixed, names, *(mats[k] for k in names))
    else:
        L, l, H = lib.lqr_backward(dims, mats, eps=eps, ws=ws, stream=_stream(spec.A.device))
    if spec.A.dim() == 3:
        L, l, H = L[0], l[0], H[0]
    return L, l, H


def kf_forward(spec: LQGSpec, Sigma0: Optional[torch.Tensor]):
    """CUDA forward Kalman-gain sweep.  Returns K shaped (T,b,y) or (S,T,b,y).

    K is differentiable with respect to the spec's A, F, V, W and Sigma0 (time-invariant specs)."""
    lib, dims, mats, ws = _gains_call(spec)
    s0 = None if Sigma0 is None else _untimed(Sigma0, spec.A.dtype)
    if _grad_wanted(spec.A, spec.F, spec.V, spec.W, Sigma0):
        mats = _gains_bases(spec, mats)
        names = ("A", "F", "V", "W") + (("Sigma0",) if s0 is not None else ())
        mats["Sigma0"] = s0
        fixed = {k: v for k, v in mats.items() if k not in names}
        K = _GainsFn.apply("kf", dims, 0.0, fixed, names, *(mats[k] for k in names))
    else:
        K = lib.kf_forward(dims, mats, sigma0=s0, ws=ws, stream=_stream(spec.A.device))
    return K[0] if spec.A.dim() == 3 else K


class _LogLikFn(torch.autograd.Function):
    """ll[S, N] = log p(x_{1:T} | x_0, theta) per parameter sample and trial, with the CUDA adjoint as backward.

    When any input requires grad the forward runs the *fused* forward+adjoint entry point with unit cotangents and
    caches the per-sample gradients; ``backward`` rescales them when the incoming cotangent is constant over the
    trials of each sample (the usual ``ll.sum()`` / per-sample weighting) and otherwise re-runs the adjoint with the
    actual per-trial cotangents.

    ``mats`` = the 7 actor base matrices, the 5 dynamics base matrices, then optionally ``Qf`` and ``Sigma0``.
    """

    @staticmethod
    def forward(ctx, x_tm, dims, has_qf, has_sigma0, n_act, *mats):
        lib = abi.load_library()
        act = dict(zip(ACT_KEYS, mats[:n_act]))
        dyn = dict(zip(DYN_KEYS, mats[n_act:n_act + len(DYN_KEYS)]))
        extra = list(mats[n_act + len(DYN_KEYS):])
        if has_qf:
            act["Qf"] = extra.pop(0)
        sigma0 = extra.pop(0) if has_sigma0 else None
        dev = x_tm.device
        need_grad = any(m.requires_grad for m in mats)
        ctx.need_grad = need_grad
        if not need_grad:
            ws = workspace(dev, lib.workspace_bytes(dims, abi.MODE_FWD, 0))
            return lib.loglik_fwd(dims, act, dyn, x_tm, sigma0=sigma0, ws=ws, stream=_stream(dev))
        for m in mats[:n_act + len(DYN_KEYS)]:
            if m.requires_grad and m.dim() == 4:
                raise NotImplementedError(
                    "lqg_b200: gradients are implemented for time-invariant specs (stride-0 time axis, as built by "
                    "lqg_b200.utils.time_stack); materialised time-varying arrays only support the forward pass.")
        ws = workspace(dev, lib.workspace_bytes(dims, abi.MODE_VJP, 0))
        ll, ga, gd, gs = lib.loglik_vjp(dims, act, dyn, x_tm, sigma0=sigma0, want_qf=has_qf, ws=ws, stream=_stream(dev))
        ctx.args = (x_tm, dims, act, dyn, sigma0)
        ctx.cached = (ga, gd, gs)
        ctx.shapes = [m.shape for m in mats]
        ctx.n_act = n_act
        ctx.has_qf, ctx.has_sigma0 = has_qf, has_sigma0
        return ll

    @staticmethod
    def backward(ctx, ll_bar):
        if not ctx.need_grad:
            return (None,) * (5 + len(ctx.shapes))
        x_tm, dims, act, dyn, sigma0 = ctx.args
        ga, gd, gs = ctx.cached
        ll_bar = ll_bar.expand(dims.S, dims.N)
        row = ll_bar[:, :1]
        # A cotangent that is constant over the trials of each sample (what `.sum()` / `.sum(-1)` / per-sample weights
        # produce: autograd hands it over as an expanded, stride-0 view) only rescales the cached unit-cotangent gradients.
        # Decided from the strides, never from the values: no host synchronisation on the autograd path.
        if dims.N == 1 or ll_bar.stride(-1) == 0:
            scale = row.reshape(dims.S, 1, 1).to(next(iter(ga.values())).dtype)
            ga = {k: v * scale for k, v in ga.items()}
            gd = {k: v * scale for k, v in gd.items()}
            gs = gs * scale if gs is not None else None
        else:
            lib = abi.load_library()
            dev = x_tm.device
            ws = workspace(dev, lib.workspace_bytes(dims, abi.MODE_VJP, 0))
            _, ga, gd, gs = lib.loglik_vjp(dims, act, dyn, x_tm, ll_bar=ll_bar.contiguous(), sigma0=sigma0,
                                           want_qf=ctx.has_qf, ws=ws, stream=_stream(dev))
        grads = [ga[k] for k in ACT_KEYS] + [gd[k] for k in DYN_KEYS] + ([ga["Qf"]] if ctx.has_qf else []) + \
                ([gs] if ctx.has_sigma0 else [])
        out = []
        for g, shp in zip(grads, ctx.shapes):
            if len(shp) == 4:          # materialised time-varying input: forward only (checked in forward)
                out.append(None)
                continue
            # time-invariant base matrix (S|1, r, c): the kernel already summed the cotangent over time (SURVEY H6)
            out.append(g.sum(0, keepdim=True) if (shp[0] == 1 and g.shape[0] != 1) else g)
        return (None, None, None, None, None, *out)


def _qf_is_default(actor: LQGSpec) -> bool:
    """True when ``spec.Qf`` is the spec's own ``Q`` base matrix (what ``time_stack_spec`` builds, lqg/utils.py:30):
    the kernels then default ``Qf`` to ``Q`` and send its gradient there."""
    Qf, Q = actor.Qf, actor.Q
    if Qf is None:
        return True
    return (Qf.data_ptr() == Q.data_ptr() and Qf.shape[-2:] == Q.shape[-2:] and Qf.stride()[-2:] == Q.stride()[-2:]
            and is_time_invariant(_as4(Q)) and Qf.dim() == Q.dim() - 1 and Qf.stride()[:-2] == Q.stride()[:-3])


def _check_no_cross_cost(actor: LQGSpec):
    """The fused likelihood assumes ``P = 0`` (state-control cross cost), true for every reference model
    (lqg/utils.py:32); a spec with ``P != 0`` would silently differ from ``lqr.backward``'s gains, so refuse it.
    Specs built by ``time_stack_spec`` are recognised without looking at the values (no host sync)."""
    from lqg_b200.utils import is_known_zero
    P = actor.P
    if P is None or is_known_zero(P):
        return
    if bool((P != 0).any()):
        raise NotImplementedError("lqg_b200: the fused log-likelihood kernels assume P = 0 (no state-control cross cost); "
                                  "use lqr.backward / conditional_moments (slow path) for specs with P != 0")


def _observed_call(lib, dims: abi.LqgkDims, actor: LQGSpec, dynamics: LQGSpec, x: torch.Tensor, Sigma0, call, x_tm=None):
    """Checks x[(S,) n, T+1, d] against the spec, packs it (unless x_tm is given), hands the base matrices (with a Qf of the
    spec's own) and Sigma0 to ``call(x_tm, act, dyn, sigma0)`` and drops the sample axis of its output for an un-batched model."""
    per_sample = x.dim() == 4
    if per_sample and x.shape[0] != dims.S:
        raise ValueError(f"per-sample observations need a leading axis of {dims.S} samples, got {x.shape[0]}")
    if dims.T != x.shape[-2] - 1:
        raise ValueError(f"need T+1 = {dims.T + 1} observations per trial, got {x.shape[-2]} (SURVEY H7: spec.T == x.shape[-2] - 1)")
    if x_tm is None:
        if per_sample:   # [S, n, T+1, d] -> [S, T+1, n, d] float32
            x_tm = x.detach().permute(0, 2, 1, 3).to(torch.float32).contiguous()
        else:
            x_tm = lib.pack_obs(x.detach(), stream=_stream(x.device))
    dt = actor.A.dtype

    def base(M):   # (S|1, r, c) base matrix of a time-invariant array (stride-0 time axis), else the (S|1, T, r, c) array
        M4 = _as4(M)
        return _row_major(M4[:, 0] if is_time_invariant(M4) else M4).to(dt)
    act, dyn = {k: base(getattr(actor, k)) for k in ACT_KEYS}, {k: base(getattr(dynamics, k)) for k in DYN_KEYS}
    if not _qf_is_default(actor):   # a terminal cost of its own (lqg/control/lqr.py:37 starts the sweep from spec.Qf)
        act["Qf"] = _untimed(actor.Qf, dt)
    s0 = None if Sigma0 is None else _untimed(Sigma0, dt)
    return _unbatch(actor, dynamics, call(x_tm, act, dyn, s0))


def log_likelihood(actor: LQGSpec, dynamics: LQGSpec, x: torch.Tensor, Sigma0: Optional[torch.Tensor] = None,
                   x_tm: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-trial log-likelihood (reference ``System.log_likelihood``, lqg/system.py:246-248).

    x: (n, T+1, d) -- one data set shared by all parameter samples -- or (S, n, T+1, d) -- one data set per sample
    (e.g. one sample per experimental condition).  Returns (n,) for an un-batched spec, (S, n) otherwise."""
    _require_cuda(actor.A, "actor spec")
    _require_cuda(x, "observations")
    lib = abi.load_library()
    dims = dims_of(actor, dynamics, x.shape[-3], x.shape[-1])
    check_supported(dims)
    _check_no_cross_cost(actor)

    def call(x_tm, act, dyn, s0):
        mats = [act[k] for k in ACT_KEYS] + [dyn[k] for k in DYN_KEYS] + [m for m in (act.get("Qf"), s0) if m is not None]
        return _LogLikFn.apply(x_tm, dims, "Qf" in act, s0 is not None, len(ACT_KEYS), *mats)
    return _observed_call(lib, dims, actor, dynamics, x, Sigma0, call, x_tm=x_tm)


def moments(actor: LQGSpec, dynamics: LQGSpec, x: torch.Tensor, Sigma0: Optional[torch.Tensor] = None, want_mu=True, want_sigma=True):
    """CUDA predictive moments of the joint state (reference ``vmap(System.conditional_moments)``, lqg/system.py:142-235):
    ``mu[(S,) n, T, nj]``, ``Sigma[(S,) T, nj, nj]``.  Returns None if no kernels are compiled for the dimensions (callers then
    use the torch slow path)."""
    _require_cuda(actor.A, "actor spec")
    lib = abi.load_library()
    n, T1, d = x.shape[-3:]
    dims = dims_of(actor, dynamics, n, d)
    if (dims.x, dims.b, dims.u, dims.y, dims.d) not in SUPPORTED_DIMS or dims.x + dims.b > 12 or dims.T != T1 - 1:
        return None
    _check_no_cross_cost(actor)
    dev = actor.A.device

    def call(x_tm, act, dyn, s0):
        ws = workspace(dev, lib.workspace_bytes(dims, abi.MODE_MOMENTS, 0))
        return lib.moments(dims, act, dyn, x_tm, sigma0=s0, want_mu=want_mu, want_sigma=want_sigma, ws=ws, stream=_stream(dev))
    return _observed_call(lib, dims, actor, dynamics, x, Sigma0, call)


def simulate(actor: LQGSpec, dynamics: LQGSpec, L, l, K, n: int, seed: int, x0=None, xhat0=None, return_all=False, C=None, D=None):
    """CUDA batched simulator (reference ``System.simulate``, lqg/system.py:62-140) for given gains ``L[(S,) T, u, b]``,
    ``l[(S,) T, u]``, ``K[(S,) T, b, y]``; returns ``x[(S,) n, T+1, xdim]`` (and xhat, y, u).  None if a dimension exceeds the
    kernel's limit (callers then use the torch slow path)."""
    _require_cuda(actor.A, "actor spec")
    lib = abi.load_library()
    dims = dims_of(actor, dynamics, n, 1)
    if max(dims.x, dims.b, dims.u, dims.y) > 40:
        return None
    dt, dev = actor.A.dtype, actor.A.device
    S = dims.S
    act = {k: _row_major(_as4(getattr(actor, k))).to(dt) for k in ("A", "B", "F")}
    dyn = {k: _row_major(_as4(getattr(dynamics, k))).to(dt) for k in DYN_KEYS}

    vec = lambda v: None if v is None else torch.as_tensor(v, dtype=dt, device=dev).reshape(-1).contiguous()
    out = lib.simulate(dims, act, dyn, _per_sample(L, 3, S, dt), _per_sample(l, 2, S, dt), _per_sample(K, 3, S, dt), seed,
                       x0=vec(x0), xhat0=vec(xhat0), return_all=return_all, stream=_stream(dev),
                       C_noise=C, D_noise=D)   # C, D: signal-dependent-noise extension
    return _unbatch(actor, dynamics, out)


def sdn_log_likelihood(actor: LQGSpec, dynamics: LQGSpec, x: torch.Tensor, L: torch.Tensor, K: torch.Tensor,
                       C: Optional[torch.Tensor] = None, D: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-trial log-likelihood under signal-dependent noise (EXTENSION, no reference counterpart; include/lqgk.h:
    lqgk_sdn_loglik_*, spec oracle/sdn_np.py).  ``L[(S,) T, u, b]``, ``K[(S,) T, b, y]``: the gains; ``C[(S,) nc, x, u]``:
    control-dependent process-noise matrices; ``D[(S,) nd, y, x]``: state-dependent observation-noise matrices.
    x as in :func:`log_likelihood`.  Forward only (gradients: lqg_b200.control.sdn.value_and_grad_fd)."""
    _require_cuda(actor.A, "actor spec")
    _require_cuda(x, "observations")
    lib = abi.load_library()
    dims = dims_of(actor, dynamics, x.shape[-3], x.shape[-1])
    if (dims.x, dims.b, dims.u, dims.y, dims.d) not in FP64_ONLY_DIMS:
        check_supported(dims)
    if dims.x + dims.b > 12:
        raise NotImplementedError("lqg_b200: the signal-dependent-noise / all-FP64 likelihood is compiled for joint dims <= 12")
    dt, dev = actor.A.dtype, actor.A.device

    def call(x_tm, act, dyn, s0):
        for M in list(act.values()) + list(dyn.values()):
            if M.dim() == 4:
                raise NotImplementedError("lqg_b200: the signal-dependent-noise likelihood needs time-invariant specs")
        return lib.sdn_loglik(dims, act, dyn, _per_sample(L, 3, dims.S, dt), _per_sample(K, 3, dims.S, dt), x_tm, C_noise=C,
                              D_noise=D, stream=_stream(dev))
    return _observed_call(lib, dims, actor, dynamics, x, None, call)
