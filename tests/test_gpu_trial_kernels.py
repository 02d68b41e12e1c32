"""Every compiled instantiation of the per-trial kernels k_trial_fwd / k_trial_rev (lqgk_kernels.cuh) against the float64
oracle.

Both kernels are compiled for every tuple of lqgk_dims.h and every RT = 1..trial_rt_max (trials per lane); a call runs the
one with RT = min(ceil(N / 32), trial_rt_max).  Each instantiation has its own code and geometry: pairs of adjacent trials
per lane plus a single column when RT is odd (trial_col), rows of ROW = 32 RT trials, NB passes over them, and a checkpoint
interval CK = trial_ck(RT) of the adjoint.  The host-side tests pin a mirror of that geometry to the library: its workspace
sizes reveal RT and CK, its kernel symbols the set of instantiations.  The GPU tests run every (tuple, RT) where its edges
are: one live lane in the last column group, an empty pair half, a partial last pass, a partial last checkpoint segment and
a horizon shorter than one segment; then observations given per sample across chunks and covariance kernel variants, in the
adjoint and in the predictive moments."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from lqg_b200 import abi
from lqg_b200.dims import SUPPORTED_DIMS
from oracle import lqg_np as O
from tests import helpers as H


# ------------------------------------------------------------------------------------------------ geometry mirror
def trial_geometry(dims):
    """trial_rt_max, trial_ck(RT) and trial_tb (lqgk_kernels.cuh) of a tuple, from the record sizes of Dims (lqgk_core.h)."""
    x, b, u, y, d = dims
    n, r, tri = x + b, x + b - d, d * (d + 1) // 2
    rec = (n * n + r * d + tri + 1 + 3) // 4 * 4                        # REC: F | J | Linv | logdet, rounded to 4 floats
    nsum = (n * n + 3) // 4 * 4 + r * d + tri                           # NSUM: Fb | Jb | Wv
    red = 32 * 36 * 4 if nsum >= 32 else 0                              # trial_red_bytes
    per_step = lambda rt: 2 * rec * 4 + r * 32 * rt * 4                # 2 record ring stages + one state slot of 32 RT trials
    ck = lambda rt: max(1, min(8, (28440 - red - 16) // per_step(rt)))  # LQGK_TRIAL_WARP_SMEM, TRIAL_CK_MAX
    return (8 if n * n <= 36 else 4), ck, (8 if rec <= 128 else (4 if rec <= 256 else 2))


def trial_rt(N, rt_max):
    return min((N + 31) // 32, rt_max)


INSTANCES = [(dims, rt) for dims in SUPPORTED_DIMS for rt in range(1, trial_geometry(dims)[0] + 1)]
MODEL = {dims: name for dims in SUPPORTED_DIMS for name, xbuy in H.MODEL_DIMS.items() if xbuy == dims[:4]}


def dims_id(dims):
    return "-".join(map(str, dims))


def test_every_compiled_tuple_has_a_model():
    assert sorted(MODEL) == sorted(SUPPORTED_DIMS)
    assert len(INSTANCES) == 52          # 3 tuples with joint dim <= 6 x 8 + 7 x 4


def _ws_bytes(lib, dims, N, T, S, mode, max_chunk, per_sample):
    d = abi.LqgkDims(S, N, T, *dims, (T + 1) * N * dims[4] if per_sample else 0)
    return int(lib.lib.lqgk_workspace_bytes(C.byref(d), mode, max_chunk))


@pytest.mark.parametrize("dims", SUPPORTED_DIMS, ids=dims_id)
def test_mirror_matches_the_library_rt(dims):
    """The repacked observations take (T+1) NB d ROW floats once, or once per sample of a 32-sample chunk with per-sample
    data: the difference of the two workspace sizes is 4 * 31 * (T+1) * d * NB * ROW bytes up to the 256-byte alignment of
    the workspace parts, which gives the padded trial count NB * ROW of the instantiation the library picks."""
    lib = abi.load_library()
    rt_max = trial_geometry(dims)[0]
    T, d = 100, dims[4]
    unit = 4 * 31 * (T + 1) * d                 # > 256 bytes: the alignment cannot blur one trial
    for rt in range(1, rt_max + 1):
        for N in [32 * (rt - 1) + 1, 32 * rt] + ([2 * 32 * rt + 3, 9 * 32 * rt - 1] if rt == rt_max else []):
            assert trial_rt(N, rt_max) == rt
            diff = (_ws_bytes(lib, dims, N, T, 1, abi.MODE_FWD, 32, True)
                    - _ws_bytes(lib, dims, N, T, 1, abi.MODE_FWD, 32, False))
            padded = round(diff / unit)
            assert abs(diff - unit * padded) < 256, (N, diff)
            assert padded == -(-N // (32 * rt)) * 32 * rt, (rt, N, padded)


@pytest.mark.parametrize("dims", SUPPORTED_DIMS, ids=dims_id)
def test_mirror_matches_the_library_ck(dims):
    """The adjoint's checkpoints take NB R ROW floats per sample and checkpoint segment, ceil(T / CK) segments: from T - 1 to
    T the workspace grows by the parts linear in T, the repacked observations' NB d ROW floats (one data set shared by the
    samples) and, when T - 1 is a multiple of CK, one more segment.  With 4,096 samples in one chunk a segment is >= 1 MB, far above the alignment
    of the workspace parts, so the steps of the workspace size give CK."""
    lib = abi.load_library()
    rt_max, ck, _ = trial_geometry(dims)
    S, d, r, Ts = 4096, dims[4], dims[0] + dims[1] - dims[4], range(1, 27)

    def steps(rt):           # size(T) - size(T - 1) for T = 2..26, less the repacked observations' part (NB = 1)
        f = [_ws_bytes(lib, dims, 32 * (rt - 1) + 1, T, S, abi.MODE_VJP, 0, False) for T in Ts]
        return np.diff(f) - 4 * d * 32 * rt

    base = steps(1).min()    # the parts linear in T: CK(1) >= 2, so some step adds no segment
    for rt in range(1, rt_max + 1):
        segs = np.rint((steps(rt) - base) / (4 * S * r * 32 * rt)).astype(int).tolist()
        nseg = lambda T: -(-T // ck(rt))
        want = [nseg(T) - nseg(T - 1) for T in Ts[1:]]
        assert segs == want, (rt, ck(rt), segs)


def _cuda_tool(name):
    path = shutil.which(name) or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)
    return path if os.path.exists(path) else None


def test_every_instantiation_is_in_the_sweep():
    """The trial-kernel instantiations liblqgk.so contains are exactly the mirror's: a new tuple, a new trial_rt_max or
    other static_for bounds fail here until the sweep below covers them."""
    dump, filt = _cuda_tool("cuobjdump"), _cuda_tool("cu++filt")
    if dump is None or filt is None:
        pytest.skip("cuobjdump / cu++filt not installed")
    syms = subprocess.run([dump, "-symbols", abi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted({w for w in syms.split() if "k_trial_fwd" in w or "k_trial_rev" in w})
    names = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    found = {"fwd": set(), "rev": set()}
    for kind, tup, rt in re.findall(r"k_trial_(fwd|rev)<lqgk::Dims<([^>]*)>,\s*(?:\(int\))?(\d+)>", names):
        found[kind].add((tuple(int(v) for v in re.findall(r"\d+", tup.replace("(int)", ""))), int(rt)))
    assert len(found["fwd"]) == len(found["rev"]) == 52
    assert found["fwd"] == found["rev"] == set(INSTANCES)


# ------------------------------------------------------------------------------------------------ the sweep (GPU)
def _sweep():
    out = []
    for dims in SUPPORTED_DIMS:
        rt_max, ck, tb = trial_geometry(dims)
        for rt in range(1, rt_max + 1):
            T = 3 * ck(rt) + 2                                  # a partial last checkpoint segment
            Ns = [32 * (rt - 1) + 1, 32 * rt - 1] + ([2 * 32 * rt + 3] if rt == rt_max else [])
            out += [(dims, rt, N, T) for N in Ns]
            al = tb // math.gcd(ck(rt), tb)
            if al > 1 and dims[0] + dims[1] <= 12:
                # the pipelined sequence cuts time on multiples of `al` checkpoint segments (where the forward kernel's record
                # chunks start): a horizon of two such cuts and a partial segment has launches with ka > 0 here too
                out.append((dims, rt, 32 * rt - 1, 2 * al * ck(rt) + 2))
        c = ck(rt_max)
        out.append((dims, rt_max, 2 * 32 * rt_max + 3, c - 1 if c > 1 else 1))   # one segment, shorter than CK
    return [pytest.param(*p, id=f"{dims_id(p[0])}-rt{p[1]}-N{p[2]}-T{p[3]}") for p in out]


def lane_positions(N, rt):
    """Trials at distinct lane positions of the instantiation: the first pair's two halves, the single column of odd RT,
    the last column of the first pass, the first of the second pass and the last trial (clipped to N)."""
    row = 32 * rt
    pos = [0, 1] + ([64 * (rt // 2)] if rt % 2 else []) + [row - 1] + ([row] if N > row else []) + [N - 1]
    return list(dict.fromkeys(min(p, N - 1) for p in pos))


def one_hot(N, rt, S):
    pos = lane_positions(N, rt)
    w = np.zeros((S, N))
    for s in range(S):
        w[s, pos[s % len(pos)]] = 1.0
    return w


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    return abi.load_library()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _vjp(lib, dev, case, dtype):
    dims = case.lqgk_dims()
    act, dyn = case.tensors(dev, dtype)
    ws = H.workspace(lib, dims, abi.MODE_VJP, dev)
    ll_bar = torch.tensor(case.w, dtype=dtype, device=dev)
    ll, ga, gd, _ = lib.loglik_vjp(dims, act, dyn, case.x_tm(lib, dev), ll_bar=ll_bar, ws=ws, stream=H.stream_of(dev))
    torch.cuda.synchronize(dev)
    return [ll] + list(ga.values()) + list(gd.values())


@pytest.mark.gpu
@pytest.mark.parametrize("dims,rt,N,T", _sweep())
def test_trial_kernel_instantiation(lib, dev, dims, rt, N, T):
    rt_max = trial_geometry(dims)[0]
    assert trial_rt(N, rt_max) == rt
    name, d, small = MODEL[dims], dims[4], dims[0] + dims[1] <= 12
    seed = 100 * rt + N + T
    # shared data, random trial weights: per-trial likelihoods and every base-matrix gradient
    case = H.Case(name, S=5, T=T, N=N, d=d, seed=seed, weights=True)
    H.check_fwd(lib, dev, case, torch.float32)
    H.check_vjp(lib, dev, case, torch.float32)
    # one data set per sample, cotangent one-hot at one lane position per sample: one trial's gradient each.  Two trials'
    # gradients differ by more than their size; one trial's own FP32 error is < 1e-4 of it, except in the point-mass models
    # (action_variability 1e-3, innovation covariance ~1e-6), where it reaches 3e-3 in dA (test_large_system_c4_full_horizon)
    g_rtol = 1e-2 if name in ("pointmass", "pmdelay2") else 1e-3
    S1 = max(5, len(lane_positions(N, rt)))
    hot = H.Case(name, S=S1, T=T, N=N, d=d, seed=seed + 1, per_sample_data=True, w=one_hot(N, rt, S1))
    H.check_vjp(lib, dev, hot, torch.float32, g_rtol=g_rtol)
    if small:
        # the pipelined launch sequence (time segments over internal streams, k_trial_* launches with ka > 0) and its
        # one-segment case on the caller's stream are the same arithmetic
        outs = []
        for overlap in (6, 0):
            lib.set_kernel_overlap(overlap)
            try:
                H.check_vjp(lib, dev, hot, torch.float64, g_rtol=g_rtol)
                outs.append(_vjp(lib, dev, hot, torch.float64))
            finally:
                lib.set_kernel_overlap(6)
        names = ["ll"] + [f"actor {k}" for k in abi.ACTOR_KEYS] + [f"dyn {k}" for k in abi.DYN_KEYS]
        for what, a, b in zip(names, *outs):
            assert torch.allclose(a, b, rtol=1e-9, atol=1e-9 * float(a.abs().max()) + 1e-300), \
                (what, float((a - b).abs().max() / a.abs().max()))
    elif rt == rt_max:
        H.check_vjp(lib, dev, hot, torch.float64, g_rtol=g_rtol)


# -------------------------------------------------------------------------- per-sample data across chunks (GPU)
def _conditions(dims):
    """Three conditions (jittered parameters, each with its own simulated trials) at RT = trial_rt_max with a second pass
    of one trial; system s of a call is condition s mod 3, which is coprime with the 32-sample chunk and the per-CTA warps."""
    rt_max, ck, _ = trial_geometry(dims)
    N = 32 * rt_max + 1
    return H.Case(MODEL[dims], S=3, T=2 * ck(rt_max) + 3, N=N, d=dims[4], seed=7, weights=True, per_sample_data=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dims", SUPPORTED_DIMS, ids=dims_id)
def test_per_sample_data_across_chunks(lib, dev, dims):
    """Per-sample observations in chunks that start at sample s0 > 0 (the repacking reads data set s0 + s), and with the
    thread-per-sample covariance kernels, which the sweep's few samples do not reach."""
    case = _conditions(dims)
    H.check_vjp_tiled(lib, dev, case, total=70, max_chunk=32)          # chunks start at samples 0, 32, 64
    if dims[0] + dims[1] <= 12:
        H.check_vjp_tiled(lib, dev, case, 352)                             # 1,056 systems: thread-per-sample covariance kernels


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [t for t in SUPPORTED_DIMS if t[0] + t[1] <= 12], ids=dims_id)
def test_moments_with_per_sample_data_across_chunks(lib, dev, dims):
    """lqgk_moments_* with one data set per sample, 70 samples in chunks of 32, against the oracle's conditional_moments at
    the tolerances of test_moments_kernel_matches_oracle (FP32 per-trial means, FP64 covariances)."""
    case = H.Case(MODEL[dims], S=3, T=40, N=5, d=dims[4], seed=11, per_sample_data=True, want_grad=False)
    S, T, N = 70, case.T, case.N
    idx = torch.arange(S, device=dev) % 3
    act, dyn = case.tensors(dev, torch.float64)
    act = {k: v[idx].contiguous() for k, v in act.items()}
    dyn = {k: v[idx].contiguous() for k, v in dyn.items()}
    x_tm = case.x_tm(lib, dev)[idx].contiguous()
    dims_c = case.lqgk_dims(S)
    ws = H.workspace(lib, dims_c, abi.MODE_MOMENTS, dev, max_chunk=32)
    mu, Sig = lib.moments(dims_c, act, dyn, x_tm, ws=ws, stream=H.stream_of(dev))
    torch.cuda.synchronize(dev)
    mu, Sig = mu.cpu().numpy(), Sig.cpu().numpy()
    ref = []
    for c in range(3):
        sa, sd = O.make_system(case.mats[c], T)
        ref.append([O.conditional_moments(sa, sd, case.X[c][i].astype(np.float64)) for i in (0, N - 1)])
    for s in range(S):
        for k, i in enumerate((0, N - 1)):
            mu_o, Sig_o = ref[s % 3][k]
            assert np.allclose(mu[s, i], mu_o, rtol=2e-4, atol=2e-4 * np.abs(mu_o).max()), (s, i)
            assert np.allclose(Sig[s], Sig_o, rtol=1e-8, atol=1e-9 * np.abs(Sig_o).max()), s
