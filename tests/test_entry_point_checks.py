"""Argument checks of the C ABI: one table of malformed calls and the LQGK_* code each entry point returns for it.

Every call here is rejected before the library makes its first CUDA call, so the pointers are fake (non-null, aligned,
never dereferenced) and the table runs without a GPU -- against liblqgk.so and against the host build of the same
entry points (tests/emul/liblqgk_emul.so; its entry points take no workspace, so the workspace cases are left out).
The host build runs each call in a forked child: a check it were missing would dereference a fake pointer, and that
must fail one case, not the test process."""
import ctypes as C
import os
import warnings

import pytest

from lqg_b200 import abi
from tests import helpers as H

OK, INVALID, UNSUPPORTED, WORKSPACE = 0, -1, -2, -3
FAKE = 1 << 20            # a 256-byte aligned address nobody dereferences
BIG_WS = 1 << 40          # workspace bytes when the workspace is not what a case is about

ACT7 = ("A", "B", "F", "V", "W", "Q", "R")
DYN5 = ("A", "B", "F", "V", "W")


def dims(x=4, b=6, u=2, y=4, d=4, S=64, N=20, T=100, stride=0):
    return abi.LqgkDims(S, N, T, x, b, u, y, d, stride)


def spec(keys, tv=(), null=()):
    sp = abi.LqgkSpec()
    for k in keys:
        setattr(sp, k, abi.LqgkMat(None if k in null else FAKE, 0, 16 if k in tv else 0))
    return sp


def noise(nc=0, nd=0, C_null=False):
    return abi.LqgkSdnNoise(abi.LqgkMat(None if C_null else FAKE, 0, 0), abi.LqgkMat(FAKE, 0, 0), nc, nd)


def sdn_spec(null=()):
    sp = abi.LqgkSdnSpec()
    for k, _ in abi.LqgkSdnSpec._fields_:
        setattr(sp, k, abi.LqgkMat(None if k in null else FAKE, 0, 0))
    return sp


def ref(s):
    return C.byref(s) if s is not None else None


P = C.c_void_p


# -- one caller per entry point: the arguments of a well-formed call, any of them replaced by keyword
def lqr_backward(lib, p, d=dims(), act=spec(ACT7), L=FAKE, ws=FAKE, ws_bytes=BIG_WS):
    return getattr(lib, "lqgk_lqr_backward_" + p)(ref(d), ref(act), C.c_double(1e-8), P(L), P(FAKE), P(FAKE), P(ws),
                                                  C.c_size_t(ws_bytes), P(None))


def kf_forward(lib, p, d=dims(), act=spec(ACT7), K=FAKE, ws=FAKE, ws_bytes=BIG_WS):
    return getattr(lib, "lqgk_kf_forward_" + p)(ref(d), ref(act), None, P(K), P(ws), C.c_size_t(ws_bytes), P(None))


def loglik_fwd(lib, p, d=dims(), act=spec(ACT7), dyn=spec(DYN5), x_tm=FAKE, ll=FAKE, ws=FAKE, ws_bytes=BIG_WS):
    return getattr(lib, "lqgk_loglik_fwd_" + p)(ref(d), ref(act), ref(dyn), None, P(x_tm), P(ll), P(ws),
                                                C.c_size_t(ws_bytes), P(None))


def loglik_vjp(lib, p, d=dims(), act=spec(ACT7), dyn=spec(DYN5), ws=FAKE, ws_bytes=BIG_WS):
    ga, gd = abi.LqgkSpecGrad(), abi.LqgkSpecGrad()
    return getattr(lib, "lqgk_loglik_vjp_" + p)(ref(d), ref(act), ref(dyn), None, P(FAKE), P(None), P(FAKE), ref(ga),
                                                ref(gd), None, P(ws), C.c_size_t(ws_bytes), P(None))


def moments(lib, p, d=dims(), mu=FAKE, Sig=FAKE, ws=FAKE, ws_bytes=BIG_WS):
    return getattr(lib, "lqgk_moments_" + p)(ref(d), ref(spec(ACT7)), ref(spec(DYN5)), None, P(FAKE), P(mu), P(Sig),
                                             P(ws), C.c_size_t(ws_bytes), P(None))


def simulate(lib, p, d=dims(S=4, N=8), nz=None):
    args = (P(FAKE), P(None), P(FAKE), P(None), P(None), C.c_uint64(0), P(FAKE), P(None), P(None), P(None), P(None))
    if nz is None:
        return getattr(lib, "lqgk_simulate_" + p)(ref(d), ref(spec(ACT7)), ref(spec(DYN5)), *args)
    return getattr(lib, "lqgk_sdn_simulate_" + p)(ref(d), ref(spec(ACT7)), ref(spec(DYN5)), ref(nz), *args)


def sdn_loglik(lib, p, d=dims(), act=spec(ACT7), nz=None):
    return getattr(lib, "lqgk_sdn_loglik_" + p)(ref(d), ref(act), ref(spec(DYN5)), ref(nz), P(FAKE), P(FAKE), P(FAKE),
                                                P(FAKE), P(None))


def sdn_gains(lib, p, b=6, u=2, y=4, nc=0, nd=0, sweeps=10, sp=None, filter_form=False):
    d = abi.LqgkSdnDims(64, 100, b, u, y, nc, nd, sweeps)
    fn = lib.lqgk_sdn_gains_filter_f64 if filter_form else lib.lqgk_sdn_gains_f64
    return fn(ref(d), ref(sp or sdn_spec()), P(FAKE), P(FAKE), P(FAKE), P(None))


def pack_obs(lib, p, N=20, T1=101, d=4, x=FAKE):
    return getattr(lib, "lqgk_pack_obs_" + p)(C.c_int32(N), C.c_int32(T1), C.c_int32(d), P(x), P(FAKE), P(None))


def workspace_bytes(lib, p, d, mode):
    fn = lib.lqgk_workspace_bytes
    fn.restype = C.c_size_t
    return fn(ref(d), C.c_int(mode), C.c_int32(0))


# (id, call(lib, precision), expected result, kind).  kind "ws": a workspace case, liblqgk.so only; "new": the host build
# rejects it with the library's code since both share their argument checks (before, the host build dereferenced a fake
# pointer, returned LQGK_OK or returned another code); "kept": rejected alike by both before.
CASES = [
    ("null-dims", lambda l, p: loglik_fwd(l, p, d=None), INVALID, "kept"),
    ("null-actor", lambda l, p: loglik_vjp(l, p, act=None), INVALID, "kept"),
    ("null-dynamics-matrix", lambda l, p: loglik_fwd(l, p, dyn=spec(DYN5, null="W")), INVALID, "new"),
    ("null-actor-matrix", lambda l, p: loglik_fwd(l, p, act=spec(ACT7, null="R")), INVALID, "new"),
    ("null-ll-out", lambda l, p: loglik_fwd(l, p, ll=None), INVALID, "new"),
    ("null-L-out", lambda l, p: lqr_backward(l, p, L=None), INVALID, "new"),
    ("null-K-out", lambda l, p: kf_forward(l, p, K=None), INVALID, "new"),
    ("moments-no-output", lambda l, p: moments(l, p, mu=None, Sig=None), INVALID, "new"),
    ("zero-trials", lambda l, p: loglik_fwd(l, p, d=dims(N=0)), INVALID, "new"),
    ("zero-samples-gains", lambda l, p: lqr_backward(l, p, d=dims(S=0)), INVALID, "new"),
    ("zero-control-dim", lambda l, p: kf_forward(l, p, d=dims(u=0)), INVALID, "new"),
    ("d-above-x", lambda l, p: loglik_fwd(l, p, d=dims(d=5)), INVALID, "new"),
    ("unsupported-tuple", lambda l, p: loglik_fwd(l, p, d=dims(x=3, b=7, u=1, y=2, d=2)), UNSUPPORTED, "kept"),
    ("unsupported-tuple-gains", lambda l, p: lqr_backward(l, p, d=dims(x=3, b=7, u=1, y=2, d=2)), UNSUPPORTED, "kept"),
    ("unsupported-tuple-vjp", lambda l, p: loglik_vjp(l, p, d=dims(x=4, b=6, u=2, y=4, d=2)), UNSUPPORTED, "kept"),
    ("x-sample-stride-misaligned-d2", lambda l, p: loglik_fwd(l, p, d=dims(2, 2, 1, 2, 2, stride=2 * 101 * 20 + 1)),
     INVALID, "new"),
    ("x-sample-stride-misaligned-d4", lambda l, p: loglik_fwd(l, p, d=dims(stride=4 * 101 * 20 + 2)), INVALID, "new"),
    ("x-sample-stride-negative", lambda l, p: loglik_vjp(l, p, d=dims(stride=-8)), INVALID, "new"),
    ("x-tm-misaligned", lambda l, p: loglik_fwd(l, p, x_tm=FAKE + 8), INVALID, "new"),
    ("time-varying-vjp", lambda l, p: loglik_vjp(l, p, act=spec(ACT7, tv="W")), UNSUPPORTED, "kept"),
    ("time-varying-dynamics-vjp", lambda l, p: loglik_vjp(l, p, dyn=spec(DYN5, tv="V")), UNSUPPORTED, "kept"),
    ("moments-large-system", lambda l, p: moments(l, p, d=dims(12, 12, 1, 3, 2)), UNSUPPORTED, "kept"),
    ("workspace-null", lambda l, p: loglik_fwd(l, p, ws=None), INVALID, "ws"),
    ("workspace-misaligned", lambda l, p: loglik_vjp(l, p, ws=FAKE + 64), INVALID, "ws"),
    ("workspace-too-small", lambda l, p: loglik_vjp(l, p, ws_bytes=1 << 10), WORKSPACE, "ws"),
    ("workspace-too-small-gains", lambda l, p: lqr_backward(l, p, ws_bytes=1 << 10), WORKSPACE, "ws"),
    ("sdn-loglik-time-varying", lambda l, p: sdn_loglik(l, p, act=spec(ACT7, tv="A")), UNSUPPORTED, "new"),
    ("sdn-loglik-nc-5", lambda l, p: sdn_loglik(l, p, nz=noise(nc=5)), INVALID, "new"),
    ("sdn-loglik-nd-5", lambda l, p: sdn_loglik(l, p, nz=noise(nd=5)), INVALID, "new"),
    ("sdn-loglik-nc-negative", lambda l, p: sdn_loglik(l, p, nz=noise(nc=-1)), INVALID, "new"),
    ("sdn-loglik-nd-negative", lambda l, p: sdn_loglik(l, p, nz=noise(nd=-1)), INVALID, "new"),
    ("sdn-loglik-C-missing", lambda l, p: sdn_loglik(l, p, nz=noise(nc=1, C_null=True)), INVALID, "new"),
    ("sdn-loglik-null-actor-matrix", lambda l, p: sdn_loglik(l, p, act=spec(ACT7, null="F")), INVALID, "new"),
    ("sdn-loglik-zero-trials", lambda l, p: sdn_loglik(l, p, d=dims(N=0)), INVALID, "new"),
    ("sdn-loglik-large-system", lambda l, p: sdn_loglik(l, p, d=dims(12, 12, 1, 3, 2)), UNSUPPORTED, "kept"),
    ("sdn-loglik-unsupported-tuple", lambda l, p: sdn_loglik(l, p, d=dims(4, 4, 1, 3, 3)), UNSUPPORTED, "kept"),
    ("sdn-simulate-nc-5", lambda l, p: simulate(l, p, nz=noise(nc=5)), INVALID, "kept"),
    ("sdn-simulate-nd-negative", lambda l, p: simulate(l, p, nz=noise(nd=-1)), INVALID, "kept"),
    ("sdn-simulate-C-missing", lambda l, p: simulate(l, p, nz=noise(nc=2, C_null=True)), INVALID, "kept"),
    ("simulate-dim-above-40", lambda l, p: simulate(l, p, d=dims(x=41, S=4, N=8)), UNSUPPORTED, "kept"),
    ("simulate-zero-trials", lambda l, p: simulate(l, p, d=dims(S=4, N=0)), INVALID, "kept"),
    ("sdn-gains-large-tuple-only", lambda l, p: sdn_gains(l, p, b=12, u=1, y=3), UNSUPPORTED, "kept"),
    ("sdn-gains-filter-large-tuple-only", lambda l, p: sdn_gains(l, p, b=12, u=1, y=3, filter_form=True), UNSUPPORTED,
     "kept"),
    ("sdn-gains-unsupported", lambda l, p: sdn_gains(l, p, b=5, u=3, y=1), UNSUPPORTED, "kept"),
    ("sdn-gains-null-xhat1", lambda l, p: sdn_gains(l, p, sp=sdn_spec(null=("xhat1",))), INVALID, "new"),
    ("sdn-gains-null-Sigma1", lambda l, p: sdn_gains(l, p, sp=sdn_spec(null=("Sigma1",))), INVALID, "new"),
    ("sdn-gains-C-missing", lambda l, p: sdn_gains(l, p, nc=1, sp=sdn_spec(null=("C",))), INVALID, "new"),
    ("sdn-gains-negative-sweeps", lambda l, p: sdn_gains(l, p, sweeps=-1, filter_form=True), INVALID, "new"),
    ("pack-obs-zero-trials", lambda l, p: pack_obs(l, p, N=0), INVALID, "new"),
    ("pack-obs-null-input", lambda l, p: pack_obs(l, p, x=None), INVALID, "new"),
    ("dims-supported-fp64-only", lambda l, p: l.lqgk_dims_supported(ref(dims(4, 4, 1, 3, 4))), 0, "kept"),
    ("dims-supported-gains-d", lambda l, p: l.lqgk_dims_supported(ref(dims(d=3))), 0, "kept"),
    ("workspace-bytes-gains-any-d", lambda l, p: int(workspace_bytes(l, p, dims(d=3), abi.MODE_GAINS) > 0), 1, "kept"),
    ("workspace-bytes-fwd-wrong-d", lambda l, p: workspace_bytes(l, p, dims(d=3), abi.MODE_FWD), 0, "kept"),
    ("workspace-bytes-null-dims", lambda l, p: workspace_bytes(l, p, None, abi.MODE_VJP), 0, "kept"),
    ("init-zero-slices", lambda l, p: l.lqgk_init(C.c_int(0)), INVALID, "kept"),
    ("set-streams-33", lambda l, p: l.lqgk_set_streams(C.c_int(33)), INVALID, "kept"),
    ("set-contrib-warps-0", lambda l, p: l.lqgk_set_contrib_warps(C.c_int(0)), INVALID, "kept"),
    ("set-warp-cov-negative", lambda l, p: l.lqgk_set_warp_cov_max_samples(C.c_int(-1)), INVALID, "kept"),
    ("set-pipeline-65-segments", lambda l, p: l.lqgk_set_pipeline(C.c_int(0), C.c_int(65)), INVALID, "kept"),
    ("set-kernel-overlap-8", lambda l, p: l.lqgk_set_kernel_overlap(C.c_int(8)), INVALID, "kept"),
    ("profile-read-null", lambda l, p: l.lqgk_profile_read(None, None, C.c_int(4)), INVALID, "kept"),
    ("peak-fma-null-sink", lambda l, p: l.lqgk_peak_fma(C.c_int(1), C.c_int(16), P(None), P(None), None), INVALID,
     "kept"),
]


class _Probe:
    """Records the entry points a case calls."""

    def __init__(self):
        self.names = []

    def __getattr__(self, name):
        self.names.append(name)
        return lambda *args: 0


def _params(path, with_ws):
    lib = C.CDLL(path) if os.path.exists(path) else None
    out = []
    for cid, call, want, kind in CASES:
        if kind == "ws" and not with_ws:
            continue
        seen = set()
        for p in ("f32", "f64"):
            probe = _Probe()
            call(probe, p)
            names = tuple(probe.names)
            if names in seen or (lib is not None and not all(hasattr(lib, n) for n in names)):
                continue
            seen.add(names)
            out.append(pytest.param(call, p, want, id=f"{cid}-{names[0][len('lqgk_'):]}"))
    return out


def _in_child(fn):
    """fn()'s return value (-128..127) from a forked child, or a description of how the child died."""
    with warnings.catch_warnings():
        # the child makes one call into the host build, whose only shared state is the C heap (which glibc re-arms in a
        # forked child), and leaves with os._exit
        warnings.simplefilter("ignore", DeprecationWarning)
        pid = os.fork()
    if pid == 0:
        try:
            rc = int(fn())
        except BaseException:
            os._exit(200)
        os._exit(rc & 0xFF)
    _, status = os.waitpid(pid, 0)
    if os.WIFSIGNALED(status):
        return f"killed by signal {os.WTERMSIG(status)}"
    code = os.WEXITSTATUS(status)
    return code - 256 if code >= 128 else code


@pytest.mark.parametrize("call, p, want", _params(abi.LIB_PATH, with_ws=True))
def test_library_rejects(call, p, want):
    assert call(C.CDLL(abi.LIB_PATH), p) == want


@pytest.mark.parametrize("call, p, want", _params(H.EMUL_PATH, with_ws=False))
def test_host_build_rejects(call, p, want):
    lib = C.CDLL(H.EMUL_PATH)
    assert _in_child(lambda: call(lib, p)) == want
