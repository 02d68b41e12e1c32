"""The adjoint of the gain sweeps (lqgk_gains_vjp_*) through liblqgk.so on the GPU: gradients against torch autograd through
the float64 oracle for every compiled tuple (thread-per-sample small systems and the warp-per-sample large one), chunking,
CUDA-graph capture, and the autograd of lqr.backward / kf.forward.  (tests/test_gains_vjp_on_host.py: the same on the host
build.)"""
import numpy as np
import pytest
import torch

from lqg_b200 import abi
from lqg_b200.belief import kf
from lqg_b200.control import lqr
from lqg_b200.utils import time_stack_spec
from tests.test_gains_vjp_on_host import GAINS_TUPLES, assert_grads_close, random_actor, run_vjp, theta_grads

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    return abi.load_library()


@pytest.mark.parametrize("which", ["L", "K", "LK"])
@pytest.mark.parametrize("tup", GAINS_TUPLES, ids=lambda t: "x%db%du%dy%d" % t)
def test_vjp_matches_torch_autograd_f64(lib, tup, which):
    got, exp = run_vjp(lib, tup, S=3, T=40, which=which, dev=DEV)
    assert_grads_close(got, exp)


@pytest.mark.parametrize("tup", GAINS_TUPLES, ids=lambda t: "x%db%du%dy%d" % t)
def test_vjp_matches_torch_autograd_f32(lib, tup):
    got, exp = run_vjp(lib, tup, S=3, T=40, which="LK", dev=DEV, dt=torch.float32, with_sigma0=True)
    assert_grads_close(got, exp, rel=1e-4, rtol=1e-4)


# (u = 1: over hundreds of steps the Riccati sweep converges and the u x u matrix H of a u = 2 system can get two nearly equal
# eigenvalues, where torch's eigvalsh backward inside the oracle returns NaN)
@pytest.mark.parametrize("tup", [(6, 6, 1, 2), (12, 12, 1, 3)], ids=["x6b6u1y2", "x12b12u1y3"])
@pytest.mark.parametrize("Qf", [False, True])
def test_vjp_long_horizon(lib, tup, Qf):
    got, exp = run_vjp(lib, tup, S=3, T=600, which="LK", dev=DEV, Qf=Qf)
    if Qf:
        got["Q"] = got["Q"] + got.pop("Qf")
    assert_grads_close(got, exp)


def _call(lib, S, T, ws, dt=torch.float64, stream=None):
    act, _ = random_actor(6, 2, 4, S, seed=5)
    act = {k: v.to(DEV, dt) for k, v in act.items()}
    g = torch.Generator().manual_seed(6)
    L_bar = torch.randn(S, T, 2, 6, generator=g, dtype=dt).to(DEV)
    K_bar = torch.randn(S, T, 6, 4, generator=g, dtype=dt).to(DEV)
    d = abi.LqgkDims(S, 1, T, 4, 6, 2, 4, 4)
    return lambda: lib.gains_vjp(d, act, L_bar=L_bar, K_bar=K_bar, ws=ws, stream=stream or torch.cuda.current_stream().cuda_stream)[0]


def test_chunked_workspace_gives_identical_gradients(lib):
    S, T = 100, 50
    d = abi.LqgkDims(S, 1, T, 4, 6, 2, 4, 4)
    big = torch.empty(lib.workspace_bytes(d, abi.MODE_GAINS_VJP, 0), dtype=torch.uint8, device=DEV)
    n32 = lib.lib.lqgk_workspace_bytes(abi.C.byref(d), abi.MODE_GAINS_VJP, 32)
    small = torch.empty(n32, dtype=torch.uint8, device=DEV)
    one, chunked = _call(lib, S, T, big)(), _call(lib, S, T, small)()
    for k in one:
        assert torch.equal(one[k], chunked[k]), k


def test_gains_vjp_is_capturable_into_a_cuda_graph_and_replays_identically(lib):
    lib.init(1)
    S, T = 64, 100
    d = abi.LqgkDims(S, 1, T, 4, 6, 2, 4, 4)
    ws = torch.empty(lib.workspace_bytes(d, abi.MODE_GAINS_VJP, 0), dtype=torch.uint8, device=DEV)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ref = {k: v.clone() for k, v in _call(lib, S, T, ws, torch.float32, st.cuda_stream)().items()}   # eager (sets kernel attributes)
    st.synchronize()
    call = _call(lib, S, T, ws, torch.float32)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        outs = call()
    for _ in range(2):
        for o in outs.values():
            o.fill_(float("nan"))
        ws.zero_()
        graph.replay()
        torch.cuda.synchronize()
        for k in ref:
            assert torch.equal(outs[k], ref[k]), k


def test_gradcheck_on_the_gpu():
    T = 8
    act, Sig = random_actor(6, 2, 4, 2, seed=3)
    m = {k: v.to(DEV).requires_grad_(True) for k, v in act.items()}
    Sig = Sig.to(DEV).requires_grad_(True)

    def gains(A, B, F, V, W, Q, R, Sigma0):
        sp = time_stack_spec(A, B, F, V, W, Q, R, T)
        return lqr.backward(sp).L, kf.forward(sp, Sigma0)
    assert torch.autograd.gradcheck(gains, tuple(m[k] for k in abi.ACTOR_KEYS) + (Sig,))


def test_batched_model_gradients_match_the_oracle_on_sampled_rows():
    """4,096 parameter samples through SubjectiveActor(dim=2): every gradient finite, 8 rows against the oracle's autograd."""
    S, T = 4096, 100
    g, = theta_grads(S, T, seed=1, dev=DEV, oracle=False)
    assert torch.isfinite(g).all()
    rows = np.sort(np.random.default_rng(2).choice(S, 8, replace=False))
    g8, go8 = theta_grads(S, T, seed=1, dev=DEV, rows=rows)
    assert torch.allclose(g8, g[rows], rtol=1e-12, atol=0)   # (the same samples in a smaller batch)
    assert torch.allclose(g8, go8, rtol=1e-8, atol=1e-10 * go8.abs().max().item()), (g8 - go8).abs().max()


def test_calls_without_gradients_make_the_launches_they_made_before(lib):
    """A spec that does not require grad takes the plain gains call: pack, sweep and one store per output."""
    act, _ = random_actor(6, 2, 4, 16, seed=2)
    sp = time_stack_spec(*(act[k].to(DEV) for k in abi.ACTOR_KEYS), 50)
    lqr.backward(sp)
    assert lib.last_launch_count() == 5   # pack, k_lqr_fwd, L, l and H out
    kf.forward(sp, None)
    assert lib.last_launch_count() == 3   # pack, k_kf_fwd, K out
    spg = time_stack_spec(*(act[k].to(DEV).requires_grad_(True) for k in abi.ACTOR_KEYS), 50)
    L = lqr.backward(spg).L
    assert lib.last_launch_count() == 5 and L.requires_grad
