"""The torch-facing drop-in layer (lqg_b200.system / tracking / runtime: per-axis factorisation, autograd Function around the
fused forward+adjoint call, per-condition data, per-trial cotangents) run on HOST tensors against the CPU build of the
kernels' own step functions (tests/emul/liblqgk_emul.so), so that `-m "not gpu"` covers the Python glue above the C ABI with
the same assertions as tests/test_gpu_api.py.  Test-only routing: the product path refuses CPU tensors and any library but
the CUDA one (test_gpu_api.py::test_no_cpu_fallback)."""
import numpy as np
import pytest
import torch

from lqg_b200 import System, abi, runtime, tracking
from oracle import lqg_np as O
from oracle import lqg_torch as OT
from tests import helpers as H


@pytest.fixture
def host(monkeypatch):
    lib = abi.Library(H.EMUL_PATH)
    monkeypatch.setattr(runtime, "_require_cuda", lambda *a, **k: None)
    monkeypatch.setattr(runtime, "_stream", lambda dev: 0)
    monkeypatch.setattr(runtime, "workspace", lambda dev, need: None)
    monkeypatch.setattr(abi, "load_library", lambda: lib)
    return lib


def _sim(mats, T, N, seed=0):
    sa, sd = O.make_system(mats, T)
    return O.simulate(sa, sd, N, np.random.default_rng(seed))


@pytest.mark.parametrize("dim", [1, 2])
def test_log_likelihood_and_parameter_gradient(host, dim):
    """(tests/test_gpu_api.py::test_log_likelihood_and_parameter_gradient on the host harness, float64 I/O)"""
    T, N, S = 60, 5, 3
    X = _sim(O.subjective_actor_mats(dim=dim, sigma_target=9.0), T, N, seed=4).astype(np.float32)
    names = ["action_cost", "action_variability", "subj_noise", "subj_vel_noise", "sigma_target", "sigma_cursor"]
    th_np = np.array([1.0, 0.5, 1.0, 0.5, 9.0, 6.0])[None] * np.exp(0.2 * np.random.default_rng(5).standard_normal((S, 6)))
    tho = torch.tensor(th_np, dtype=torch.float64, requires_grad=True)
    a, d = OT.subjective_actor(dim=dim, **{n: tho[:, i] for i, n in enumerate(names)})
    llo = OT.log_likelihood(a, d, torch.tensor(X, dtype=torch.float64))
    llo.sum().backward()
    th = torch.tensor(th_np, dtype=torch.float64, requires_grad=True)
    m = tracking.SubjectiveActor(dim=dim, T=T, **{n: th[:, i] for i, n in enumerate(names)})
    ll = m.log_likelihood(torch.tensor(X))
    assert ll.shape == (S, N)
    ll.sum().backward()
    assert np.allclose(ll.detach().numpy(), llo.detach().numpy(), rtol=1e-5)
    g, go = th.grad.numpy(), tho.grad.numpy()
    assert np.allclose(g, go, rtol=1e-3, atol=1e-5 * np.abs(go).max(axis=1, keepdims=True)), np.abs(g / go - 1).max()
    if dim == 2:   # the general (un-factorised, n = 10) step functions give the same numbers
        ll2 = System(m.actor, m.dynamics).log_likelihood(torch.tensor(X))
        assert np.allclose(ll2.detach().numpy(), llo.detach().numpy(), rtol=1e-5)


def test_per_trial_weights_take_the_explicit_adjoint_path(host):
    T, N = 50, 6
    X = torch.tensor(_sim(O.bounded_actor_mats(), T, N, seed=2).astype(np.float32))
    sig = torch.tensor(6.0, dtype=torch.float64, requires_grad=True)
    ll = tracking.BoundedActor(T=T, sigma_target=sig).log_likelihood(X)
    assert ll.shape == (N,)
    w = torch.linspace(0.5, 1.5, N, dtype=torch.float64)
    (ll * w).sum().backward()
    so = torch.tensor(6.0, dtype=torch.float64, requires_grad=True)
    a, d = OT.bounded_actor(sigma_target=so)
    (OT.log_likelihood(a, d, X.double()) * w).sum().backward()
    assert np.isclose(sig.grad.item(), so.grad.item(), rtol=1e-3)


def test_per_condition_data_in_one_call(host):
    """Config c2's layout: one sample per condition, each with its own trials (lqg/infer/models.py:38-61 loops over them)."""
    T, N, sig = 50, 4, [8.5, 19.9, 51.6]
    Xs, lls, grads = [], [], []
    for c, s_t in enumerate(sig):
        X = _sim(O.subjective_actor_mats(dim=2, sigma_target=s_t), T, N, seed=10 + c).astype(np.float32)
        Xs.append(X)
        so = torch.tensor(s_t, dtype=torch.float64, requires_grad=True)
        a, d = OT.subjective_actor(dim=2, sigma_target=so)
        ll = OT.log_likelihood(a, d, torch.tensor(X, dtype=torch.float64))
        ll.sum().backward()
        lls.append(ll.detach().numpy()); grads.append(so.grad.item())
    st = torch.tensor(sig, dtype=torch.float64, requires_grad=True)
    ll = tracking.SubjectiveActor(dim=2, T=T, sigma_target=st).log_likelihood(torch.tensor(np.stack(Xs)))
    assert ll.shape == (len(sig), N)
    ll.sum().backward()
    assert np.allclose(ll.detach().numpy(), np.stack(lls), rtol=1e-5)
    assert np.allclose(st.grad.numpy(), np.array(grads), rtol=1e-3)


@pytest.mark.parametrize("name,cls,kw", [("subjective", tracking.SubjectiveActor, {}), ("bounded2", tracking.BoundedActor, {"dim": 2})])
def test_predictive_moments(host, name, cls, kw):
    """runtime.moments (what System.conditional_moments / belief_tracking_distribution call on the GPU, lqg/system.py:142-235,
    250-257): mu[n, T, nj], Sigma[T, nj, nj] against the oracle's literal restatement of the reference scan."""
    T, N = 40, 3
    mats = H.model_mats(name)
    X = _sim(mats, T, N, seed=3).astype(np.float32)
    model = cls(T=T, dtype=torch.float64, device="cpu", **kw)
    mu, Sig = runtime.moments(model.actor, model.dynamics, torch.tensor(X))
    sa, sd = O.make_system(mats, T)
    for i in range(N):
        mo, So = O.conditional_moments(sa, sd, X[i].astype(np.float64))
        assert np.allclose(mu[i].numpy(), mo, rtol=1e-4, atol=1e-4 * np.abs(mo).max()), (i, np.abs(mu[i].numpy() - mo).max())
        assert np.allclose(Sig.numpy(), So, rtol=1e-9, atol=1e-12)
