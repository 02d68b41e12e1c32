"""Likelihood under signal-dependent noise (extension, NO reference counterpart -> parity unpinned by the reference; spec:
oracle/sdn_np.py).  not-gpu: the oracle is pinned (a) by its exact reduction to the reference-restating oracle when the
multiplicative noise vanishes, (b) by Monte Carlo simulation of the generative model (the moment recursion is exact for the
unconditional first two moments), (c) the kernels' step functions (host build, tests/emul) reproduce the oracle.
gpu: the CUDA kernel against the oracle, and its reduction to lqgk_loglik_fwd at zero multiplicative noise."""
import numpy as np
import pytest
import torch

from lqg_b200 import abi
from oracle import lqg_np as O
from oracle import sdn_np as S
from tests import helpers as H

T = 40


def _system(name="subjective", T=T, **kw):
    mats = H.model_mats(name, **kw)
    sa, sd = O.make_system(mats, T)
    L, _, _ = O.lqr_backward(sa)
    K = O.kf_forward(sa, sa["V"][0] @ sa["V"][0].T)
    return mats, sa, sd, L, K


def _noise(sd, c_mult, d_mult):
    """Control-dependent motor noise along B (|u|-proportional) and state-dependent observation noise along F."""
    return [c_mult * sd["B"][0]], [d_mult * sd["F"][0]]


def test_oracle_reduces_to_reference_without_multiplicative_noise():
    mats, sa, sd, L, K = _system()
    X = O.simulate(sa, sd, 4, np.random.default_rng(0))
    assert np.abs(S.sdn_log_likelihood(sa, sd, L, K, [], [], X) - O.log_likelihood(sa, sd, X)).max() < 1e-10
    mus, Sigs = S.sdn_conditional_moments(sa, sd, L, K, [], [], X[0])
    mr, Sr = O.conditional_moments(sa, sd, X[0])
    assert np.abs(mus - mr).max() < 1e-10 and np.abs(Sigs - Sr).max() < 1e-10


def test_moment_recursion_matches_monte_carlo():
    mats, sa, sd, L, K = _system(T=30)
    C, D = _noise(sd, 60.0, 0.6)
    x0 = np.array([2.0, -1.0])
    mus, Sigs = S.sdn_moments(sa, sd, L, K, C, D, x0=x0)
    m0, S0 = S.sdn_moments(sa, sd, L, K, [], [], x0=x0)
    assert np.abs(Sigs[-1] - S0[-1]).max() > 0.2 * np.abs(S0[-1]).max()      # the multiplicative terms matter here
    n = 300000
    xs, xh = S.sdn_simulate(sa, sd, L, K, C, D, n, np.random.default_rng(1), x0=x0)
    for t in (10, 30):
        z = np.concatenate([xs[:, t], xh[:, t]], axis=1)
        sd_t = np.sqrt(np.diag(Sigs[t]))
        assert np.abs(z.mean(0) - mus[t]).max() < 5 * sd_t.max() / np.sqrt(n)
        emp = np.cov(z.T)
        assert np.abs(emp - Sigs[t]).max() < 0.02 * np.abs(Sigs[t]).max(), (t, np.abs(emp - Sigs[t]).max() / np.abs(Sigs[t]).max())


def test_true_noise_model_explains_sdn_data_better():
    mats, sa, sd, L, K = _system(T=60)
    C, D = _noise(sd, 60.0, 0.6)
    xs, _ = S.sdn_simulate(sa, sd, L, K, C, D, 64, np.random.default_rng(2))
    ll_true = S.sdn_log_likelihood(sa, sd, L, K, C, D, xs)
    ll_plain = S.sdn_log_likelihood(sa, sd, L, K, [], [], xs)
    assert ll_true.mean() > ll_plain.mean()


def _run_library(lib, dev, name, S_, N, c_mults, d_mults, dtype, T_=T, seed=0, shared_noise=False, d=None):
    x, b, u, y = H.MODEL_DIMS[name]
    params = H.jittered_params(name, S_, seed)
    mats = [H.model_mats(name, **kw) for kw in params]
    sys = [O.make_system(m, T_) for m in mats]
    gains = [(O.lqr_backward(sa)[0], O.kf_forward(sa, sa["V"][0] @ sa["V"][0].T)) for sa, _ in sys]
    noise = [_noise(sd, c_mults[0 if shared_noise else s], d_mults[0 if shared_noise else s]) for s, (_, sd) in enumerate(sys)]
    rng = np.random.default_rng(seed + 1)
    d = d if d is not None else {"hand": 2, "pointmass": 2}.get(name, x)   # observed dims of the compiled tuple
    X = S.sdn_simulate(sys[0][0], sys[0][1], *gains[0], *noise[0], N, rng)[0][..., :d].astype(np.float32)
    ref = np.stack([S.sdn_log_likelihood(sa, sd, Lk[0], Lk[1], nz[0] if c_mults[0] else [], nz[1] if d_mults[0] else [],
                                         X.astype(np.float64)) for (sa, sd), Lk, nz in zip(sys, gains, noise)])
    t = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)
    act = {k: t(np.stack([m[0][k] for m in mats])) for k in "ABFVWQR"}
    dyn = {k: t(np.stack([m[1][k] for m in mats])) for k in "ABFVW"}
    Lt, Kt = t(np.stack([g[0] for g in gains])), t(np.stack([g[1] for g in gains]))
    Cn = t(np.stack([np.stack(nz[0]) for nz in noise])) if c_mults[0] else None
    Dn = t(np.stack([np.stack(nz[1]) for nz in noise])) if d_mults[0] else None
    if shared_noise:
        Cn = Cn[0] if Cn is not None else None
        Dn = Dn[0] if Dn is not None else None
    x_tm = torch.tensor(np.ascontiguousarray(X.transpose(1, 0, 2)), dtype=torch.float32, device=dev)
    dims = abi.LqgkDims(S_, N, T_, x, b, u, y, d)
    ll = lib.sdn_loglik(dims, act, dyn, Lt, Kt, x_tm, Cn, Dn)
    if dev.type == "cuda":
        torch.cuda.synchronize()
    return ll.double().cpu().numpy(), ref, (dims, act, dyn, x_tm)


@pytest.mark.parametrize("name", ["subjective", "bounded", "relobs", "subjective2", "hand"])
def test_step_functions_match_oracle_on_host(name):
    lib = abi.Library(H.EMUL_PATH)
    S_ = 3
    ll, ref, _ = _run_library(lib, torch.device("cpu"), name, S_, 3, [60.0, 20.0, 90.0], [0.6, 0.2, 0.9], torch.float64)
    assert np.allclose(ll, ref, rtol=1e-9, atol=1e-9), np.abs(ll - ref).max()
    ll0, ref0, _ = _run_library(lib, torch.device("cpu"), name, S_, 3, [0.0] * 3, [0.0] * 3, torch.float64)
    assert np.allclose(ll0, ref0, rtol=1e-9, atol=1e-9)
    assert np.abs(ll - ll0).max() > 1e-3 * np.abs(ll0).max()          # the multiplicative terms change the answer


@pytest.mark.gpu
@pytest.mark.parametrize("name,dtype,tol", [("subjective", torch.float64, 1e-9), ("subjective", torch.float32, 1e-4),
                                            ("bounded", torch.float64, 1e-9), ("relobs", torch.float64, 1e-9),
                                            ("subjective2", torch.float64, 1e-9), ("hand", torch.float64, 1e-8)])
def test_cuda_kernel_matches_oracle(name, dtype, tol):
    lib = abi.load_library()
    dev = torch.device("cuda:0")
    S_, N = 5, 7
    rng = np.random.default_rng(5)
    cm, dm = list(60.0 * np.exp(0.3 * rng.standard_normal(S_))), list(0.6 * np.exp(0.3 * rng.standard_normal(S_)))
    ll, ref, _ = _run_library(lib, dev, name, S_, N, cm, dm, dtype)
    assert np.allclose(ll, ref, rtol=tol, atol=tol * 10), np.abs(ll - ref).max()
    ll, ref, _ = _run_library(lib, dev, name, S_, N, cm, dm, dtype, shared_noise=True)
    assert np.allclose(ll, ref, rtol=tol, atol=tol * 10)


@pytest.mark.gpu
def test_cuda_kernel_reduces_to_the_main_path_without_multiplicative_noise():
    """nc = nd = 0: lqgk_sdn_loglik == lqgk_loglik_fwd (whose per-trial part is FP32) == the reference-restating oracle."""
    lib = abi.load_library()
    dev = torch.device("cuda:0")
    ll, ref, (dims, act, dyn, x_tm) = _run_library(lib, dev, "subjective", 4, 9, [0.0] * 4, [0.0] * 4, torch.float64, T_=200)
    assert np.allclose(ll, ref, rtol=1e-10, atol=1e-9)
    ws = torch.empty(lib.workspace_bytes(dims, abi.MODE_FWD, 0), dtype=torch.uint8, device=dev)
    main = lib.loglik_fwd(dims, act, dyn, x_tm, ws=ws, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.allclose(main.double().cpu().numpy(), ll, rtol=1e-5), np.abs(main.double().cpu().numpy() - ll).max()


def _channel_noise_np(sd, c_scale, d_scale):
    """NumPy twin of lqg_b200.control.sdn.channel_noise."""
    Bd, Fd = sd["B"][0], sd["F"][0]
    C = [c_scale * np.outer(Bd[:, i], np.eye(Bd.shape[1])[i]) for i in range(Bd.shape[1])]
    D = [d_scale * np.outer(np.eye(Fd.shape[0])[j], Fd[j]) for j in range(Fd.shape[0])]
    return C, D


def test_per_channel_noise_keeps_the_axes_of_a_2d_model_independent():
    """What System.log_likelihood_sdn relies on for dim > 1 models: with per-channel proportional noise the likelihood of the
    2-axis model is the sum of the 1-axis model's likelihoods on each axis' (target, cursor) columns."""
    T_ = 25
    m2, sa2, sd2, L2, K2 = _system("subjective2", T=T_)
    m1, sa1, sd1, L1, K1 = _system("subjective", T=T_)
    C2, D2 = _channel_noise_np(sd2, 60.0, 0.6)
    C1, D1 = _channel_noise_np(sd1, 60.0, 0.6)
    X = S.sdn_simulate(sa2, sd2, L2, K2, C2, D2, 3, np.random.default_rng(4))[0]
    ll2 = S.sdn_log_likelihood(sa2, sd2, L2, K2, C2, D2, X)
    d = X.shape[-1] // 2
    ll1 = sum(S.sdn_log_likelihood(sa1, sd1, L1, K1, C1, D1, X[..., a * d:(a + 1) * d]) for a in range(2))
    assert np.allclose(ll2, ll1, rtol=1e-10), (ll2, ll1)


def test_channel_noise_matches_its_numpy_twin():
    from lqg_b200.control import sdn
    from lqg_b200.tracking import SubjectiveActor
    for dim in (1, 2):
        model = SubjectiveActor(dim=dim, T=10, dtype=torch.float64, device="cpu")
        _, sa, sd, _, _ = _system("subjective" if dim == 1 else "subjective2", T=10)
        C, D = _channel_noise_np(sd, 3.0, 0.25)
        assert np.allclose(sdn.channel_noise(model, 3.0, "control").numpy(), np.stack(C))
        assert np.allclose(sdn.channel_noise(model, 0.25, "observation").numpy(), np.stack(D))
    model = SubjectiveActor(dim=1, T=10, dtype=torch.float64, sigma_target=torch.tensor([5.0, 6.0, 7.0], dtype=torch.float64))
    Cb = sdn.channel_noise(model, torch.tensor([1.0, 2.0, 3.0], dtype=torch.float64), "control")
    assert tuple(Cb.shape) == (3, 1, 2, 1) and np.allclose(Cb[2].numpy(), 3.0 * np.stack(_channel_noise_np(sd := _system("subjective", T=10)[2], 1.0, 0.0)[0]))


def test_batched_central_differences():
    from lqg_b200.control import sdn
    th = torch.tensor([0.7, -1.3, 2.0], dtype=torch.float64)
    f = lambda Th: (Th ** 3).sum(-1) + Th[:, 0] * Th[:, 1]
    v, g = sdn.value_and_grad_fd(f, th)
    assert abs(float(v) - float(f(th[None])[0])) < 1e-12
    assert np.allclose(g.numpy(), (3 * th ** 2 + torch.tensor([th[1], th[0], 0.0])).numpy(), rtol=1e-7)


@pytest.mark.gpu
def test_public_api_sdn_likelihood_and_fd_gradient():
    """System.log_likelihood_sdn on the GPU: dim=2 model factorised over axes == oracle on the 2-axis system; batched
    central-difference gradient through the model constructor == oracle finite differences."""
    from lqg_b200.control import sdn
    from lqg_b200.tracking import SubjectiveActor
    dev = torch.device("cuda:0")
    T_ = 60
    m2, sa2, sd2, L2, K2 = _system("subjective2", T=T_)
    C2, D2 = _channel_noise_np(sd2, 60.0, 0.6)
    X = S.sdn_simulate(sa2, sd2, L2, K2, C2, D2, 6, np.random.default_rng(7))[0].astype(np.float32)
    ref = S.sdn_log_likelihood(sa2, sd2, L2, K2, C2, D2, X.astype(np.float64))
    xg = torch.tensor(X, device=dev)
    model = SubjectiveActor(dim=2, T=T_, dtype=torch.float64, device=dev)
    ll = model.log_likelihood_sdn(xg, signal_dep_noise=60.0, obs_dep_noise=0.6)
    assert np.allclose(ll.cpu().numpy(), ref, rtol=1e-8), np.abs(ll.cpu().numpy() - ref).max()
    # unfactorised kernel on the full 2-axis system (explicit matrices)
    ll_full = model.log_likelihood_sdn(xg, C=torch.tensor(np.stack(C2), device=dev), D=torch.tensor(np.stack(D2), device=dev))
    assert np.allclose(ll_full.cpu().numpy(), ref, rtol=1e-8)

    names = ("action_cost", "sigma_target", "signal_dep_noise", "obs_dep_noise")
    th0 = torch.tensor([1.0, 6.0, 60.0, 0.6], dtype=torch.float64, device=dev)

    def total(Th):
        mdl = SubjectiveActor(dim=2, T=T_, dtype=torch.float64, device=dev, action_cost=Th[:, 0], sigma_target=Th[:, 1])
        return mdl.log_likelihood_sdn(xg, signal_dep_noise=Th[:, 2], obs_dep_noise=Th[:, 3]).sum(-1)

    v, g = sdn.value_and_grad_fd(total, th0)
    assert abs(float(v) - ref.sum()) < 1e-8 * abs(ref.sum())

    def total_np(th):
        mats = O.subjective_actor_mats(dim=2, action_cost=th[0], sigma_target=th[1])
        sa, sd = O.make_system(mats, T_)
        L, _, _ = O.lqr_backward(sa)
        K = O.kf_forward(sa, sa["V"][0] @ sa["V"][0].T)
        C, D = _channel_noise_np(sd, th[2], th[3])
        return S.sdn_log_likelihood(sa, sd, L, K, C, D, X.astype(np.float64)).sum()

    th = th0.cpu().numpy()
    for p in range(len(names)):
        h = 1e-5 * abs(th[p])
        e = np.zeros_like(th); e[p] = h
        g_ref = (total_np(th + e) - total_np(th - e)) / (2 * h)
        assert abs(float(g[p]) - g_ref) <= 1e-4 * abs(g_ref) + 1e-7, (names[p], float(g[p]), g_ref)


def test_all_fp64_path_point_mass_with_four_observed_states_on_host():
    """Tuple (4,4,1,3,4) is compiled for the all-FP64 per-trial kernel only (lqgk_dims.h: LQGK_FOR_EACH_FP64_ONLY_DIMS)."""
    lib = abi.Library(H.EMUL_PATH)
    ll, ref, _ = _run_library(lib, torch.device("cpu"), "pointmass", 2, 3, [0.0] * 2, [0.0] * 2, torch.float64, T_=60, d=4)
    assert np.allclose(ll, ref, rtol=1e-8), np.abs(ll / ref - 1).max()


@pytest.mark.gpu
def test_log_likelihood_fp64_point_mass_all_states_observed():
    """PointMassBoundedActor with all four states observed (lqg/tracking/point_mass.py:7-47): innovation covariance with condition
    number ~1e9, out of reach of the FP32 per-trial arithmetic of the main path -> System.log_likelihood_fp64."""
    from lqg_b200.tracking import PointMassBoundedActor
    dev = torch.device("cuda:0")
    T_ = 200
    mats = O.point_mass_mats()
    sa, sd = O.make_system(mats, T_)
    X = O.simulate(sa, sd, 5, np.random.default_rng(11))
    ref = O.log_likelihood(sa, sd, X)
    model = PointMassBoundedActor(T=T_, dtype=torch.float64, device=dev)
    ll = model.log_likelihood_fp64(torch.tensor(X, device=dev))
    # observations are FP32 at the C ABI: evaluate the oracle on the same rounded data
    ref32 = O.log_likelihood(sa, sd, X.astype(np.float32).astype(np.float64))
    assert np.allclose(ll.cpu().numpy(), ref32, rtol=1e-6), (ll.cpu().numpy(), ref32, ref)


@pytest.mark.gpu
def test_per_condition_data_sets():
    """x_sample_stride != 0: every parameter sample (experimental condition) has its own trials (config c2's layout)."""
    from lqg_b200.tracking import SubjectiveActor
    dev = torch.device("cuda:0")
    T_, N, sig = 50, 4, [8.5, 19.9, 51.6]
    ref, xs = [], []
    for c, st in enumerate(sig):
        _, sa, sd, L, K = _system("subjective", T=T_, sigma_target=st)
        C, D = _channel_noise_np(sd, 40.0, 0.4)
        X = S.sdn_simulate(sa, sd, L, K, C, D, N, np.random.default_rng(20 + c))[0].astype(np.float32)
        xs.append(X)
        ref.append(S.sdn_log_likelihood(sa, sd, L, K, C, D, X.astype(np.float64)))
    model = SubjectiveActor(dim=1, T=T_, dtype=torch.float64, device=dev, sigma_target=torch.tensor(sig, dtype=torch.float64, device=dev))
    ll = model.log_likelihood_sdn(torch.tensor(np.stack(xs), device=dev), signal_dep_noise=40.0, obs_dep_noise=0.4)
    assert tuple(ll.shape) == (3, N) and np.allclose(ll.cpu().numpy(), np.stack(ref), rtol=1e-8)


def _route_python_api_to_host_harness(monkeypatch):
    """Runs the torch-facing API (lqg_b200.system / runtime / control.sdn) on HOST tensors against the CPU build of the kernels'
    step functions (tests/emul), so that `-m "not gpu"` covers the Python plumbing above the C ABI.  Test-only: the product path
    refuses CPU tensors and any library but the CUDA one."""
    from lqg_b200 import runtime
    from lqg_b200.control import sdn
    lib = abi.Library(H.EMUL_PATH)

    def solve(A, B, Hm, Q, R, Om_xi, Om_omega, Sigma1, xhat1, T, C=None, D=None, Qf=None, sweeps=10, form="predictor"):
        f = lambda v: None if v is None else torch.as_tensor(v).to(torch.float64)
        mats = dict(A=f(A), B=f(B), H=f(Hm), Q=f(Q), R=f(R), Qf=f(Qf), Om_xi=f(Om_xi), Om_omega=f(Om_omega), Sigma1=f(Sigma1),
                    xhat1=f(xhat1), C=f(C), D=f(D))
        return sdn.SDNGains(*lib.sdn_gains(mats, T, sweeps, filter_form=form == "filter"))

    monkeypatch.setattr(sdn, "solve", solve)
    monkeypatch.setattr(runtime, "_require_cuda", lambda *a, **k: None)
    monkeypatch.setattr(runtime, "_stream", lambda dev: 0)
    monkeypatch.setattr(abi, "load_library", lambda: lib)
    monkeypatch.setattr(lib, "pack_obs", lambda x, stream=0: x.permute(1, 0, 2).to(torch.float32).contiguous(), raising=False)
    return lib


def test_python_api_with_sdn_aware_actor_on_host(monkeypatch):
    """System.log_likelihood_sdn(gains="sdn") of a 2-axis model: per-axis factorisation -> filter-form gain iterations on the
    actor's model -> per-trial likelihood, against the oracle evaluated on the full 2-axis system."""
    from lqg_b200.tracking import SubjectiveActor
    _route_python_api_to_host_harness(monkeypatch)
    T_ = 40
    model = SubjectiveActor(dim=2, T=T_, dtype=torch.float64, device="cpu")
    _, sa, sd, _, _ = _system("subjective2", T=T_)
    Ca, Da = _channel_noise_np(sa, 40.0, 0.4)                       # the actor's own input / observation maps
    A0 = {k: sa[k][0] for k in "ABFVWQR"}
    Lo, Ko, _ = S.filter_solve(A=A0["A"], B=A0["B"], F=A0["F"], C=Ca, D=Da, Q=A0["Q"], R=A0["R"], Qf=A0["Q"], Om_xi=A0["V"] @ A0["V"].T,
                               Om_om=A0["W"] @ A0["W"].T, Sigma0=A0["V"] @ A0["V"].T, xhat0=np.zeros(6), T=T_, sweeps=6)
    C, D = _channel_noise_np(sd, 40.0, 0.4)
    X = S.sdn_simulate(sa, sd, Lo, Ko, C, D, 3, np.random.default_rng(0))[0].astype(np.float32)
    ref = S.sdn_log_likelihood(sa, sd, Lo, Ko, C, D, X.astype(np.float64))
    ll = model.log_likelihood_sdn(torch.tensor(X), signal_dep_noise=40.0, obs_dep_noise=0.4, gains="sdn")
    assert np.allclose(ll.numpy(), ref, rtol=1e-9), np.abs(ll.numpy() - ref).max()
    # an actor unaware of the multiplicative noise (the reference's own gains) gives a different likelihood
    # (explicit gains: the unfactorised 2-axis kernel; lqr.backward / kf.forward themselves need the GPU)
    L0, _, _ = O.lqr_backward(sa)
    K0 = O.kf_forward(sa, sa["V"][0] @ sa["V"][0].T)
    ll_plain = model.log_likelihood_sdn(torch.tensor(X), signal_dep_noise=40.0, obs_dep_noise=0.4, gains=(torch.tensor(L0), torch.tensor(K0)))
    assert np.allclose(ll_plain.numpy(), S.sdn_log_likelihood(sa, sd, L0, K0, C, D, X.astype(np.float64)), rtol=1e-9)
    assert np.abs(ll_plain.numpy() - ll.numpy()).max() > 1e-3


@pytest.mark.gpu
def test_sdn_simulator_matches_the_exact_moment_recursion():
    """lqgk_sdn_simulate (System.simulate_sdn): mean and covariance of the simulated (x, xhat)_t equal the oracle's EXACT
    unconditional moments (sdn_moments) where the multiplicative terms change the covariance by > 20 %."""
    from lqg_b200.tracking import SubjectiveActor
    dev = torch.device("cuda:0")
    T_, n, x0 = 30, 200000, [2.0, -1.0]
    model = SubjectiveActor(dim=1, T=T_, dtype=torch.float64, device=dev)
    x, xh, y, u = model.simulate_sdn(5, n=n, signal_dep_noise=60.0, obs_dep_noise=0.6, x0=x0, return_all=True)
    assert tuple(x.shape) == (n, T_ + 1, 2) and tuple(xh.shape) == (n, T_ + 1, 3)
    _, sa, sd, L, K = _system("subjective", T=T_)
    C, D = _channel_noise_np(sd, 60.0, 0.6)
    mus, Sigs = S.sdn_moments(sa, sd, L, K, C, D, x0=np.array(x0))
    _, S0 = S.sdn_moments(sa, sd, L, K, [], [], x0=np.array(x0))
    assert np.abs(Sigs[-1] - S0[-1]).max() > 0.2 * np.abs(S0[-1]).max()
    for t in (10, T_):
        z = torch.cat([x[:, t], xh[:, t]], 1).cpu().numpy()
        assert np.abs(z.mean(0) - mus[t]).max() < 5 * np.sqrt(np.diag(Sigs[t])).max() / np.sqrt(n)
        emp = np.cov(z.T)
        assert np.abs(emp - Sigs[t]).max() < 0.02 * np.abs(Sigs[t]).max(), (t, np.abs(emp - Sigs[t]).max() / np.abs(Sigs[t]).max())
    # the simulated data are plausible under the matching likelihood model: higher mean log-likelihood than without the noise terms
    xs = x[:512].to(torch.float32)
    assert model.log_likelihood_sdn(xs, signal_dep_noise=60.0, obs_dep_noise=0.6).mean() > model.log_likelihood_sdn(xs).mean()


def test_oracle_gradient_by_autograd_equals_central_differences():
    """The reference gradient of the signal-dependent-noise likelihood in the GPU tests is a central difference of the NumPy
    oracle; an independent torch-autograd twin of the same recursion (oracle/lqg_torch.py) gives the same value and gradient."""
    from oracle import lqg_torch as OT
    T_ = 25
    th0 = np.array([1.0, 6.0, 40.0, 0.4])                              # action_cost, sigma_target, signal_dep_noise, obs_dep_noise

    def total_np(th):
        mats = O.subjective_actor_mats(dim=1, action_cost=th[0], sigma_target=th[1])
        sa, sd = O.make_system(mats, T_)
        L, _, _ = O.lqr_backward(sa)
        K = O.kf_forward(sa, sa["V"][0] @ sa["V"][0].T)
        C, D = _channel_noise_np(sd, th[2], th[3])
        return S.sdn_log_likelihood(sa, sd, L, K, C, D, X).sum()

    _, sa, sd, L, K = _system("subjective", T=T_)
    X = S.sdn_simulate(sa, sd, L, K, *_channel_noise_np(sd, 40.0, 0.4), 3, np.random.default_rng(9))[0]
    th = torch.tensor(th0, dtype=torch.float64, requires_grad=True)
    a, d = OT.subjective_actor(dim=1, action_cost=th[0], sigma_target=th[1])
    ll = OT.sdn_log_likelihood(a, d, torch.tensor(X), th[2], th[3])
    ll.sum().backward()
    assert abs(ll.sum().item() - total_np(th0)) < 1e-9 * abs(total_np(th0))
    for p in range(4):
        h = 1e-5 * th0[p]
        e = np.zeros(4); e[p] = h
        fd = (total_np(th0 + e) - total_np(th0 - e)) / (2 * h)
        assert abs(th.grad[p].item() - fd) <= 1e-5 * abs(fd) + 1e-8, (p, th.grad[p].item(), fd)
