"""The adjoint of the gain sweeps (lqgk_gains_vjp_*) and the autograd it gives lqr.backward / kf.forward, on the host build
of the kernels' step functions (tests/emul/liblqgk_emul_gains.so): gradients against torch autograd through the float64 oracle
(oracle/lqg_torch.py), the entry points' argument checks (against liblqgk.so too, with fake pointers), and the Python layer
(gradcheck, parameter gradients of a tracking model).  tests/test_gpu_gains_vjp.py runs the same comparison on the GPU."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from lqg_b200 import abi, runtime, tracking
from lqg_b200.belief import kf
from lqg_b200.control import lqr
from lqg_b200.dims import SUPPORTED_DIMS
from lqg_b200.utils import time_stack_spec
from oracle import lqg_torch as OT
from tests import helpers as H
from tests.test_entry_point_checks import ACT7, BIG_WS, FAKE, INVALID, UNSUPPORTED, WORKSPACE, P, _in_child, dims, ref, spec

EMUL_GAINS_PATH = os.path.join(H.ROOT, "tests", "emul", "liblqgk_emul_gains.so")   # (built by __graft_entry__.build)
GAINS_TUPLES = sorted({t[:4] for t in SUPPORTED_DIMS})
SUBJ = ["action_cost", "action_variability", "subj_noise", "subj_vel_noise", "sigma_target", "sigma_cursor"]


# ------------------------------------------------------------------------------------------ ABI against torch autograd
def random_actor(b, u, y, S, seed):
    """Per-sample actor matrices of a stable, well-conditioned system (F shared by the samples: a stride-0 sample axis)."""
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    eye = lambda n: torch.eye(n, dtype=torch.float64)
    Mq, Mr, Ms = r(S, b, b), r(S, u, u), r(S, b, b)
    return dict(A=0.9 * eye(b) + 0.05 * r(S, b, b) / b ** 0.5, B=0.5 * r(S, b, u), F=r(1, y, b),
                V=0.3 * eye(b) + 0.05 * r(S, b, b), W=eye(y) + 0.1 * r(S, y, y), Q=Mq @ Mq.mT / b + 0.1 * eye(b),
                R=Mr @ Mr.mT / u + 0.5 * eye(u)), Ms @ Ms.mT / b + 0.1 * eye(b)


def oracle_grads(act, T, L_bar, K_bar, Sigma0=None):
    """Gradients of <L_bar, L> + <K_bar, K> by torch autograd through oracle/lqg_torch.py (Q, R, Sigma0 enter symmetrised,
    as the kernels read them; the Riccati sweep starts from Q, as lqg/utils.py:30 builds Qf)."""
    m = {k: v.detach().clone().requires_grad_(True) for k, v in act.items()}
    s0 = None if Sigma0 is None else Sigma0.detach().clone().requires_grad_(True)
    sym = lambda X: 0.5 * (X + X.mT)
    loss = 0.0
    if L_bar is not None:
        L = OT.lqr_backward(m["A"], m["B"], sym(m["Q"]), sym(m["R"]), T)
        loss = loss + (L.transpose(0, 1) * L_bar).sum()
    if K_bar is not None:
        P0 = m["V"] @ m["V"].mT if s0 is None else sym(s0)
        K = OT.kf_forward(m["A"], m["F"], m["V"], m["W"], P0, T)
        loss = loss + (K.transpose(0, 1) * K_bar).sum()
    leaves = list(m.values()) + ([s0] if s0 is not None else [])
    gs = torch.autograd.grad(loss, leaves, allow_unused=True)
    return {k: torch.zeros_like(v) if g is None else g for (k, v), g in zip(list(m.items()) + [("Sigma0", s0)], gs)}


def run_vjp(lib, tup, S, T, which, dev="cpu", dt=torch.float64, Qf=False, with_sigma0=False, seed=0, ws=None):
    """(kernel gradients, oracle gradients) of <L_bar, L> + <K_bar, K> for random cotangents; which: "L", "K" or "LK"."""
    x, b, u, y = tup
    act, Sig = random_actor(b, u, y, S, seed)
    g = torch.Generator().manual_seed(seed + 1)
    L_bar = torch.randn(S, T, u, b, generator=g, dtype=torch.float64) if "L" in which else None
    K_bar = torch.randn(S, T, b, y, generator=g, dtype=torch.float64) if "K" in which else None
    Sigma0 = Sig if with_sigma0 else None
    want = abi.ACTOR_KEYS + (("Qf",) if Qf else ())
    mats = {k: v.to(dev, dt) for k, v in act.items()}
    if Qf:
        mats["Qf"] = mats["Q"].clone()
    d = abi.LqgkDims(S, 1, T, x, b, u, y, 1)
    to = lambda t: None if t is None else t.to(dev, dt)
    if ws is None and dev != "cpu":
        ws = torch.empty(lib.workspace_bytes(d, abi.MODE_GAINS_VJP, 0), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream if dev != "cpu" else 0
    got, gs = lib.gains_vjp(d, mats, sigma0=to(Sigma0), L_bar=to(L_bar), K_bar=to(K_bar), want=want, ws=ws, stream=st)
    got = {k: v.double().cpu() for k, v in got.items()}
    got["F"] = got["F"].sum(0, keepdim=True)   # F is shared by the samples
    if gs is not None:
        got["Sigma0"] = gs.double().cpu()
    exp = oracle_grads(act, T, L_bar, K_bar, Sigma0=Sigma0)
    return got, exp


def assert_grads_close(got, exp, rel=1e-8, rtol=0.0):
    for k, g in got.items():
        e = exp[k]
        scale = max(e.abs().max().item(), 1e-300)
        err = (g - e).abs()
        assert bool((err <= rel * scale + rtol * e.abs()).all()), (k, (err.max() / scale).item())


@pytest.fixture(scope="module")
def emul():
    return abi.Library(EMUL_GAINS_PATH)


@pytest.mark.parametrize("which", ["L", "K", "LK"])
@pytest.mark.parametrize("tup", GAINS_TUPLES, ids=lambda t: "x%db%du%dy%d" % t)
def test_vjp_matches_torch_autograd(emul, tup, which):
    got, exp = run_vjp(emul, tup, S=3, T=40, which=which)
    assert_grads_close(got, exp)


@pytest.mark.parametrize("Qf, with_sigma0", [(False, False), (True, False), (False, True), (True, True)])
def test_defaulted_and_explicit_terminal_cost_and_prior(emul, Qf, with_sigma0):
    """Qf absent -> its gradient is Q's; an explicit Qf (here equal to Q) gets its own, and Q's + Qf's is the oracle's Q
    gradient.  Sigma0 absent -> V V^T and its gradient goes to V; an explicit Sigma0 gets its own."""
    got, exp = run_vjp(emul, (4, 6, 2, 4), S=3, T=40, which="LK", Qf=Qf, with_sigma0=with_sigma0)
    if Qf:
        q, qf = got.pop("Q"), got.pop("Qf")
        assert qf.abs().max() > 0
        got["Q"] = q + qf
    assert ("Sigma0" in got) == with_sigma0
    assert_grads_close(got, {k: exp[k] for k in got})


# ------------------------------------------------------------------------------------------ argument checks
def gains_vjp(lib, p, d=None, act=None, L_bar=FAKE, K_bar=FAKE, ws=FAKE, ws_bytes=BIG_WS):
    d = dims() if d is None else d
    act = spec(ACT7) if act is None else act
    ga = abi.LqgkSpecGrad()
    return getattr(lib, "lqgk_gains_vjp_" + p)(ref(d) if d != "null" else None, ref(act) if act != "null" else None, None,
                                                C.c_double(1e-8), P(L_bar), P(K_bar), ref(ga), None, P(ws), C.c_size_t(ws_bytes),
                                                P(None))


def _with_P():
    sp = spec(ACT7)
    sp.P = abi.LqgkMat(FAKE, 0, 0)
    return sp


CASES = [
    ("no-cotangent", dict(L_bar=None, K_bar=None), INVALID, False),
    ("null-dims", dict(d="null"), INVALID, False),
    ("null-actor", dict(act="null"), INVALID, False),
    *[(f"null-{k}", dict(act=spec(ACT7, null=k)), INVALID, False) for k in ACT7],
    ("zero-samples", dict(d=dims(S=0)), INVALID, False),
    ("time-varying", dict(act=spec(ACT7, tv="A")), UNSUPPORTED, False),
    ("time-varying-L-only", dict(act=spec(ACT7, tv="R"), K_bar=None), UNSUPPORTED, False),
    ("cross-cost", dict(act=_with_P()), UNSUPPORTED, False),
    ("unsupported-tuple", dict(d=dims(x=3, b=7, u=1, y=2, d=2)), UNSUPPORTED, False),
    ("workspace-null", dict(ws=None), INVALID, True),
    ("workspace-misaligned", dict(ws=FAKE + 64), INVALID, True),
    ("workspace-too-small", dict(ws_bytes=1 << 10), WORKSPACE, True),
]


def _params(ws_cases):
    return [pytest.param(kw, p, want, id=f"{cid}-{p}") for cid, kw, want, ws in CASES if ws_cases or not ws for p in ("f32", "f64")]


@pytest.mark.parametrize("kw, p, want", _params(True))
def test_library_rejects(kw, p, want):
    assert gains_vjp(C.CDLL(abi.LIB_PATH), p, **kw) == want


@pytest.mark.parametrize("kw, p, want", _params(False))
def test_host_build_rejects(kw, p, want):
    lib = C.CDLL(EMUL_GAINS_PATH)
    assert _in_child(lambda: gains_vjp(lib, p, **kw)) == want


def test_workspace_bytes():
    fn = C.CDLL(abi.LIB_PATH).lqgk_workspace_bytes
    fn.restype = C.c_size_t
    wb = lambda d, chunk=0: fn(ref(d), C.c_int(abi.MODE_GAINS_VJP), C.c_int32(chunk))
    for x, b, u, y in GAINS_TUPLES:
        assert wb(dims(x, b, u, y, d=3)) > 0                      # (d is not read)
        assert wb(dims(x, b, u, y, d=3, S=4096)) > wb(dims(x, b, u, y, d=3, S=4096), 32) > 0
    assert wb(dims(x=3, b=7, u=1, y=2, d=2)) == 0


# ------------------------------------------------------------------------------------------ the Python layer
@pytest.fixture
def host(monkeypatch, emul):
    monkeypatch.setattr(runtime, "_require_cuda", lambda *a, **k: None)
    monkeypatch.setattr(runtime, "_stream", lambda dev: 0)
    monkeypatch.setattr(runtime, "workspace", lambda dev, need: None)
    monkeypatch.setattr(abi, "load_library", lambda: emul)
    return emul


def _base_inputs(S=2, seed=3):
    act, Sig = random_actor(6, 2, 4, S, seed)
    return {k: v.requires_grad_(True) for k, v in act.items()}, Sig.requires_grad_(True)


def test_gradcheck_lqr_backward(host):
    T = 8
    m, _ = _base_inputs()

    def L_of(A, B, Q, R):
        return lqr.backward(time_stack_spec(A, B, m["F"].detach(), m["V"].detach(), m["W"].detach(), Q, R, T)).L
    assert torch.autograd.gradcheck(L_of, (m["A"], m["B"], m["Q"], m["R"]))


def test_gradcheck_kf_forward(host):
    T = 8
    m, Sig = _base_inputs()

    def K_of(A, F, V, W, Sigma0):
        return kf.forward(time_stack_spec(A, m["B"].detach(), F, V, W, m["Q"].detach(), m["R"].detach(), T), Sigma0)
    assert torch.autograd.gradcheck(K_of, (m["A"], m["F"], m["V"], m["W"], Sig))


def test_l_and_H_are_not_differentiable_and_no_grad_calls_stay_plain(host):
    m, _ = _base_inputs()
    sp = time_stack_spec(*(m[k] for k in abi.ACTOR_KEYS), 8)
    g = lqr.backward(sp)
    assert g.L.requires_grad and not g.l.requires_grad and not g.H.requires_grad
    with torch.no_grad():
        assert lqr.backward(sp).L.grad_fn is None and kf.forward(sp, None).grad_fn is None
    plain = time_stack_spec(*(m[k].detach() for k in abi.ACTOR_KEYS), 8)
    assert lqr.backward(plain).L.grad_fn is None and kf.forward(plain, None).grad_fn is None


def test_cross_cost_is_refused(host):
    m, _ = _base_inputs()
    sp = time_stack_spec(*(m[k] for k in abi.ACTOR_KEYS), 8)
    sp = sp._replace(P=torch.ones_like(sp.P))
    with pytest.raises(NotImplementedError):
        lqr.backward(sp)


def subjective_gains_loss(theta, T, wL, wK, oracle):
    """A loss on the gains of SubjectiveActor(dim=2) with parameters theta[S, 6]: lqg_b200 or the oracle."""
    kw = {n: theta[:, i] for i, n in enumerate(SUBJ)}
    if oracle:
        a, _ = OT.subjective_actor(dim=2, **kw)
        L = OT.lqr_backward(a["A"], a["B"], a["Q"], a["R"], T).transpose(0, 1)
        K = OT.kf_forward(a["A"], a["F"], a["V"], a["W"], a["V"] @ a["V"].mT, T).transpose(0, 1)
    else:
        m = tracking.SubjectiveActor(dim=2, T=T, **kw)
        L, K = lqr.backward(m.actor).L, kf.forward(m.actor, None)
    return (L * wL).sum() + (K * wK).sum() + (L ** 2).sum()


def theta_grads(S, T, seed=0, dev="cpu", rows=None, oracle=True):
    """d loss / d theta of subjective_gains_loss from lqg_b200 on `dev` (then from the oracle, with `oracle`), for the samples
    `rows` of S (all of them by default); on the host."""
    rng = np.random.default_rng(seed)
    th = np.array([1.0, 0.5, 1.0, 0.5, 9.0, 6.0])[None] * np.exp(0.2 * rng.standard_normal((S, 6)))
    wL, wK = rng.standard_normal((S, T, 2, 6)), rng.standard_normal((S, T, 6, 4))
    if rows is not None:
        th, wL, wK = th[rows], wL[rows], wK[rows]
    out = []
    for o in ((False, True) if oracle else (False,)):
        d = "cpu" if o else dev   # (the oracle's model matrices live on the host)
        t = torch.tensor(th, dtype=torch.float64, device=d, requires_grad=True)
        subjective_gains_loss(t, T, torch.tensor(wL, device=d), torch.tensor(wK, device=d), o).backward()
        out.append(t.grad.cpu())
    return out


def test_parameter_gradients_of_a_loss_on_the_gains(host):
    g, go = theta_grads(S=3, T=40)
    assert torch.allclose(g, go, rtol=1e-8, atol=1e-10 * go.abs().max().item()), (g - go).abs().max()
