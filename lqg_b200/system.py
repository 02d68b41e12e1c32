"""``System`` / ``Dynamics`` / ``Actor`` / ``LQG`` / ``NumpyroLQG`` -- drop-in for ``lqg/system.py``.

Hot path (CUDA): ``log_likelihood`` and ``conditional_distribution(x).log_prob(x[:, 1:])`` (lqg/system.py:237-248)
with the adjoint as autograd backward.  Slow paths (torch ops on the GPU around the CUDA gain kernels):
``conditional_moments`` (:142-235), ``belief_tracking_distribution`` (:250-257) and ``simulate`` (:62-140).
Arrays are torch tensors; a leading parameter-sample axis plays the role of ``jax.vmap``.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

from lqg_b200 import runtime
from lqg_b200.belief import kf
from lqg_b200.control import lqr
from lqg_b200.spec import LQGSpec
from lqg_b200.utils import time_stack_spec

mT = lambda M: M.transpose(-1, -2)


class MultivariateNormalSeq:
    """Minimal stand-in for ``numpyro.distributions.MultivariateNormal(mu, Sigma)[.to_event(1)]`` (numpyro is not
    available in this image): holds per-step moments and evaluates the log-density by Cholesky (system.py:244,257)."""

    def __init__(self, loc, covariance_matrix, event_dims=1):
        self.loc, self.covariance_matrix, self.event_dims = loc, covariance_matrix, event_dims

    def shape(self):
        return tuple(self.loc.shape)

    @property
    def batch_shape(self):
        return tuple(self.loc.shape[:-1 - (self.event_dims - 1)]) if self.event_dims > 1 else tuple(self.loc.shape[:-1])

    @property
    def event_shape(self):
        return tuple(self.loc.shape[-self.event_dims:])

    def log_prob(self, value):
        Lc = torch.linalg.cholesky(self.covariance_matrix)
        diff = (value - self.loc).unsqueeze(-1)
        z = torch.linalg.solve_triangular(Lc.expand(diff.shape[:-2] + Lc.shape[-2:]), diff, upper=False).squeeze(-1)
        d = value.shape[-1]
        lp = -0.5 * d * math.log(2 * math.pi) - torch.log(torch.diagonal(Lc, dim1=-2, dim2=-1)).sum(-1) - 0.5 * (z * z).sum(-1)
        for _ in range(self.event_dims - 1):
            lp = lp.sum(-1)
        return lp


class ConditionalDistribution:
    """p(x_{1:T} | x_0, theta) for the trials ``x`` it was built from (``System.conditional_distribution``).

    ``batch_shape = (n,)``, ``event_shape = (T, d)`` as in the reference (system.py:244 ``.to_event(1)``;
    tests/infer_test.py:16 checks ``.shape()[1] == T``).  ``log_prob(x[:, 1:])`` is the fused CUDA likelihood."""

    def __init__(self, system: "System", x: torch.Tensor, Sigma0=None):
        self.system, self.x, self.Sigma0 = system, x, Sigma0

    def shape(self):
        n, T1, d = self.x.shape
        return (n, T1 - 1, d)

    @property
    def batch_shape(self):
        return (self.x.shape[0],)

    @property
    def event_shape(self):
        return (self.x.shape[1] - 1, self.x.shape[2])

    def log_prob(self, value: torch.Tensor) -> torch.Tensor:
        if value.shape != self.x[:, 1:].shape:
            raise ValueError(f"expected observations of shape {tuple(self.x[:, 1:].shape)}")
        same = value.data_ptr() == self.x[:, 1:].data_ptr() or bool(torch.equal(value, self.x[:, 1:]))
        if same:
            return self.system.log_likelihood(self.x, Sigma0=self.Sigma0)
        # different values under the moments conditioned on self.x: slow path
        d = self.x.shape[-1]
        mu, Sigma = self.system._moments(self.x, self.Sigma0)
        return MultivariateNormalSeq(mu[..., :d], Sigma[..., :d, :d].unsqueeze(-4), event_dims=2).log_prob(value)


class System:
    def __init__(self, actor: LQGSpec, dynamics: LQGSpec):
        self.actor = actor
        self.dynamics = dynamics

    # -- dimensions (system.py:17-60)
    @property
    def T(self):
        return self.dynamics.A.shape[-3]

    @property
    def xdim(self):
        return self.dynamics.A.shape[-1]

    @property
    def ydim(self):
        return self.dynamics.F.shape[-2]

    @property
    def bdim(self):
        return self.actor.A.shape[-1]

    @property
    def udim(self):
        return self.dynamics.B.shape[-1]

    @property
    def device(self):
        return self.actor.A.device

    @property
    def dtype(self):
        return self.actor.A.dtype

    def to(self, *args, **kw) -> "System":
        mv = lambda s: LQGSpec(*[v.to(*args, **kw) if torch.is_tensor(v) else v for v in s])
        new = object.__new__(type(self))
        new.__dict__.update(self.__dict__)
        new.actor = mv(self.actor)
        new.dynamics = new.actor if self.dynamics is self.actor else mv(self.dynamics)
        axis = getattr(self, "_axis_system", None)
        if axis is not None:   # the factorised dim > 1 likelihood runs on this cached 1-axis model: move it too
            new._axis_system = axis.to(*args, **kw)
        return new

    def _default_sigma0(self, Sigma0):
        if Sigma0 is not None:
            return torch.as_tensor(Sigma0, dtype=self.dtype, device=self.device)
        V0 = self.actor.V[..., 0, :, :]
        return V0 @ mT(V0)

    def _gains(self, Sigma0=None):
        gains = lqr.backward(self.actor)
        K = kf.forward(self.actor, Sigma0=self._default_sigma0(Sigma0))
        return gains, K

    # -- hot path ------------------------------------------------------------------------------------------
    def log_likelihood(self, x: torch.Tensor, Sigma0=None) -> torch.Tensor:
        """log p(x_{i,1:T} | x_{i,0}) per trial, summed over time (system.py:246-248).  x: (n, T+1, d), or
        (S, n, T+1, d) to give every parameter sample (e.g. experimental condition) its own trials."""
        axis = getattr(self, "_axis_system", None)
        if axis is not None and Sigma0 is None and x.shape[-1] == self.xdim:
            # Exact factorisation (SURVEY 7.2, checked to 1e-15): a dim-axis tracking model with shared parameters is
            # block diagonal, so its likelihood is the sum over axes of the 1-axis model's likelihood on that axis'
            # (target, cursor) columns.  The per-sample recursions then run once on n/dim-sized matrices and the
            # axes become extra trials: x[n, T+1, dim*da] -> [dim*n, T+1, da].
            lead, (n, T1, d) = x.shape[:-3], x.shape[-3:]
            dim = self.dim
            xa = x.reshape(*lead, n, T1, dim, d // dim).movedim(-2, -4).reshape(*lead, dim * n, T1, d // dim)
            ll = axis.log_likelihood(xa)
            return ll.reshape(*ll.shape[:-1], dim, n).sum(-2)
        s0 = None if Sigma0 is None else torch.as_tensor(Sigma0, dtype=self.dtype, device=self.device)
        return runtime.log_likelihood(self.actor, self.dynamics, x.to(self.device), Sigma0=s0)

    def conditional_distribution(self, x: torch.Tensor, Sigma0=None) -> ConditionalDistribution:
        return ConditionalDistribution(self, x, Sigma0)

    def simulate_sdn(self, rng_key=0, n=1, signal_dep_noise=None, obs_dep_noise=None, C=None, D=None, gains=None, x0=None, xhat0=None,
                     Sigma0=None, return_all=False):
        """``simulate`` (system.py:62-140) under signal-dependent noise -- the generative model of ``log_likelihood_sdn``
        (EXTENSION, oracle/sdn_np.py: sdn_simulate): control-dependent process noise ``sum_i eps'_i C_i u_t`` and state-dependent
        observation noise ``sum_j eta'_j D_j x_{t+1}`` on top of V, W.  Arguments as in ``log_likelihood_sdn``; CUDA only."""
        C, D, L, l, K = self._sdn_inputs(signal_dep_noise, obs_dep_noise, C, D, gains, Sigma0)
        out = runtime.simulate(self.actor, self.dynamics, L, l, K, n, int(rng_key), x0=x0, xhat0=xhat0, return_all=return_all, C=C, D=D)
        if out is None:
            raise NotImplementedError("simulate_sdn: a dimension exceeds the simulator kernel's limit (40)")
        return out

    def log_likelihood_fp64(self, x: torch.Tensor, Sigma0=None) -> torch.Tensor:
        """``log_likelihood`` with the per-trial recursion in FP64 as well (the all-FP64 kernel k_sdn_loglik without
        multiplicative noise): for models whose innovation covariance is too ill-conditioned for the FP32 per-trial
        arithmetic of the main path, e.g. ``PointMassBoundedActor`` with all four states observed
        (lqg/tracking/point_mass.py:7-47).  Forward only; gradients: lqg_b200.control.sdn.value_and_grad_fd."""
        g, K = self._gains(Sigma0)
        return runtime.sdn_log_likelihood(self.actor, self.dynamics, x.to(self.device), g.L, K)

    def log_likelihood_sdn(self, x: torch.Tensor, signal_dep_noise=None, obs_dep_noise=None, C=None, D=None, gains=None,
                           Sigma0=None) -> torch.Tensor:
        """log p(x | theta) under signal-dependent noise -- an EXTENSION of the reference (docs/README.md:60-62 names it as
        future work; lqg/infer/prior.py:11 only reserves the parameter name ``signal_dep_noise``), see
        lqg_b200.control.sdn and oracle/sdn_np.py.  The plant gets control-dependent process noise and state-dependent
        observation noise on top of V, W; the experimenter's filter (system.py:142-248) matches the first two moments of
        every predictive distribution.  Noise model: either the scalars ``signal_dep_noise`` / ``obs_dep_noise`` (per-channel
        proportional noise, lqg_b200.control.sdn.channel_noise; parameters may be batched like the model's own) or explicit
        matrices ``C[(S,) nc, x, u]``, ``D[(S,) nd, y, x]``.  ``gains``: None = the actor model's own lqr.backward / kf.forward
        (an actor unaware of the multiplicative noise), ``"sdn"`` = the filter-form Todorov iterations on the actor's model with
        the same per-channel scales (lqg_b200.control.sdn.solve_for_actor), or an explicit pair (L, K)."""
        axis = getattr(self, "_axis_system", None)
        if axis is not None and C is None and D is None and (gains is None or gains == "sdn") and Sigma0 is None and x.shape[-1] == self.xdim:
            # per-channel noise keeps the axes of a dim > 1 tracking model independent: same factorisation as log_likelihood
            lead, (n, T1, d) = x.shape[:-3], x.shape[-3:]
            dim = self.dim
            xa = x.reshape(*lead, n, T1, dim, d // dim).movedim(-2, -4).reshape(*lead, dim * n, T1, d // dim)
            ll = axis.log_likelihood_sdn(xa, signal_dep_noise=signal_dep_noise, obs_dep_noise=obs_dep_noise, gains=gains)
            return ll.reshape(*ll.shape[:-1], dim, n).sum(-2)
        C, D, L, _, K = self._sdn_inputs(signal_dep_noise, obs_dep_noise, C, D, gains, Sigma0)
        return runtime.sdn_log_likelihood(self.actor, self.dynamics, x.to(self.device), L, K, C=C, D=D)

    def _sdn_inputs(self, signal_dep_noise, obs_dep_noise, C, D, gains, Sigma0):
        """(C, D, L, l, K) of simulate_sdn / log_likelihood_sdn: the noise matrices (from the per-channel scales unless given)
        and the gains named by ``gains``; l is the affine control term of the actor's own gains, None for the others."""
        from lqg_b200.control import sdn
        if C is None and signal_dep_noise is not None:
            C = sdn.channel_noise(self, signal_dep_noise, "control")
        if D is None and obs_dep_noise is not None:
            D = sdn.channel_noise(self, obs_dep_noise, "observation")
        if gains is None:
            g, K = self._gains(Sigma0)
            return C, D, g.L, g.l, K
        if not isinstance(gains, str):
            L, K = gains
            return C, D, L, None, K
        if gains != "sdn":
            raise ValueError("gains must be None, 'sdn' or a pair (L, K)")
        # the actor plans and filters knowing about the multiplicative noise: filter-form Todorov iterations on its own model
        sg = sdn.solve_for_actor(self, signal_dep_noise=signal_dep_noise, obs_dep_noise=obs_dep_noise, Sigma0=Sigma0)
        L, K = (sg.L, sg.K) if self.actor.A.dim() == 4 else (sg.L[0], sg.K[0])
        return C, D, L, None, K

    # -- slow paths ----------------------------------------------------------------------------------------
    def _joint(self, gains_L, K):
        """Joint (x, xhat) transition F[...,T,n,n] and noise factor G[...,T,n,x+y] (system.py:163-207)."""
        cast = lambda spec: LQGSpec(*[v.to(K.dtype) if torch.is_tensor(v) else v for v in spec])
        a, dn = cast(self.actor), cast(self.dynamics)
        top = torch.cat([dn.A.expand(K.shape[:-2] + dn.A.shape[-2:]), dn.B @ gains_L], -1)
        bot = torch.cat([K @ dn.F @ dn.A, a.A + a.B @ gains_L - K @ a.F @ a.A + K @ (dn.F @ dn.B - a.F @ a.B) @ gains_L], -1)
        Fj = torch.cat([top, bot], -2)
        zeros = torch.zeros(K.shape[:-2] + (self.xdim, self.ydim), dtype=K.dtype, device=K.device)
        Gj = torch.cat([torch.cat([dn.V.expand(K.shape[:-2] + dn.V.shape[-2:]), zeros], -1),
                        torch.cat([K @ dn.F @ dn.V, K @ dn.W], -1)], -2)
        return Fj, Gj

    def _moments(self, x: torch.Tensor, Sigma0=None):
        """mu[..., n_trials, T, n], Sigma[..., T, n, n]: predictive moments of (x, xhat)_{t+1} given x_{0..t}.
        CUDA kernels (lqgk_moments_*) for the compiled small systems, torch float64 otherwise."""
        if self.actor.A.is_cuda:
            s0 = None if Sigma0 is None else torch.as_tensor(Sigma0, dtype=self.dtype, device=self.device)
            out = runtime.moments(self.actor, self.dynamics, x.to(self.device), Sigma0=s0)
            if out is not None:
                return out
        return self._moments_torch(x, Sigma0)

    def _moments_torch(self, x: torch.Tensor, Sigma0=None):
        """Host-side slow path of _moments (dimension tuples without kernels; also the check of the kernels in tests)."""
        x = x.to(self.device, torch.float64)
        n, T1, d = x.shape
        gains, K = self._gains(Sigma0)
        Fj, Gj = self._joint(gains.L.double(), K.double())
        T = Fj.shape[-3]
        if T != T1 - 1:
            raise ValueError(f"need T+1 = {T + 1} observations per trial, got {T1}")
        batch = Fj.shape[:-3]
        nj = Fj.shape[-1]
        mu = torch.zeros(batch + (n, nj), dtype=torch.float64, device=self.device)
        mu[..., :d] = x[:, 0]
        Sig = Gj[..., 0, :, :] @ mT(Gj[..., 0, :, :])
        mus, Sigs = [], []
        for t in range(T):
            F, G = Fj[..., t, :, :], Gj[..., t, :, :]
            FS = F @ Sig
            Soo = Sig[..., :d, :d]
            w = torch.linalg.solve(Soo, mT(x[:, t] - mu[..., :d]))
            mu = mu @ mT(F) + mT(FS[..., :, :d] @ w)
            Sig = FS @ mT(F) + G @ mT(G) - FS[..., :, :d] @ torch.linalg.solve(Soo, (Sig @ mT(F))[..., :d, :])
            mus.append(mu)
            Sigs.append(Sig)
        return torch.stack(mus, -2), torch.stack(Sigs, -3)

    def conditional_moments(self, x: torch.Tensor, Sigma0=None):
        """One trial ``x[T+1, d]`` -> ``mu[T, n]``, ``Sigma[T, n, n]`` (system.py:142-235)."""
        mu, Sigma = self._moments(x.unsqueeze(0), Sigma0)
        return mu[..., 0, :, :].to(self.dtype), Sigma.to(self.dtype)

    def belief_tracking_distribution(self, x: torch.Tensor, Sigma0=None) -> MultivariateNormalSeq:
        """Moments of the belief xhat given the observed states (system.py:250-257)."""
        d = self.xdim
        mu, Sigma = self._moments(x, Sigma0)
        return MultivariateNormalSeq(mu[..., d:].to(self.dtype), Sigma[..., d:, d:].unsqueeze(-4).to(self.dtype))

    def simulate(self, rng_key=None, n=1, x0=None, xhat0=None, Sigma0=None, return_all=False):
        """Simulate n trials (system.py:62-140).  ``rng_key``: int seed or ``torch.Generator`` (the reference's JAX
        threefry stream cannot be reproduced; samples differ, the distribution does not).  Un-batched specs only."""
        dev, dt = self.device, self.dtype
        if self.actor.A.dim() != 3 and (dev.type != "cuda" or isinstance(rng_key, torch.Generator)):
            raise NotImplementedError("simulate() of a batched system needs the CUDA simulator (device 'cuda', integer seed)")
        if isinstance(rng_key, torch.Generator):
            gen = rng_key
        else:
            gen = torch.Generator(device=dev)
            gen.manual_seed(int(rng_key) if rng_key is not None else 0)
        gains, K = self._gains(Sigma0)
        if dev.type == "cuda" and not isinstance(rng_key, torch.Generator):
            # batched Philox simulator kernel (lqgk_simulate_*): one thread per trial
            out = runtime.simulate(self.actor, self.dynamics, gains.L, gains.l, K, n, int(rng_key) if rng_key is not None else 0,
                                   x0=x0, xhat0=xhat0, return_all=return_all)
            if out is not None:
                return out
        T, xd, bd, yd = self.T, self.xdim, self.bdim, self.ydim
        x = torch.zeros(n, xd, dtype=dt, device=dev) if x0 is None else torch.as_tensor(x0, dtype=dt, device=dev).expand(n, xd).clone()
        xh = torch.zeros(n, bd, dtype=dt, device=dev) if xhat0 is None else torch.as_tensor(xhat0, dtype=dt, device=dev).expand(n, bd).clone()
        eps = torch.randn(T, n, xd, dtype=dt, device=dev, generator=gen)
        eta = torch.randn(T, n, yd, dtype=dt, device=dev, generator=gen)
        a, dn = self.actor, self.dynamics
        xs, xhs, ys, us = [x], [xh], [], []
        for t in range(T):
            u = xh @ mT(gains.L[t]) + gains.l[t]
            x = x @ mT(dn.A[t]) + u @ mT(dn.B[t]) + eps[t] @ mT(dn.V[t])
            y = x @ mT(dn.F[t]) + eta[t] @ mT(dn.W[t])
            xp = xh @ mT(a.A[t]) + u @ mT(a.B[t])
            xh = xp + (y - xp @ mT(a.F[t])) @ mT(K[t])
            xs.append(x); xhs.append(xh); ys.append(y); us.append(u)
        X = torch.stack(xs, 1)
        if return_all:
            return X, torch.stack(xhs, 1), torch.stack(ys, 1), torch.stack(us, 1)
        return X

    def to_numpyro(self, Sigma0=None, xdim=None):
        return NumpyroLQG(self, Sigma0=Sigma0, xdim=xdim)


def _mat(M, ref=None):
    return torch.as_tensor(M) if not torch.is_tensor(M) else M


def Dynamics(A, B, F, V, W, T=1000) -> LQGSpec:
    """system.py:331-345."""
    A, B, F, V, W = map(_mat, (A, B, F, V, W))
    xdim, udim = A.shape[-1], B.shape[-1]
    kw = dict(dtype=A.dtype, device=A.device)
    return time_stack_spec(A=A, B=B, F=F, V=V, W=W, Q=torch.zeros(xdim, xdim, **kw), R=torch.zeros(udim, udim, **kw), T=T)


def Actor(A, B, F, V, W, Q, R, T=1000) -> LQGSpec:
    """system.py:348-349."""
    return time_stack_spec(*map(_mat, (A, B, F, V, W, Q, R)), T=T)


class LQG(System):
    """system.py:352-356."""

    def __init__(self, A, B, F, V, W, Q, R, T=1000):
        spec = time_stack_spec(*map(_mat, (A, B, F, V, W, Q, R)), T=T)
        super().__init__(actor=spec, dynamics=spec)


class NumpyroLQG:
    """Distribution adaptor with the reference's contract (system.py:358-376): ``event_shape = (T+1, xdim)``,
    ``batch_shape = ()``, ``log_prob(x[n,T+1,d]) -> [n]``, ``sample(key, sample_shape)``.  numpyro itself is not
    installable in this image, so this is a plain class with the same methods (see INTEGRATION.md for the
    numpyro/JAX binding)."""

    def __init__(self, system: System, xdim=None, Sigma0=None):
        self.system = system
        self.Sigma0 = Sigma0
        xdim = system.xdim if xdim is None else xdim
        self.event_shape = (system.T + 1, xdim)
        self.batch_shape = ()

    def log_prob(self, x):
        return self.system.log_likelihood(x, Sigma0=self.Sigma0)

    def sample(self, key, sample_shape=()):
        if len(sample_shape) == 0:
            return self.system.simulate(key, n=1, Sigma0=self.Sigma0)[0]
        return self.system.simulate(key, n=sample_shape[0], Sigma0=self.Sigma0)
