#!/usr/bin/env python
"""bench.py -- headline metric of BASELINE.json: trial log-lik+grad evals/sec on B200, with roofline fractions,
next to the reference algorithm on the host CPU.

Workload = config c3 of BASELINE.json exactly ("Batched likelihood sweep: 65,536 parameter samples x 100 trials x T=1200,
sharded over 1/2/4/8 B200"): SubjectiveActor 2-D tracking, N=100 trials x T=1200, a sweep of 65,536 parameter samples IN
TOTAL, sharded over the GPUs by parameter samples (STRONG scaling: every rank evaluates 65,536 / n_gpus samples).  One
"step" = one log-likelihood + parameter-gradient evaluation of all 65,536 samples (6,553,600 trial evals).  Data are
synthetic: the c3 legs (GPU and CPU) take them from the oracle's restatement of System.simulate (NumPy PCG64, seed 7), the
secondary GPU workloads from the product's own System.simulate (torch Philox); parameter samples are
theta_true * exp(0.25 z), z ~ N(0, I_6), seed 11.

  value : device-resident (base matrices + observations already in HBM) through the C ABI, CUDA events, max over ranks;
          every rank ends the step with the complete sweep result (all-gather of the per-sample [ll, base-matrix gradients]
          through lqg_b200.parallel -- the path's one collective).
  e2e   : through the public API (lqg_b200.tracking.SubjectiveActor(...).log_likelihood(x).sum().backward()) with
          theta and x in pinned HOST memory every step: H2D of this rank's theta slice + observations, model construction,
          fused forward+adjoint, all-gather of [ll, grad] over the ranks, D2H of ll[S] and grad[S,6].
  roofline : dominant kernel.  `frac` = FP32 operations the kernel EXECUTES (instruction counts of this very build from the
          committed ncu capture, profiles/r02_counters.json, keyed by a hash of the kernel sources) / its live CUDA-event time,
          against the FP32 FMA peak measured in this run (MEASURED_PEAKS.json has no FP32 figure).  `algorithmic_frac` keeps the
          SURVEY 8(d) dense-count convention.  `bound` = whichever of the step's HBM floor and FP32 floor is larger.
  cpu_baseline : the oracle's torch-float64 port of the reference algorithm (autodiff through the three scans),
          all host threads, on a bounded sample (64 samples x 100 trials x T=1200).
  secondary : BASELINE configs c2 (6 conditions x 20 trials, conditions sharded over the ranks + one all-reduce of
          [ll, grad]), c5 (one leapfrog of 4,096 lock-step chains, chains sharded over the ranks) at every N; c4 at N=1.

`--impl reference` runs only the CPU port (the real JAX reference is not installable in this image).
`--dump-outputs DIR` writes what the last timed step of the value and e2e legs computed as DIR/<name>.npy; the inputs of
those legs come from seeded NumPy generators only, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

PARAM_NAMES = ("action_cost", "action_variability", "subj_noise", "subj_vel_noise", "sigma_target", "sigma_cursor")
THETA_TRUE = (1.0, 0.5, 1.0, 0.5, 19.9, 6.0)
DIMS = dict(x=4, b=6, u=2, y=4, d=4)
COUNTERS = os.path.join(ROOT, "profiles", "r02_counters.json")


# ----------------------------------------------------------------------------------------------- flop model
def mm(m, k, n):
    return 2 * m * k * n


def sample_flops(x, b, u, y):
    lqr = (2 * mm(u, b, b) + mm(u, b, u) + mm(u, b, 1) + 10 * u ** 3 + (2 * u ** 3) // 3 + 2 * u * u * b + 2 * u * u
           + 2 * mm(b, b, b) + mm(b, u, u) + 3 * mm(b, u, b) + 4 * b * b + mm(b, b, 1) + 3 * mm(b, u, 1) + mm(u, u, 1) + 4 * b)
    kf = (3 * mm(b, b, b) + b * b + mm(y, b, b) + mm(y, b, y) + mm(y, y, y) + y * y + 2 * y ** 3 + mm(b, b, y) + mm(b, y, y)
          + mm(b, y, b) + b + mm(b, b, b))
    return lqr, kf


def algorithmic_flops(x, b, u, y, d, N, T):
    """Forward flops of one system evaluation, SURVEY 8(d) convention (dense algebra of the reference recursions).
    Returns (per-sample-per-step, per-trial-per-step, forward total).  fwd+grad = 3x forward by convention."""
    n, m = x + b, x + y
    lqr, kf = sample_flops(x, b, u, y)
    joint = (mm(x, u, b) + 2 * (mm(b, y, x) + mm(b, x, x)) + 2 * mm(b, u, b) + mm(b, y, b) + mm(b, b, b) + mm(y, x, u)
             + mm(y, b, u) + y * u + mm(b, y, u) + 3 * b * b + mm(b, y, y))
    cov = 2 * mm(n, n, n) + mm(n, m, n) + 2 * (d ** 3 // 3) + 2 * n * d * d + mm(n, d, n) + 2 * n * n + d
    trial = 2 * n * n + 2 * n * d + n + d * d + 4 * d
    per_sample = lqr + kf + joint + cov
    return per_sample, trial, T * (per_sample + N * trial)


NOT_ON_THE_PROFILED_PATH = ("lqgk_sdn.cuh", "lqgk_api.cu")   # signal-dependent-noise extension; entry-point validation / dispatch


def source_sha():
    """Hash of the sources that determine the code of the kernels of the fused log-likelihood + gradient call (kernels, step
    functions, launch sequence, dimension tuples): ties profiles/r02_counters.json (per-sample instruction and byte counts from
    an ncu capture) to the build being timed.  The signal-dependent-noise extension and the extern "C" dispatcher are not part
    of that path and do not enter the hash."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "lqg_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")) and f not in NOT_ON_THE_PROFILED_PATH:
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------------------------- helpers
def make_data(N, T, seed=7):
    """Synthetic tracking data for the c3 legs: float64 restatement of System.simulate (oracle), NumPy PCG64."""
    from oracle import lqg_np as O
    kw = dict(zip(PARAM_NAMES, THETA_TRUE))
    sa, sd = O.make_system(O.subjective_actor_mats(dim=2, **kw), T)
    return O.simulate(sa, sd, N, np.random.default_rng(seed)).astype(np.float32)


def make_data_gpu(N, T, dev, seed=7, **overrides):
    """Synthetic tracking data for the secondary GPU workloads from the product's own simulator (lqg_b200 System.simulate,
    torch Philox)."""
    from lqg_b200.tracking import SubjectiveActor
    kw = dict(zip(PARAM_NAMES, THETA_TRUE))
    kw.update(overrides)
    return SubjectiveActor(dim=2, T=T, device=dev, **kw).simulate(seed, n=N).to(torch.float32)


def make_theta(S, seed):
    rng = np.random.default_rng(seed)
    return (np.asarray(THETA_TRUE)[None] * np.exp(0.25 * rng.standard_normal((S, len(THETA_TRUE))))).astype(np.float32)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons of one GPU during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", float("inf"))
        inside = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.15]
        # nvidia-smi needs a few hundred ms per sample on an 8-GPU box: fall back to the samples nearest to the region
        use = inside if inside else [r for _, r in self.rows[-3:]]
        for r in use:
            f = [c.strip() for c in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_inside_timed_region": len(inside), "reasons": sorted(reasons)}


def cpu_port_eval(S, N, T, X, seed=3):
    """One fwd+grad evaluation of S samples with the oracle's torch-float64 port on all host threads.  Returns seconds."""
    from oracle import lqg_torch as OT
    torch.set_num_threads(os.cpu_count() or 1)
    th = torch.tensor(make_theta(S, seed), dtype=torch.float64, requires_grad=True)
    Xt = torch.tensor(X, dtype=torch.float64)
    t0 = time.perf_counter()
    a, d = OT.subjective_actor(dim=2, **{n: th[:, i] for i, n in enumerate(PARAM_NAMES)})
    ll = OT.log_likelihood(a, d, Xt)
    ll.sum().backward()
    assert torch.isfinite(th.grad).all()
    return time.perf_counter() - t0


DUMP_MAX_BYTES = 16 << 20      # per array of --dump-outputs (three arrays: at most 48 MiB in all)


def dump(out_dir, **arrays):
    """--dump-outputs: every tensor as out_dir/<name>.npy in its own dtype (float32 / float64).  An array larger than
    DUMP_MAX_BYTES keeps a fixed, seeded sample of its rows (NumPy default_rng(0), in row order), so that runs with the same
    arguments write the same elements and two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        keep = max(1, DUMP_MAX_BYTES // (t[0].numel() * t.element_size()))
        if t.shape[0] > keep:
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        a = t.detach().cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def timed(fn, reps, warm, barrier):
    """ms per call of fn: CUDA events on the current stream, bracketed by barriers (the caller takes the max over ranks)."""
    for _ in range(warm):
        out = fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / reps, out


# ----------------------------------------------------------------------------------------------- secondary workloads
def bench_c2(dev, barrier, reps=10):
    """Config c2 of BASELINE.json (latency case): SubjectiveActor 2-D, 6 blob-width conditions x 20 trials x T=1200, gradient
    w.r.t. 5 shared + 6 per-condition parameters.  The conditions are the kernels' sample axis (every condition its own
    trials); with several GPUs the conditions are sharded over the ranks and ONE all-reduce sums [ll, grad] (the collective the
    north star names; lqg_b200.parallel.trial_sharded_value_and_grad).  Returns ms per evaluation."""
    from lqg_b200 import parallel
    from lqg_b200.tracking import SubjectiveActor
    sig = [8.5, 9.7, 11.8, 19.9, 28.5, 51.6]
    T, N = 1200, 20
    x = torch.stack([make_data_gpu(N, T, dev, seed=c, sigma_target=s_t, action_cost=1.0, sigma_cursor=6.0) for c, s_t in enumerate(sig)])
    cond = torch.arange(len(sig), device=dev)

    def local(idx):   # idx: this rank's conditions -> (sum ll, grad[5 + 6])
        shared = torch.tensor([1.0, 0.5, 1.0, 0.5, 6.0], device=dev, requires_grad=True)   # cost, variab., subj, subj_vel, sigma_cursor
        st = torch.tensor(sig, device=dev, requires_grad=True)
        if idx.numel() == 0:
            return torch.zeros((), device=dev), torch.zeros(5 + len(sig), device=dev)
        m = SubjectiveActor(dim=2, T=T, device=dev, action_cost=shared[0], action_variability=shared[1], subj_noise=shared[2],
                            subj_vel_noise=shared[3], sigma_cursor=shared[4], sigma_target=st[idx])
        ll = m.log_likelihood(x[idx]).sum()
        ll.backward()
        return ll.detach(), torch.cat([shared.grad, st.grad])

    ms, (ll, g) = timed(lambda: parallel.trial_sharded_value_and_grad(local, cond), reps, 3, barrier)
    assert torch.isfinite(ll) and torch.isfinite(g).all()
    # the same evaluation replayed from a CUDA graph (lqg_b200.graphs): the local part is captured, the all-reduce stays outside
    from lqg_b200.graphs import GraphedValueAndGrad
    lo, hi = parallel.shard_range(len(sig), *parallel.world())
    # EVERY rank runs the same sequence of collectives below, also the ranks that own no condition (more GPUs than conditions:
    # 8 ranks, 6 conditions) -- they contribute zeros.  (A rank-dependent number of all-reduces deadlocks NCCL.)
    gv, idx = None, cond[lo:hi]
    th = torch.tensor([1.0, 0.5, 1.0, 0.5, 6.0] + sig, device=dev)
    if hi > lo:
        def fn(theta):   # theta = [5 shared | 6 sigma_target]
            m = SubjectiveActor(dim=2, T=T, device=dev, action_cost=theta[0], action_variability=theta[1], subj_noise=theta[2],
                                subj_vel_noise=theta[3], sigma_cursor=theta[4], sigma_target=theta[5:][idx])
            return m.log_likelihood(x[idx])

        gv = GraphedValueAndGrad(fn, th)

    def graphed():
        if gv is not None:
            out, grad = gv(th)
            packed = torch.cat([out.sum().reshape(1), grad])
        else:
            packed = torch.zeros(1 + th.numel(), device=dev)
        return parallel.allreduce_sum(packed)

    ms_graph, packed = timed(graphed, reps, 3, barrier)
    assert torch.allclose(packed[0], ll, rtol=1e-5) and torch.allclose(packed[1:], g, rtol=1e-3, atol=1e-4 * g.abs().max().item())
    return ms, ms_graph


def bench_c2_sdn(dev, reps=5):
    """Config c2 as BASELINE.json words it ("... with signal-dependent noise"): the c2 model with per-channel control- and
    state-dependent noise (System.log_likelihood_sdn; an EXTENSION -- the reference has no signal-dependent noise, parity is
    unpinned, DESIGN.md).  The covariance pass is per (condition x trial) here, FP64, one thread per system; the gradient
    w.r.t. 5 shared + 6 per-condition + 2 noise parameters is a batched central difference (27 parameter vectors x 6 conditions
    in one launch set).  Rank 0 only (no sharding: 240 systems).  Returns ms per value+gradient evaluation and per value."""
    from lqg_b200.control import sdn
    from lqg_b200.tracking import SubjectiveActor
    sig = [8.5, 9.7, 11.8, 19.9, 28.5, 51.6]
    T, N = 1200, 20
    x = torch.stack([make_data_gpu(N, T, dev, seed=c, sigma_target=s_t, action_cost=1.0, sigma_cursor=6.0) for c, s_t in enumerate(sig)])
    nc = len(sig)

    def total(Th):   # Th[P', 13] = [5 shared | 6 sigma_target | signal_dep_noise, obs_dep_noise] -> summed ll per parameter vector
        Pn = Th.shape[0]
        rep = lambda v: v.repeat_interleave(nc)                           # (parameter vector, condition) pairs as the sample axis
        m = SubjectiveActor(dim=2, T=T, device=dev, dtype=torch.float64, action_cost=rep(Th[:, 0]), action_variability=rep(Th[:, 1]),
                            subj_noise=rep(Th[:, 2]), subj_vel_noise=rep(Th[:, 3]), sigma_cursor=rep(Th[:, 4]),
                            sigma_target=Th[:, 5:5 + nc].reshape(-1))
        ll = m.log_likelihood_sdn(x.repeat(Pn, 1, 1, 1), signal_dep_noise=rep(Th[:, 11]), obs_dep_noise=rep(Th[:, 12]))
        return ll.reshape(Pn, nc, N).sum((1, 2))

    th = torch.tensor([1.0, 0.5, 1.0, 0.5, 6.0] + sig + [20.0, 0.2], device=dev, dtype=torch.float64)
    ms_grad, (v, g) = timed(lambda: sdn.value_and_grad_fd(total, th), reps, 2, lambda: torch.cuda.synchronize())
    ms_val, v1 = timed(lambda: total(th[None]), reps, 2, lambda: torch.cuda.synchronize())
    assert torch.isfinite(v) and torch.isfinite(g).all() and torch.allclose(v1[0], v)
    return ms_grad, ms_val


def bench_c5(dev, barrier, chains=4096, N=100, T=1200, reps=5):
    """Config c5 of BASELINE.json without numpyro (not installable): the work of ONE leapfrog step of 4,096 lock-step chains =
    one fused log-likelihood + gradient evaluation of 4,096 parameter vectors on the c3 data, chains sharded over the ranks
    (every rank owns its chains: no collective per leapfrog, SURVEY 8e).  Returns ms per evaluation."""
    from lqg_b200 import parallel
    from lqg_b200.tracking import SubjectiveActor
    x = make_data_gpu(N, T, dev)
    theta = torch.tensor(make_theta(chains, 23), device=dev)

    def local(th):
        th = th.detach().requires_grad_()
        m = SubjectiveActor(dim=2, T=T, device=dev, **{n: th[:, i] for i, n in enumerate(PARAM_NAMES)})
        ll = m.log_likelihood(x).sum(-1)
        ll.sum().backward()
        return ll.detach(), th.grad

    ms, (ll, g) = timed(lambda: parallel.sharded_value_and_grad(local, theta, gather=False), reps, 2, barrier)
    assert torch.isfinite(ll).all() and torch.isfinite(g).all()
    # the same evaluation replayed from a CUDA graph (what jax.jit of the potential energy is in the reference's numpyro loop)
    from lqg_b200.graphs import GraphedValueAndGrad
    lo, hi = parallel.shard_range(chains, *parallel.world())

    def fn(th):
        m = SubjectiveActor(dim=2, T=T, device=dev, **{n: th[:, i] for i, n in enumerate(PARAM_NAMES)})
        return m.log_likelihood(x).sum(-1)

    gv = GraphedValueAndGrad(fn, theta[lo:hi])
    ms_graph, (ll2, g2) = timed(lambda: gv(theta[lo:hi]), reps, 2, barrier)
    assert torch.allclose(ll2, ll, rtol=1e-5) and torch.allclose(g2, g, rtol=1e-3, atol=1e-4 * g.abs().max().item())
    return ms, ms_graph


def bench_c4(dev, S=4096, N=50, T=600, reps=2):
    """Config c4 of BASELINE.json: TemporalDelayModel(PointMassBoundedActor(T=600), delay=2) -- 12-dim state, joint dim 24
    (large-system kernels, lqgk_big.cuh) --, 4,096 parameter samples x 50 trials, log-likelihood + gradient w.r.t. 4
    parameters per sample through the public API.  Returns (trial-evals/s, ms per evaluation, per-kernel ms)."""
    from lqg_b200.tracking import PointMassBoundedActor
    from lqg_b200.tracking.delay import TemporalDelayModel
    base = dict(action_variability=1e-3, sigma_target=6.0, sigma_cursor=6.0, action_cost=0.01)
    x = TemporalDelayModel(PointMassBoundedActor(T=T, device=dev, **base), 2).simulate(13, n=N)[..., :2].to(torch.float32)
    rng = np.random.default_rng(17)
    th = {k: torch.tensor(v * np.exp(0.25 * rng.standard_normal(S)), dtype=torch.float32, device=dev, requires_grad=True)
          for k, v in base.items()}

    def evaluate():
        for t in th.values():
            t.grad = None
        ll = TemporalDelayModel(PointMassBoundedActor(T=T, device=dev, **th), 2).log_likelihood(x).sum()
        ll.backward()
        return ll

    from lqg_b200 import abi
    lib = abi.load_library()
    evaluate()
    torch.cuda.synchronize()
    lib.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ll = evaluate()
    e1.record()
    torch.cuda.synchronize()
    prof = lib.profile_read()
    lib.profile_enable(False)
    ms = e0.elapsed_time(e1) / reps
    assert torch.isfinite(ll) and all(torch.isfinite(t.grad).all() for t in th.values())
    # the same evaluation replayed from a CUDA graph (model construction by ~100 small torch kernels on [S, 12, 12] matrices and
    # its backward are a fifth of the eager time)
    ms_graph = None
    try:
        from lqg_b200.graphs import GraphedValueAndGrad
        names = list(base)
        th0 = torch.stack([th[k].detach() for k in names], 1)

        def fn(tt):
            return TemporalDelayModel(PointMassBoundedActor(T=T, device=dev, **{k: tt[:, i] for i, k in enumerate(names)}), 2).log_likelihood(x)

        gv = GraphedValueAndGrad(fn, th0)
        ms_graph, (ll_g, g_g) = timed(lambda: gv(th0), reps, 1, lambda: torch.cuda.synchronize())
        assert torch.allclose(ll_g.sum(), ll.detach(), rtol=1e-4)
    except Exception as e:   # the graph is an optimisation of the measurement, never a requirement
        print("bench_c4: CUDA-graph replay unavailable:", repr(e), file=sys.stderr)
    return S * N / ((ms_graph or ms) * 1e-3), ms, {k: round(v[0] / reps, 2) for k, v in prof.items() if v[1]}, ms_graph


# ----------------------------------------------------------------------------------------------- reference arm
def workload_config(args, world, note=None):
    cfg = {"workload": "c3: batched likelihood sweep, 65,536 parameter samples x 100 trials x T=1200 (SubjectiveActor dim=2: x=4,b=6,u=2,"
                       "y=4,d=4), log-lik + gradient, sharded over the GPUs by parameter samples",
           "samples_total": args.samples, "samples_per_gpu": args.samples // world, "trials": args.trials, "T": args.T,
           "params": len(PARAM_NAMES),
           "sharding": "parameter samples across GPUs (no data-path collective); one all-gather of the per-sample [ll, gradients] "
                       "(lqg_b200.parallel) so every rank holds the whole sweep",
           "cache": "per-step workspace traffic (tens of GB) >> 126 MB L2; no explicit flush needed"}
    if note:
        cfg["note"] = note
    return cfg


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, T, S = args.trials, args.T, args.cpu_samples
    X = make_data(N, T)
    times = []
    for i in range(args.warmup + args.steps):
        dt = cpu_port_eval(S, N, T, X, seed=3 + i)
        if i >= args.warmup:
            times.append(dt)
    sec = float(np.mean(times))
    val = S * N / sec
    cores = os.cpu_count() or 1
    line = {"impl": "reference", "metric": "trial log-lik+grad evals/sec", "value": val, "unit": "trial-evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, max(1, args.gpus),
                                      note=f"CPU port of the reference algorithm (oracle/lqg_torch.py) on a bounded sample of the workload: "
                                           f"{S} of the {args.samples} parameter samples per step; the JAX reference is not installable in this image"),
            "cpu_baseline": {"value": val, "unit": "trial-evals/s", "cores": cores, "kind": "port",
                             "sample": f"{S} parameter samples x {N} trials x T={T}, fwd+grad by torch autograd, float64"},
            "e2e": {"value": val, "unit": "trial-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch.distributed as dist

    from lqg_b200 import abi, parallel, runtime
    from lqg_b200.tracking import SubjectiveActor

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # a collective mismatch must fail within minutes, not after NCCL's default 10-minute watchdog
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    lib = abi.load_library()
    if args.streams > 0:
        lib.set_streams(args.streams)
    if args.overlap >= 0:
        lib.set_kernel_overlap(args.overlap)
    if args.contrib_warps > 0:
        lib.lib.lqgk_set_contrib_warps(args.contrib_warps)
    if args.pipe_max >= 0:
        lib.set_pipeline(args.pipe_max, args.pipe_segments)
    S_total, N, T = args.samples, args.trials, args.T
    lo, hi = parallel.shard_range(S_total, rank, world)
    S = hi - lo                                        # this rank's samples (strong scaling)
    theta_all = make_theta(S_total, 11)
    theta_np = theta_all[lo:hi]
    P = theta_np.shape[1]

    # ---------------- device-resident leg (C ABI)
    theta = torch.tensor(theta_np, device=dev)
    model = SubjectiveActor(dim=2, T=T, device=dev, **{n: theta[:, i] for i, n in enumerate(PARAM_NAMES)})
    X = make_data(N, T)                               # seeded NumPy, so the inputs do not depend on the build being timed
    x_dev = torch.tensor(X, device=dev)
    if args.no_factorize:
        sysm, xk, Nk = model, x_dev, N
        dims = abi.LqgkDims(S, N, T, DIMS["x"], DIMS["b"], DIMS["u"], DIMS["y"], DIMS["d"])
    else:
        # what SubjectiveActor(dim=2).log_likelihood does: identical independent axes -> the 1-axis system with the
        # two axes of every trial as separate trials (exact; lqg_b200/system.py)
        sysm = model._axis_system
        xk = x_dev.reshape(N, T + 1, 2, 2).permute(2, 0, 1, 3).reshape(2 * N, T + 1, 2)
        Nk = 2 * N
        dims = abi.LqgkDims(S, Nk, T, 2, 3, 1, 2, 2)
    x_tm = lib.pack_obs(xk.contiguous(), stream=torch.cuda.current_stream().cuda_stream)
    act = {k: runtime._row_major(getattr(sysm.actor, k)[:, 0]) for k in abi.ACTOR_KEYS}
    dyn = {k: runtime._row_major(getattr(sysm.dynamics, k)[:, 0]) for k in abi.DYN_KEYS}
    ws_bytes_one_chunk = lib.workspace_bytes(dims, abi.MODE_VJP, args.chunk)
    ws = runtime.workspace(dev, ws_bytes_one_chunk)

    def step_resident():
        st = torch.cuda.current_stream().cuda_stream
        ll, ga, gd, _ = lib.loglik_vjp(dims, act, dyn, x_tm, ws=ws, stream=st)
        # the sweep result of this rank: per sample [sum_i ll_i, all base-matrix gradients]; gathered so that every rank holds
        # the complete sweep (the path's one collective, lqg_b200.parallel)
        packed = torch.cat([ll.sum(1, keepdim=True)] + [g.reshape(S, -1) for g in list(ga.values()) + list(gd.values())], 1)
        return parallel.gather_samples(packed, S_total), ll

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()                                   # started before the warm-up so samples exist when the timed region begins
    for _ in range(args.warmup):
        res, ll_trials = step_resident()
    barrier()
    launches_per_step = lib.last_launch_count()
    lib.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_start()
    e0.record()
    for _ in range(args.steps):
        res, ll_trials = step_resident()
    e1.record()
    barrier()
    sampler.mark_end()
    ms = e0.elapsed_time(e1)
    prof = lib.profile_read()
    lib.profile_enable(False)
    clocks = sampler.stop()
    if args.dump_outputs:
        # sweep[S_total, 1 + G]: per parameter sample [sum_i ll_i, the actor's (A B F V W Q R) and the dynamics' (A B F V W)
        # base-matrix gradients, each row-major] -- what every rank holds after the step.  ll[S_total, N]: per-trial
        # log-likelihoods in the public API's layout (the axes the factorised kernels see as separate trials summed back into
        # one trial, as SubjectiveActor.log_likelihood does), gathered from all ranks.
        ll = parallel.gather_samples(ll_trials.reshape(S, -1, N).sum(1), S_total)
        if rank == 0:
            dump(args.dump_outputs, sweep=res, ll=ll)
        del ll
    del ll_trials
    # The pipelined launch sequence overlaps kernels of different streams, so the per-kernel event times above include the
    # time a kernel shares the SMs with others.  Two extra steps (outside the timed region) with the plain sequence give
    # every kernel's time when it runs alone -- reported next to the live numbers.
    lib.set_pipeline(0, args.pipe_segments)
    step_resident()
    lib.profile_enable(True)
    for _ in range(2):
        step_resident()
    torch.cuda.synchronize()
    prof_alone = {k: (v[0] / 2, v[1] / 2) for k, v in lib.profile_read().items()}
    lib.profile_enable(False)
    lib.set_pipeline(args.pipe_max if args.pipe_max >= 0 else (1 << 30), args.pipe_segments)
    assert res.shape[0] == S_total and torch.isfinite(res).all(), "non-finite sweep result in the timed region"
    del res
    t_ms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    ms_per_step = ms / args.steps
    value = S_total * N / (ms_per_step * 1e-3)

    # ---------------- end-to-end leg through the public API, host buffers
    theta_host = torch.tensor(theta_np).pin_memory()
    x_host = torch.tensor(X).pin_memory()
    out_host = torch.empty((S_total, 1 + P), dtype=torch.float32).pin_memory()

    def step_e2e():
        th = theta_host.to(dev, non_blocking=True).requires_grad_()
        xd = x_host.to(dev, non_blocking=True)
        m = SubjectiveActor(dim=2, T=T, device=dev, **{n: th[:, i] for i, n in enumerate(PARAM_NAMES)})
        lls = m.log_likelihood(xd).sum(-1)
        lls.sum().backward()
        full = parallel.gather_samples(torch.cat([lls.detach()[:, None], th.grad], 1), S_total)   # [S_total, 1 + P] on every rank
        out_host.copy_(full, non_blocking=True)
        return full

    for _ in range(max(1, min(args.warmup, 2))):
        step_e2e()
    barrier()
    e0.record()
    for _ in range(args.steps):
        full = step_e2e()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump(args.dump_outputs, e2e_ll_grad=full)                  # [S_total, 1 + 6]: sum_i ll_i, d/dtheta (PARAM_NAMES order)
    t_e = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_ms = float(t_e.item()) / args.steps
    e2e_val = S_total * N / (e2e_ms * 1e-3)
    assert np.isfinite(out_host.numpy()).all()

    # ---------------- secondary workloads (every rank takes part: they shard over the ranks)
    secondary = []
    if not args.no_secondary:
        # a failing secondary workload must not take the primary line down with it (deterministic failures hit every rank at
        # the same point, so the ranks stay in step; anything else ends in the 180 s NCCL watchdog)
        def guarded(fn, *a):
            try:
                return fn(*a)
            except Exception as e:
                print(f"bench: secondary workload {fn.__name__} failed: {e!r}", file=sys.stderr)
                return float("nan"), float("nan")

        c2_ms, c2_g = guarded(bench_c2, dev, barrier)
        c5_ms, c5_g = guarded(bench_c5, dev, barrier)
        t2 = torch.tensor([c2_ms, c5_ms, c2_g or 0.0, c5_g or 0.0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        c2_ms, c5_ms, c2_g, c5_g = [float(v) for v in t2.tolist()]
        secondary.append({"workload": "c2: SubjectiveActor dim=2, 6 conditions x 20 trials x T=1200, grad wrt 5 shared + 6 per-condition "
                                      "parameters, public API; conditions sharded over the GPUs + one all-reduce of [ll, grad] (latency-bound)",
                          "value": 6 * 20 / (c2_g * 1e-3), "unit": "trial-evals/s", "ms_per_eval": c2_g, "ms_per_eval_eager": c2_ms,
                          "note": "ms_per_eval = the evaluation replayed from a CUDA graph (lqg_b200.graphs); eager = launched op by op"})
        secondary.append({"workload": "c5: one leapfrog of 4,096 lock-step chains = one fused log-lik+gradient of 4,096 parameter vectors x 100 "
                                      "trials x T=1200, chains sharded over the GPUs, public API (numpyro/NUTS itself is not installable here)",
                          "value": 1e3 / c5_g, "unit": "leapfrog-equivalents/s", "ms_per_eval": c5_g, "ms_per_eval_eager": c5_ms,
                          "chains_per_gpu": 4096 // world,
                          "note": "ms_per_eval = the evaluation replayed from a CUDA graph (lqg_b200.graphs); eager = launched op by op"})

        if rank == 0:
            sdn_grad_ms, sdn_val_ms = guarded(bench_c2_sdn, dev)
            secondary.append({"workload": "c2 with signal-dependent noise (EXTENSION, parity unpinned by the reference): SubjectiveActor dim=2 "
                                          "+ per-channel control-/state-dependent noise, 6 conditions x 20 trials x T=1200, per-trial FP64 "
                                          "covariance pass (k_sdn_loglik), value + central-difference gradient w.r.t. 13 parameters "
                                          "(27 x 6 systems batched), public API, one GPU",
                              "value": 6 * 20 / (sdn_grad_ms * 1e-3), "unit": "trial-evals/s", "ms_per_eval": sdn_grad_ms,
                              "ms_per_value_only": sdn_val_ms})
        if world > 1:
            dist.barrier()

    if rank == 0:
        # ---------------- roofline of the dominant kernel + whole step
        per_sample, per_trial, fwd = algorithmic_flops(DIMS["x"], DIMS["b"], DIMS["u"], DIMS["y"], DIMS["d"], N, T)
        step_flops = 3.0 * fwd * S_total                           # fwd+grad = 3x forward (SURVEY 8d convention)
        lqr_f, kf_f = [T * v for v in sample_flops(DIMS["x"], DIMS["b"], DIMS["u"], DIMS["y"])]
        cov_f = T * per_sample - lqr_f - kf_f
        kind_flops = {"lqr_fwd": lqr_f, "kf_fwd": kf_f, "cov_fwd": cov_f, "trial_fwd": T * N * per_trial,
                      "lqr_rev": 2 * lqr_f, "kf_rev": 2 * kf_f, "cov_rev": 2 * cov_f, "trial_rev": 2 * T * N * per_trial}
        fp32_peak = lib.peak_fma(False, dev)
        fp64_peak = lib.peak_fma(True, dev)
        groups = {"lqr_fwd": ["lqr_fwd"], "kf_fwd": ["kf_fwd"], "cov_fwd": ["cov_fwd"], "trial_fwd": ["trial_fwd"],
                  "trial_rev": ["trial_rev"], "cov_rev": ["cov_rev", "cov_contrib", "reduce"], "kf_rev": ["kf_rev"],
                  "lqr_rev": ["lqr_rev"], "boundary": ["pack", "unpack", "misc"]}
        kernels = {}
        for g, members in groups.items():
            g_ms = sum(prof[m][0] for m in members if m in prof) / args.steps
            g_cnt = sum(prof[m][1] for m in members if m in prof) / args.steps
            if g_cnt == 0:
                continue
            entry = {"ms_per_step": g_ms, "ms_per_step_alone": sum(prof_alone[m][0] for m in members if m in prof_alone),
                     "launches_per_step": g_cnt, "share": g_ms / ms_per_step,
                     "kernels": {"k_" + m: prof[m][0] / args.steps for m in members if m in prof and prof[m][1] > 0}}
            if g in kind_flops:
                entry["algorithmic_tflops"] = kind_flops[g] * S / (g_ms * 1e-3) / 1e12
            kernels[g] = entry
        dom = max((k for k in kernels if k in kind_flops), key=lambda k: kernels[k]["ms_per_step"])
        dom_kernel = max(kernels[dom]["kernels"], key=lambda k: kernels[dom]["kernels"][k])
        dom_ms = kernels[dom]["kernels"][dom_kernel]                  # live CUDA-event time of that kernel per step
        # launches of that kernel per step: sample chunks x time segments of the pipelined sequence.  Flops / bytes per launch =
        # per-step total / launches, so achieved (per launch / launch duration) = per-step total / per-step kernel time
        dom_launches = max(1.0, float(prof[dom_kernel[2:]][1]) / args.steps)
        launch_ms = dom_ms / dom_launches
        samples_per_launch = S                                         # every launch covers all samples of the chunk (one time segment)
        dom_ms_alone = prof_alone[dom_kernel[2:]][0]
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        # instruction counts / DRAM bytes of THIS build from the committed ncu capture (tools/ncu_counters.py)
        counters, counters_note, cj = None, None, None
        if os.path.exists(COUNTERS):
            cj = json.load(open(COUNTERS))
            same_shape = cj.get("trials") == dims.N and cj.get("T") == T and cj.get("kernel_dims") == [dims.x, dims.b, dims.u, dims.y, dims.d]
            if cj.get("source_sha") != source_sha():
                counters_note = (f"profiles/r02_counters.json is from another build ({cj.get('source_sha')} != {source_sha()}): "
                                 "executed-flop fraction and traffic not reported")
            elif not same_shape:
                counters_note = "profiles/r02_counters.json was captured on another launch shape: executed-flop fraction and traffic not reported"
            else:
                counters = cj
        else:
            counters_note = "profiles/r02_counters.json missing: executed-flop fraction and traffic not reported"
        ck = counters["kernels"].get(dom_kernel) if counters else None
        executed = traffic = None
        if ck:
            # per sample of one launch; the capture used fewer samples per launch than this run (ncu replays every kernel ~40x):
            # both quantities are per-sample constants of the kernel (no cross-sample reuse), so they scale with the samples
            flops = ck["fp32_flops_per_sample"] * S / dom_launches
            executed = {"tflops": flops / (launch_ms * 1e-3) / 1e12, "frac": flops / (launch_ms * 1e-3) / 1e12 / fp32_peak,
                        "frac_when_running_alone": ck["fp32_flops_per_sample"] * S / (dom_ms_alone * 1e-3) / 1e12 / fp32_peak,
                        "ms_per_step_live_overlapped": dom_ms, "ms_per_step_alone": dom_ms_alone,
                        "fp32_flops_per_launch": flops, "warp_instructions_per_sample_step": ck["inst_per_sample_step"],
                        "fp32_share_of_instructions": ck["fp32_inst_share"],
                        "ncu_fma_pipe_cycles_active_pct": ck["fma_pipe_cycles_active_pct"], "ncu_issue_active_pct": ck["issue_active_pct"],
                        "source": f"profiles/r02_counters.json (ncu --set full of this build, {cj['samples_per_launch']} samples per launch, scaled per sample)"}
            traffic = ck["dram_bytes_per_sample"] * S / dom_launches
        achieved_alg = kernels[dom]["algorithmic_tflops"]
        # floors of the whole step (this rank's share)
        step_exec_flops = step_bytes = fp32_floor = fp64_floor = hbm_floor = None
        bound = "fp32"
        if counters:
            step_exec_flops = sum(v["fp32_flops_per_sample"] * S for v in counters["kernels"].values())
            step_fp64_flops = sum(v.get("fp64_flops_per_sample", 0.0) * S for v in counters["kernels"].values())
            step_bytes = sum(v["dram_bytes_per_sample"] * S for v in counters["kernels"].values())
            fp32_floor = step_exec_flops / (fp32_peak * 1e12) * 1e3
            fp64_floor = step_fp64_flops / (fp64_peak * 1e12) * 1e3
            hbm_floor = step_bytes / (hbm_peak * 1e9) * 1e3
            bound = "hbm" if hbm_floor > fp32_floor + fp64_floor else "fp32"
        if bound == "hbm" and traffic:
            r_ach, r_peak, r_unit = traffic / (launch_ms * 1e-3) / 1e9, hbm_peak, "GB/s"
        elif executed:
            r_ach, r_peak, r_unit = executed["tflops"], fp32_peak, "TFLOP/s"
        else:
            r_ach, r_peak, r_unit = None, fp32_peak, "TFLOP/s"
        roofline = {"bound": bound, "kernel": dom_kernel, "achieved": r_ach, "peak": r_peak, "unit": r_unit,
                    "frac": (r_ach / r_peak) if r_ach is not None else None, "traffic": traffic,
                    "launch_ms": launch_ms, "launches_per_step": dom_launches, "samples_per_launch": samples_per_launch,
                    "time_steps_per_launch": T / dom_launches,
                    "peak_source": "FFMA micro-kernel measured in this run (lqgk_peak_fma); MEASURED_PEAKS.json has no FP32 figure; nominal 74.5",
                    "note": "achieved = FP32 operations the kernel executes (FFMA2 = 2 FMAs per lane, all 32 lanes counted; counts from the ncu "
                            "capture of this build) / live CUDA-event time.  algorithmic_* = SURVEY 8(d) dense count of the reference recursion the "
                            "kernel replaces (adjoint = 2x forward), which the reduced form + per-axis factorisation undercut -- an algorithmic "
                            "saving, not pipe utilisation",
                    "executed": executed, "counters_note": counters_note,
                    "algorithmic_achieved_tflops": achieved_alg, "algorithmic_frac": achieved_alg / fp32_peak,
                    "algorithmic_flops_per_launch": kind_flops[dom] * S / dom_launches,
                    "fp64_peak_tflops_measured": fp64_peak,
                    "step": {"ms": ms_per_step, "fp32_floor_ms": fp32_floor, "fp64_floor_ms": fp64_floor, "hbm_floor_ms": hbm_floor,
                             "executed_fp32_flops": step_exec_flops, "dram_bytes": step_bytes,
                             "algorithmic_flops": step_flops,
                             "algorithmic_frac": step_flops / (ms_per_step * 1e-3) / 1e12 / fp32_peak / world},
                    "hbm": {"kernel_gbs": (traffic / (launch_ms * 1e-3) / 1e9) if traffic else None,
                            "kernel_frac": (traffic / (launch_ms * 1e-3) / 1e9 / hbm_peak) if traffic else None,
                            "step_gbs": (step_bytes / (ms_per_step * 1e-3) / 1e9) if step_bytes else None,
                            "step_frac": (step_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_peak) if step_bytes else None,
                            "peak_gbs": hbm_peak, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s",
                            "workspace_bytes_per_sample": ws_bytes_one_chunk / max(1, min(S, args.chunk) if args.chunk > 0 else S)}}
        # ---------------- CPU baseline (bounded sample) on this box's host cores
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            sec = cpu_port_eval(args.cpu_samples, N, T, make_data(N, T))
            cpu = {"value": args.cpu_samples * N / sec, "unit": "trial-evals/s", "cores": os.cpu_count() or 1, "kind": "port",
                   "sample": f"{args.cpu_samples} parameter samples x {N} trials x T={T}, one fwd+grad eval by torch-float64 "
                             f"autograd over the oracle's restatement of the reference scans ({sec:.1f} s)"}
        if world == 1 and not args.no_secondary and not args.no_c4:
            try:
                c4_val, c4_ms, c4_k, c4_g = bench_c4(dev)
            except Exception as e:
                print(f"bench: secondary workload bench_c4 failed: {e!r}", file=sys.stderr)
                c4_val, c4_ms, c4_k, c4_g = float("nan"), float("nan"), {}, None
            secondary.append({"workload": "c4: TemporalDelayModel(PointMassBoundedActor, delay=2) (x=b=12, joint dim 24), 4,096 parameter "
                                          "samples x 50 trials x T=600, grad wrt 4 parameters per sample, public API (large-system kernels)",
                              "value": c4_val, "unit": "trial-evals/s", "ms_per_eval": c4_g or c4_ms, "ms_per_eval_eager": c4_ms,
                              "kernel_ms": c4_k, "note": "ms_per_eval = replayed from a CUDA graph when available; kernel_ms = per-kernel "
                                                         "CUDA-event times of the eager evaluation"})
        line = {"metric": "trial log-lik+grad evals/sec", "value": value, "unit": "trial-evals/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64 per-sample recursions + f32 per-trial recursions (f32 I/O)",
                "data": "synthetic", "config": dict(workload_config(args, world), kernel_dims=[dims.x, dims.b, dims.u, dims.y, dims.d],
                                                    kernel_trials=dims.N, factorized_axes=not args.no_factorize,
                                                    chunks_per_step=-(-S // args.chunk) if args.chunk > 0 else 1),
                "trial_steps_per_sec": value * T,
                "e2e": {"value": e2e_val, "unit": "trial-evals/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": int(theta_host.numel() * 4 + x_host.numel() * 4),
                        "d2h_bytes_per_step": int(out_host.numel() * 4)},
                "gpu_launches": int(launches_per_step * args.steps),
                "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu, "secondary": secondary or None, "clocks": clocks}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def _claim_stdout():
    """Route everything that libraries print on fd 1 (e.g. the NCCL version banner) to stderr; the one JSON line is
    written to the real stdout by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def _finite(o):
    """Strict JSON: non-finite floats (a failed secondary workload) become null."""
    if isinstance(o, float):
        return o if np.isfinite(o) else None
    if isinstance(o, dict):
        return {k: _finite(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_finite(v) for v in o]
    return o


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(_finite(line), allow_nan=False) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=65536, help="parameter samples per step IN TOTAL (config c3: 65,536), sharded over the GPUs")
    ap.add_argument("--trials", type=int, default=100)
    ap.add_argument("--T", type=int, default=1200)
    ap.add_argument("--chunk", type=int, default=0, help="max samples per internal workspace chunk (0 = as many as fit)")
    ap.add_argument("--cpu-samples", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the secondary c4 (large-system) measurement")
    ap.add_argument("--no-secondary", action="store_true", help="skip all secondary workloads (c2, c4, c5)")
    ap.add_argument("--streams", type=int, default=0, help="internal concurrent sample slices (0 = library default)")
    ap.add_argument("--contrib-warps", type=int, default=0)
    ap.add_argument("--overlap", type=int, default=-1, help="kernel-overlap mask (see lqgk_set_kernel_overlap); -1 = library default")
    ap.add_argument("--pipe-max", type=int, default=-1, help="largest chunk (samples) that uses the pipelined launch sequence; -1 = library default")
    ap.add_argument("--pipe-segments", type=int, default=6)
    ap.add_argument("--no-factorize", action="store_true", help="run the general 2-D (n=10) kernels instead of the per-axis factorisation")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (device-resident sweep and "
                                                          "per-trial log-likelihoods, end-to-end ll + gradient) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
