"""Times lqr.backward + kf.forward with their gradients (the gains adjoint, lqgk_gains_vjp_*) and, as the comparison, torch
autograd through the float64 oracle (oracle/lqg_torch.py) on the same GPU.

    python tools/bench_gains_vjp.py [--reps 3] [--out FILE]

Workloads (FP64 I/O, parameters of every sample drawn around the model defaults, loss = sum(L) + sum(K)):
  c3: SubjectiveActor(dim=2), 65,536 samples, T = 1200 (the flagship model and size of bench.py)
  c4: TemporalDelayModel(PointMassBoundedActor, delay=2), 4,096 samples, T = 600 (the large-system kernels)
The oracle keeps every intermediate of the T-step recursions for autograd, which does not fit in memory at those sample
counts; it runs on the first --oracle-samples samples and its time is reported at that count (per-sample times are given for
both).  Times are CUDA events around each phase after one warm-up evaluation; one JSON line goes to stdout (and --out)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lqg_b200.belief import kf
from lqg_b200.control import lqr
from oracle import lqg_torch as OT

SUBJ = dict(action_cost=1.0, action_variability=0.5, subj_noise=1.0, subj_vel_noise=0.5, sigma_target=9.0, sigma_cursor=6.0)
PM = dict(action_variability=1e-3, sigma_target=6.0, sigma_cursor=6.0, action_cost=0.01)


def model(name, th, T, dev):
    from lqg_b200.tracking import PointMassBoundedActor, SubjectiveActor
    from lqg_b200.tracking.delay import TemporalDelayModel
    if name == "c3":
        return SubjectiveActor(dim=2, T=T, device=dev, **th)
    return TemporalDelayModel(PointMassBoundedActor(T=T, device=dev, **th), 2)


def params(name, S, dev):
    rng = np.random.default_rng(3)
    base = SUBJ if name == "c3" else PM
    return {k: torch.tensor(v * np.exp(0.2 * rng.standard_normal(S)), dtype=torch.float64, device=dev, requires_grad=True)
            for k, v in base.items()}


def gains_lqg_b200(m, T):
    return lqr.backward(m.actor).L, kf.forward(m.actor, None)


def gains_oracle(m, T):
    a = {k: getattr(m.actor, k).select(-3, 0) for k in ("A", "B", "F", "V", "W", "Q", "R")}
    return OT.lqr_backward(a["A"], a["B"], a["Q"], a["R"], T), OT.kf_forward(a["A"], a["F"], a["V"], a["W"], a["V"] @ a["V"].mT, T)


def time_one(name, S, T, gains, reps, dev):
    """(forward ms, backward ms): medians over `reps` evaluations after one warm-up."""
    th = params(name, S, dev)
    fwd, bwd = [], []
    for r in range(reps + 1):
        for t in th.values():
            t.grad = None
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        L, K = gains(model(name, th, T, dev), T)
        loss = L.sum() + K.sum()
        e1.record()
        loss.backward()
        e2.record()
        e2.synchronize()
        assert all(torch.isfinite(t.grad).all() for t in th.values())
        if r > 0:
            fwd.append(e0.elapsed_time(e1))
            bwd.append(e1.elapsed_time(e2))
        del L, K, loss
    return float(np.median(fwd)), float(np.median(bwd))


def card(dev):
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={dev.index or 0}", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [v.strip() for v in q.split(",")]
    except Exception as e:   # (the timing does not depend on it; the record says why it is missing)
        info["power_limit"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--oracle-samples", type=int, nargs=2, default=(512, 256), metavar=("C3", "C4"))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"tool": "bench_gains_vjp", "card": card(dev), "io": "float64", "loss": "sum(L) + sum(K)", "workloads": {}}
    for (name, S, T), So in zip((("c3", 65536, 1200), ("c4", 4096, 600)), a.oracle_samples):
        f, b = time_one(name, S, T, gains_lqg_b200, a.reps, dev)
        fo, bo = time_one(name, So, T, gains_oracle, max(1, a.reps - 2), dev)
        torch.cuda.empty_cache()
        res["workloads"][name] = {
            "S": S, "T": T,
            "lqg_b200": {"forward_ms": f, "backward_ms": b, "us_per_sample": 1e3 * (f + b) / S},
            "oracle_torch_autograd": {"S": So, "forward_ms": fo, "backward_ms": bo, "us_per_sample": 1e3 * (fo + bo) / So}}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
