"""Latency / strong-scaling regime: ms per log-likelihood+gradient through the public API as a function of the number of
parameter samples and of the library's concurrent sample slices (lqgk_set_streams).
python tools/bench_streams.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from lqg_b200 import abi
from lqg_b200.tracking import SubjectiveActor

dev = torch.device("cuda:0")
lib = abi.load_library()
N, T = 100, 1200
x = bench.make_data_gpu(N, T, dev)


def run(S, reps=5):
    theta = torch.tensor(bench.make_theta(S, 11), device=dev, requires_grad=True)

    def ev():
        theta.grad = None
        m = SubjectiveActor(dim=2, T=T, device=dev, **{n: theta[:, i] for i, n in enumerate(bench.PARAM_NAMES)})
        ll = m.log_likelihood(x).sum()
        ll.backward()
        return ll
    ev(); ev(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ev()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


streams = (1, 2, 4, 8, 16)
print("| samples | " + " | ".join(f"{n} slices" for n in streams) + " |\n|---:|" + "---:|" * len(streams))
for S in (512, 1024, 2048, 4096, 8192, 16384, 32768):
    row = []
    for n in streams:
        lib.set_streams(n)
        row.append(run(S))
    lib.set_streams(1)
    print(f"| {S} | " + " | ".join(f"{v:.2f}" for v in row) + " |")
