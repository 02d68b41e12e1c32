"""GPU parity tests proper: the CUDA library, called through the C ABI, against the float64 oracle.

Tolerances are the north star's: gains and log-likelihood rtol 1e-4, gradients rtol 1e-3 (vs float64)."""
import numpy as np
import pytest
import torch

from lqg_b200 import abi
from tests import helpers as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    return abi.load_library()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.mark.parametrize("name,d", [("bounded", 2), ("subjective", 2), ("relobs", 2), ("bounded2", 4), ("relobs2", 4),
                                    ("subjective2", 4), ("pointmass", 2), ("hand", 2), ("delay2", 2)])
def test_gains_match_oracle(lib, dev, name, d):
    case = H.Case(name, S=3, T=300, N=2, d=d, want_grad=False)
    H.check_gains(lib, dev, case, torch.float64, rtol=1e-9)
    H.check_gains(lib, dev, case, torch.float32, rtol=1e-4)


@pytest.mark.parametrize("name,d,N", [("bounded", 2, 20), ("subjective", 2, 33), ("relobs", 2, 7), ("bounded2", 4, 64),
                                      ("relobs2", 4, 20), ("subjective2", 4, 100), ("pointmass", 2, 50), ("hand", 2, 50),
                                      ("delay2", 2, 40)])
def test_loglik_and_gradients_match_oracle(lib, dev, name, d, N):
    case = H.Case(name, S=3, T=200, N=N, d=d, weights=True)
    H.check_fwd(lib, dev, case, torch.float32)
    H.check_fwd(lib, dev, case, torch.float64)
    H.check_vjp(lib, dev, case, torch.float32)
    H.check_vjp(lib, dev, case, torch.float64)


def test_large_system_c4(lib, dev):
    """BASELINE config c4 model: TemporalDelayModel(PointMassBoundedActor, delay=2): x=b=12, joint dim 24 -- the
    large-system kernels (lqgk_bigw.cuh), 50 trials as in the config."""
    case = H.Case("pmdelay2", S=40, T=120, N=50, d=2, weights=True)
    H.check_gains(lib, dev, case, torch.float64, rtol=1e-9)
    H.check_fwd(lib, dev, case, torch.float32)
    H.check_vjp(lib, dev, case, torch.float32)
    H.check_vjp(lib, dev, case, torch.float64, max_chunk=32)      # two chunks


def test_large_system_c4_full_horizon(lib, dev):
    """c4 horizon T=600, 50 trials: log-likelihood rtol 1e-4 and PARAMETER gradients rtol 1e-3.  (With action_variability
    1e-3 the innovation covariance is ~1e-6 and the FP32 per-trial arithmetic leaves 3e-3..6e-3 relative error in single
    base-matrix cotangents such as dA, which no model parameter feeds; the per-matrix check is made at T=120 above.)"""
    case = H.Case("pmdelay2", S=3, T=600, N=50, d=2)
    assert H.check_param_vjp(lib, dev, case, torch.float32) < 1e-3


@pytest.mark.parametrize("name,d,N", [("bounded", 2, 20), ("subjective", 2, 33), ("relobs", 2, 7), ("subjective2", 4, 40), ("pointmass", 2, 20),
                                      ("hand", 2, 20), ("delay2", 2, 20)])
def test_many_samples_use_the_thread_per_sample_covariance_kernels(lib, dev, name, d, N):
    """Calls with at most 512 samples (lqgk_set_warp_cov_max_samples) run the warp-per-sample covariance kernels (everything
    above in this file); larger ones the thread-per-sample kernels with the TMA rings -- checked here against the same
    oracle (samples repeated)."""
    case = H.Case(name, S=3, T=100, N=N, d=d, weights=True)
    H.check_vjp_tiled(lib, dev, case, reps=352)       # 1,056 systems


def test_covariance_kernel_variants_agree(lib, dev):
    """Same call with the threshold forced either way: thread-per-sample and warp-per-sample covariance kernels give the same
    log-likelihoods and gradients (to FP64 rounding of the gradient accumulators)."""
    case = H.Case("subjective", S=40, T=120, N=30, d=2, weights=True)
    try:
        lib.set_warp_cov_max_samples(0)
        H.check_vjp(lib, dev, case, torch.float64)
        H.check_fwd(lib, dev, case, torch.float32)
        lib.set_warp_cov_max_samples(1 << 30)
        H.check_vjp(lib, dev, case, torch.float64)
        H.check_fwd(lib, dev, case, torch.float32)
    finally:
        lib.set_warp_cov_max_samples(512)
    case = H.Case("subjective2", S=70, T=60, N=12)
    H.check_vjp(lib, dev, case, torch.float32)                  # one chunk, 3 warps, padded
    H.check_vjp(lib, dev, case, torch.float32, max_chunk=32)    # three chunks
    H.check_fwd(lib, dev, case, torch.float32, max_chunk=32)


def test_more_trials_than_one_pass(lib, dev):
    case = H.Case("bounded", S=2, T=50, N=150)
    H.check_vjp(lib, dev, case, torch.float32)


@pytest.mark.parametrize("name,d,N", [("bounded", 2, 301), ("subjective", 2, 300), ("bounded2", 4, 150), ("subjective2", 4, 131),
                                      ("delay2", 2, 129)])
def test_several_trial_passes_and_odd_trial_counts(lib, dev, name, d, N):
    """More trials than one pass of 32 x RT per warp (RT <= 8 small systems, <= 4 larger ones): the second pass starts at
    base > 0 and accumulates into the per-step sums; odd N exercises the zero pad element of the paired state history."""
    case = H.Case(name, S=3, T=40, N=N, d=d, weights=True)
    H.check_fwd(lib, dev, case, torch.float32)
    H.check_vjp(lib, dev, case, torch.float32)


def test_config_c1_shape(lib, dev):
    """BASELINE config 1: BoundedActor 1-D, T=500, 20 trials (reference tests/infer_test.py:19-26 shape)."""
    case = H.Case("bounded", S=1, T=500, N=20, seed=123)
    H.check_vjp(lib, dev, case, torch.float32)
    assert -1.3e3 < case.ll.mean() < -0.9e3


def test_config_c2_horizon(lib, dev):
    """BASELINE config 2 shape: SubjectiveActor 2-D, T=1200, 20 trials, 6 conditions (sigma_target varies)."""
    case = H.Case("subjective2", S=6, T=1200, N=20, seed=5)
    H.check_vjp(lib, dev, case, torch.float32)


@pytest.mark.parametrize("name,d,N,T,reps", [("subjective", 2, 33, 205, 1), ("subjective", 2, 33, 205, 400), ("subjective2", 4, 40, 131, 1),
                                             ("bounded", 2, 301, 97, 200), ("delay2", 2, 20, 150, 1)])
def test_one_segment_and_many_segments_agree(lib, dev, name, d, N, T, reps):
    """The launch sequence cut into time segments over internal streams (the default, so every other test in this file runs
    it) and its one-segment case on the caller's stream (pipeline off, or kernel overlap off) are the same arithmetic: all
    match the oracle, and each other to FP64-summation-order accuracy.  T is not a multiple of the checkpoint interval or the
    segment count; reps > 1 tiles the samples beyond 512 to reach the thread-per-sample covariance kernels."""
    case = H.Case(name, S=3, T=T, N=N, d=d, weights=True)
    outs = []
    for max_samples, segments, overlap in ((0, 6, 6), (1 << 20, 6, 6), (1 << 20, 11, 6), (1 << 20, 1000, 6), (1 << 20, 6, 0)):
        lib.set_pipeline(max_samples, min(segments, 64))
        lib.set_kernel_overlap(overlap)
        try:
            if reps == 1:
                H.check_vjp(lib, dev, case, torch.float32)
            else:
                H.check_vjp_tiled(lib, dev, case, reps, torch.float32)
            dims = case.lqgk_dims()
            act, dyn = case.tensors(dev, torch.float64)
            x_tm = lib.pack_obs(torch.tensor(case.X, device=dev))
            ws = H.workspace(lib, dims, abi.MODE_VJP, dev)
            ll, ga, gd, _ = lib.loglik_vjp(dims, act, dyn, x_tm, ws=ws, stream=H.stream_of(dev))
            torch.cuda.synchronize()
            outs.append([ll] + list(ga.values()) + list(gd.values()))
        finally:
            lib.set_pipeline(1 << 30, 6)
            lib.set_kernel_overlap(6)
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert torch.allclose(a, b, rtol=1e-9, atol=1e-9 * float(a.abs().max()) + 1e-300)
