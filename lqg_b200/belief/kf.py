"""Forward Kalman-gain recursion -- drop-in for ``lqg/belief/kf.py:6-21``.

``forward(spec, Sigma0)`` returns ``K[T,b,y]`` (or ``[S,T,b,y]``) from one CUDA kernel (``k_kf_fwd``: one thread
per parameter sample, FP64, t = 0..T-1).

``K`` is differentiable with respect to the spec's ``A``, ``F``, ``V``, ``W`` and ``Sigma0`` (time-invariant specs; without
``Sigma0`` the prior V V^T sends its gradient to ``V``): the backward is one CUDA adjoint call (``lqgk_gains_vjp_*``)."""
import torch

from lqg_b200 import runtime
from lqg_b200.spec import LQGSpec


def forward(spec: LQGSpec, Sigma0: torch.Tensor) -> torch.Tensor:
    return runtime.kf_forward(spec, Sigma0)
