"""Backward Riccati recursion for the LQR control gains -- drop-in for ``lqg/control/lqr.py:8-42``.

``backward(spec, eps)`` returns ``Gains(L, l, H)`` with the reference's shapes ``L[T,u,b]``, ``l[T,u]``,
``H[T,u,u]`` (``H`` is the eigen-shifted ``Ht`` as in lqr.py:36,42).  The sweep runs in one CUDA kernel
(``k_lqr_fwd``: one thread per parameter sample, FP64, t = T-1..0).

``L`` is differentiable with respect to the spec's ``A``, ``B``, ``Q``, ``R`` and ``Qf`` (time-invariant specs, ``P = 0``): its
backward is one CUDA adjoint call (``lqgk_gains_vjp_*``) that recomputes the sweep and runs the Riccati adjoint.  ``l`` and
``H`` are not differentiable (``l`` is zero in every reference model; ``H`` is a by-product).  Without inputs that require
grad the call is the plain gains call."""
from typing import NamedTuple, Optional

import torch

from lqg_b200 import runtime
from lqg_b200.spec import LQGSpec


class Gains(NamedTuple):
    """LQR control gains"""

    L: torch.Tensor
    l: torch.Tensor
    H: Optional[torch.Tensor] = None


def backward(spec: LQGSpec, eps: float = 1e-8) -> Gains:
    L, l, H = runtime.lqr_backward(spec, eps=eps)
    return Gains(L=L, l=l, H=H)
