"""lqg_b200.io.load_tracking_data against the output of the reference's own loader (lqg/io.py) on the reference's data file,
whose first blob-width condition tests/golden/ref_c2r_bounded_realdata_T1067.npz stores.  The data file is not part of this
repository, so the test writes a data.mat of the same layout (per trial: blob width in pixels, raw target and response traces)
whose first condition holds the stored traces inside the clip / delay windows and NaN outside them, with five further
conditions of random walks, trials of all widths interleaved.  Every trial of the stored condition gets its own offsets of
target and response (the real file's traces are screen positions, not centred): the loader must remove them through its
per-trial mean subtraction and its re-referencing to the first target sample."""
import os

import numpy as np
import scipy.io as spio

from lqg_b200 import io
from tests import helpers as H

DELAY, CLIP = 12, 120
SIGMA_PX = (11, 13, 17, 21, 25, 29)                   # blob widths in pixels (uint8, as in the reference's data file)
WIDTHS = (15.0, 17.0, 22.0, 28.0, 33.0, 38.0)         # the same in arcmin, rounded; the first is the stored condition


def test_loader_matches_reference_loader_output(tmp_path):
    X = np.load(os.path.join(H.ROOT, "tests", "golden", "ref_c2r_bounded_realdata_T1067.npz"))["X"]   # [20, 1068, 2]
    n, steps = X.shape[0], X.shape[1] + CLIP + DELAY
    rng = np.random.default_rng(0)
    sigma = rng.permutation(np.repeat(np.array(SIGMA_PX, dtype=np.uint8), n))
    walk = np.cumsum(rng.standard_normal((len(sigma), steps, 2)), axis=1)
    target, response = walk[..., 0], walk[..., 1]
    first = np.flatnonzero(sigma == SIGMA_PX[0])
    target[first], response[first] = np.nan, np.nan
    target[first, CLIP:steps - DELAY] = X[..., 0]
    response[first, CLIP + DELAY:] = X[..., 1]
    offset = rng.integers(-40, 40, (n, 2))
    target[first] += offset[:, :1]
    response[first] += offset[:, 1:]
    spio.savemat(str(tmp_path / "data.mat"), dict(sigma=sigma, target=target, response=response))

    data, sigmas = io.load_tracking_data(delay=DELAY, clip=CLIP, data_path=str(tmp_path))
    assert data.shape == (6, 20, 1068, 2) and data.dtype == np.float32 and len(sigmas) == 6
    assert np.array_equal(sigmas, WIDTHS) and np.isfinite(data).all()
    assert np.all(data[:, :, 0, 0] == 0.0)
    # The target channel comes back up to float32 rounding.  The response channel differs by the shift the reference's float32
    # mean subtraction left in its output: there the per-trial means of target and response, equal in exact arithmetic,
    # differ by up to 1.4e-3.
    assert np.abs(data[0, ..., 0] - X[..., 0]).max() <= 1e-5
    assert np.abs(data[0, ..., 1] - X[..., 1]).max() <= 2e-3
