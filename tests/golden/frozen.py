"""Storage format of the frozen reference outputs (ref_slam.npz, ref_slam_params.npz, msrd_b2s3.npz), shared by the
scripts that write them and the tests that read them, so that every fixture file stays under 1 MB.

  * An array with many rows (a map's points, normals, colours, confidences; a frame map's pixels) is stored as
    `<key>/sample`: every ROW_STRIDE-th row (PIXEL_STRIDE-th pixel of a frame map), plus `<key>/sum` and
    `<key>/abs_sum`: float64 column sums and absolute sums over ALL rows.  `assert_rows_close` compares the sampled rows
    element by element and the sums with the bound that the same element-wise tolerance implies for every row, so
    rows outside the sample are still checked in aggregate.
  * Index tables are stored in the narrowest integer type that holds them; `load` widens every integer array back to
    int64.
"""
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROW_STRIDE = 8
PIXEL_STRIDE = 17  # coprime with the image widths and heights used, so the sample walks across rows and columns


def pack_rows(out, key, a, stride=ROW_STRIDE):
    a = np.asarray(a)
    out[key + "/sample"] = a[::stride]
    out[key + "/sum"] = a.astype(np.float64).sum(0)
    out[key + "/abs_sum"] = np.abs(a.astype(np.float64)).sum(0)


def narrow_int(a):
    a = np.asarray(a)
    for t in (np.int16, np.int32):
        if a.size == 0 or (a.min() >= np.iinfo(t).min and a.max() <= np.iinfo(t).max):
            return a.astype(t)
    return a


def load(name):
    """The fixture file `name` as a dict of numpy arrays, integer arrays widened to int64."""
    with np.load(os.path.join(HERE, name)) as z:
        return {k: (z[k].astype(np.int64) if np.issubdtype(z[k].dtype, np.signedinteger) else z[k]) for k in z.files}


def assert_rows_close(got, ref, key, rtol, atol, stride=ROW_STRIDE):
    """`got` (all rows, in the reference's order) against the rows stored under `key` with pack_rows."""
    got = got.detach().cpu().numpy() if torch.is_tensor(got) else np.asarray(got)
    sample = np.asarray(ref[key + "/sample"])
    assert got[::stride].shape == sample.shape, (key, got.shape, sample.shape)
    torch.testing.assert_close(torch.from_numpy(got[::stride]), torch.from_numpy(sample), rtol=rtol, atol=atol)
    bound = got.shape[0] * atol + rtol * np.asarray(ref[key + "/abs_sum"])
    diff = np.abs(got.astype(np.float64).sum(0) - np.asarray(ref[key + "/sum"]))
    assert np.all(diff <= bound * (1 + 1e-9) + 1e-12), (key, diff, bound)
