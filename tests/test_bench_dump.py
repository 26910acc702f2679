"""bench.py --dump-outputs: every matrix's shape and row totals in full, its entries in full or, above the entry
cap, as an evenly spaced sample; float32 / float64 only and at most 64 MB in all.  No GPU needed."""

import os

import numpy as np

import bench


def test_dump_outputs_is_exact_sampled_and_bounded(tmp_path):
    rng = np.random.RandomState(0)
    n = 3 * bench.DUMP_ENTRIES["basefc"] + 5
    row = np.sort(rng.randint(0, 70000, n)).astype(np.int32)
    col = rng.randint(0, 10000, n).astype(np.int32)
    val = rng.randint(1, 100, n).astype(np.int32)
    small = (np.array([0, 2, 2], np.int32), np.array([1, 0, 3], np.int32), np.array([5, 7, 1 << 25], np.int32), (3, 4))
    empty = (np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32), (6, 4))
    bench.dump_outputs(str(tmp_path), {"basefc": (row, col, val, (70000, 10000)), "baf_ad": small, "baf_dp": small,
                                       "baf_oth": empty})
    files = sorted(os.listdir(tmp_path))
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 * 10 ** 6
    got = {f[:-len(".npy")]: np.load(tmp_path / f) for f in files}
    assert len(got) == 4 * 5 and all(a.dtype in (np.float32, np.float64) for a in got.values())

    cap = bench.DUMP_ENTRIES["basefc"]
    idx = np.arange(cap, dtype=np.int64) * n // cap
    assert got["basefc_shape"].tolist() == [70000, 10000, n]
    assert np.array_equal(got["basefc_row_sum"], np.bincount(row, weights=val, minlength=70000))
    for k, a in (("row", row), ("col", col), ("val", val)):
        assert got["basefc_" + k].dtype == np.float32 and np.array_equal(got["basefc_" + k], a[idx])

    # below the cap: every entry; a count float32 cannot hold exactly is written as float64
    assert got["baf_ad_val"].dtype == np.float64 and got["baf_ad_val"].tolist() == [5, 7, 1 << 25]
    assert got["baf_ad_row"].tolist() == [0, 2, 2] and got["baf_ad_col"].tolist() == [1, 0, 3]
    assert got["baf_ad_row_sum"].tolist() == [5, 0, 7 + (1 << 25)]
    assert got["baf_oth_shape"].tolist() == [6, 4, 0] and got["baf_oth_row_sum"].tolist() == [0] * 6
    assert len(got["baf_oth_val"]) == 0
