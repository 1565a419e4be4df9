"""bench.py --dump-outputs: the stored sample of a large output is the same on every run, the dump stays under
64 MB, and float64 outputs are not narrowed."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_fixed_sample_and_dtypes(tmp_path):
    n = bench.DUMP_SAMPLE + 4096
    big = torch.arange(n, dtype=torch.float32) * 0.5
    outs = (big, torch.tensor(1.25, dtype=torch.float64), torch.tensor([3.0, 4.0], dtype=torch.float16))
    names = ("big", "scalar", "small")
    bench.dump_outputs(str(tmp_path / "a"), names, outs)
    bench.dump_outputs(str(tmp_path / "b"), names, [t.clone() for t in outs])
    a = {k: np.load(tmp_path / "a" / (k + ".npy")) for k in names}
    b = {k: np.load(tmp_path / "b" / (k + ".npy")) for k in names}
    for k in names:
        assert np.array_equal(a[k], b[k])
    assert a["big"].dtype == np.float32 and a["big"].shape == (bench.DUMP_SAMPLE,)
    idx = a["big"] * 2                                     # the values are their own flat indices
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n
    assert a["scalar"].dtype == np.float64 and a["scalar"].shape == () and float(a["scalar"]) == 1.25
    assert a["small"].dtype == np.float32 and a["small"].tolist() == [3.0, 4.0]
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in names) <= 64 << 20
