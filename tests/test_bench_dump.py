"""bench.py --dump-outputs: what the last timed step computed is written as float32 .npy files, and
an array too large to write whole is the same seeded sample of its elements on every run."""
import numpy as np
import torch

import bench


def test_dump_outputs_float32_whole_and_sampled(tmp_path):
    n = bench.DUMP_MAX_ELEMS
    small = torch.randn(3, 5, dtype=torch.bfloat16)
    big = torch.arange(2 * n + 8, dtype=torch.float32).reshape(-1, 8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), [("out", big), ("loss", torch.tensor(1.5)),
                                               ("grad.w", small)])
    a = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ("out", "loss", "grad.w")}
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss"].shape == () and float(a["loss"]) == 1.5
    assert np.array_equal(a["grad.w"], small.float().numpy())
    # sampled: n distinct flat indices in ascending order, identical from run to run
    idx = a["out"].astype(np.int64)
    assert idx.shape == (n,) and np.all(np.diff(idx) > 0) and idx[-1] < big.numel()
    assert np.array_equal(a["out"], np.load(tmp_path / "b" / "out.npy"))
