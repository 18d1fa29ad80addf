"""bench.py's host-side bookkeeping (no GPU): the byte count of the stand-alone InstanceNorm applies that are left, and the rule that a
measured-traffic figure is only quoted for the sources and the micro-batch it was captured on."""
import json
import os

import pytest

from tests.conftest import ROOT


def test_standalone_apply_bytes():
    import bench
    c, H, W = 64, 512, 512
    msb3 = 3 * (2 * 128 * 256 * 256 + 256 * 128 * 128)                 # down1, up1 (C = 128 at H/2) and down2 (C = 256 at H/4): 2 reads + 1 write
    assert bench.standalone_apply_elems(3, c, H, W) == msb3
    assert bench.standalone_apply_elems(5, c, H, W) == msb3 + 2 * c * H * W + 3 * c * H * W      # + initial IN (1R + 1W) + up2's block


def test_measured_traffic_is_tied_to_sources_and_micro_batch():
    import bench
    d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    v, note = bench.measured_traffic("conv_dram_bytes_per_launch", d.get("micro_batch", 16))
    if d["csrc_sha"] == bench.csrc_digest():
        assert v == d["conv_dram_bytes_per_launch"] and d["ncu_file"] in note
        other, why = bench.measured_traffic("conv_dram_bytes_per_launch", d.get("micro_batch", 16) * 2)
        assert other is None and "micro-batch" in why
    else:
        assert v is None and "stale" in note


def test_output_dump_is_a_fixed_sample(tmp_path):
    """--dump-outputs: a small output is written whole; a large one as the same DUMP_MAX_ELEMS-element sample in every run."""
    import numpy as np
    import torch
    import bench
    small = torch.rand(2, 3, 8, 8)
    assert np.array_equal(bench.dump_sample(small), small.numpy())
    big = torch.arange(bench.DUMP_MAX_ELEMS + 1000, dtype=torch.float32)
    s = bench.dump_sample(big)
    assert s.shape == (bench.DUMP_MAX_ELEMS,) and np.array_equal(s, bench.dump_sample(big.clone()))
    assert (np.diff(s) > 0).all()                                     # distinct elements, in index order
    half = bench.dump_sample(big, bench.DUMP_MAX_ELEMS // 2)            # each of two ranks samples its share of the budget
    assert half.shape == (bench.DUMP_MAX_ELEMS // 2,)
    bench.write_outputs(str(tmp_path), {"stylised": half}, rank=1, world=2)
    assert np.array_equal(np.load(tmp_path / "stylised_rank1.npy"), half)
    with pytest.raises(AssertionError):                               # a full budget on each of two ranks is over 64 MB
        bench.write_outputs(str(tmp_path), {"stylised": s}, rank=0, world=2)
