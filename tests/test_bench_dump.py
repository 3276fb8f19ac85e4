"""bench.py --dump-outputs without a GPU: which files, in which types, which rows, within the size limit."""
import os

import numpy as np
import pytest
import torch

import bench
from frb_baseband_b200.plan import Plan, PlanConfig


class _FakePlan:
    """What dump_outputs asks of a plan besides the rows: the output sample type and the rescale statistics."""
    view_rows = Plan.view_rows

    def __init__(self, out_nbit, nchan):
        self.cfg = PlanConfig(nchan=nchan, bw_mhz=[-32.0, 32.0], out_nbit=out_nbit)
        self.row_bytes = 2 * nchan * (4 if out_nbit == -32 else out_nbit // 8)

    def rescale(self):
        m = np.arange(2 * self.cfg.nchan, dtype=np.float32).reshape(2, 1, -1)
        return m, 1.0 / (m + 1.0)


@pytest.mark.parametrize("out_nbit,rows", [(8, 1000), (16, 300), (-32, 50), (8, 0)])
def test_dump_outputs(tmp_path, monkeypatch, out_nbit, rows):
    """64 float32 rows at most here: 1000 and 300 rows are sampled, 50 are dumped whole."""
    pl = _FakePlan(out_nbit, 32)
    monkeypatch.setattr(bench, "DUMP_ROW_BYTES", 64 * 4 * 64)
    out = torch.randint(0, 256, (rows + 5, pl.row_bytes), dtype=torch.uint8, generator=torch.Generator().manual_seed(1))
    if out_nbit == -32:
        out[:, 3::4] = 0x3f                                     # finite floats
    got = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch, pl, out, rows)
        got.append({f[:-4]: np.load(tmp_path / d / f) for f in sorted(os.listdir(tmp_path / d))})
    a, b = got
    assert sorted(a) == ["rescale_mean", "rescale_scale", "row_index", "rows"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)          # the sample is seeded
    idx = a["row_index"].astype(np.int64)
    assert len(idx) == min(rows, 64) and np.all(np.diff(idx) > 0) and (idx.size == 0 or idx[-1] < rows)
    want = pl.view_rows(out[torch.from_numpy(idx)].numpy()).astype(np.float32)
    assert a["rows"].shape == (len(idx), 64) and np.array_equal(a["rows"], want)
    assert np.array_equal(a["rescale_mean"], pl.rescale()[0])


@pytest.mark.parametrize("name", sorted(bench.CONFIGS))
def test_dump_fits_64_mib(name):
    """Row sample, its index and the statistics of every configuration stay within 64 MiB."""
    c = bench.CONFIGS[name]
    elems = c["nif"] * c["nchan"] * (4 if c["pol"] in ("coherence", "IQUV") else 1)
    n = bench.DUMP_ROW_BYTES // (4 * elems)
    assert n >= 1000 and 4 * n * elems + 8 * n + 2 * 4 * elems <= 64 << 20
