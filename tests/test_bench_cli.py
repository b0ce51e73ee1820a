"""CPU tests of bench.py's command line and of --dump-outputs (the step results written for output-by-output comparison of
two builds)."""
import os
import sys

import numpy as np
import pytest
import torch

import bench


def _results(B=40, n=30, n_out=50):
    """Shaped like a c1 step's results; every value encodes its instance (row), so sampled rows can be traced back."""
    row = torch.arange(B, dtype=torch.float64)
    return dict(alpha=row[:, None] + torch.linspace(0, 0.5, n, dtype=torch.float64),
                status=torch.zeros(B, dtype=torch.int32),
                n_out=(row + 7).to(torch.int32),
                raceline=row[:, None, None].expand(B, n_out, 2).contiguous(),
                side=torch.arange(8, dtype=torch.float64),             # a result of another batch size (c5's alpha_mc)
                qp_solves=123)                                          # a plain count (c3)


def _files(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_every_result_in_float64_unsampled_when_it_fits(tmp_path):
    res = _results()
    bench.dump_outputs(res, str(tmp_path))
    got = _files(tmp_path)
    assert set(got) == set(res)
    for k, a in got.items():
        assert a.dtype == np.float64
        assert np.array_equal(a, np.asarray(res[k]))


def test_dump_samples_the_same_instances_of_every_array_within_the_limit(tmp_path):
    res = _results()
    limit = 4096 * len(res) + 12_000
    for d in ("a", "b"):
        bench.dump_outputs(res, str(tmp_path / d), limit=limit)
    a, b = _files(tmp_path / "a"), _files(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= limit
    for k in a:
        assert np.array_equal(a[k], b[k])                                   # the sample depends on the shapes only
    rows = a["alpha"][:, 0]
    assert 0 < len(rows) < 40 and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["n_out"], rows + 7) and np.array_equal(a["raceline"][:, 0, 0], rows)
    assert a["qp_solves"] == 123 and 0 < len(a["side"]) < 8


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
