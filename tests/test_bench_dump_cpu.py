"""bench.py --dump-outputs (CPU): the files two builds are compared by -- one Float64 .npy per operation of the
step plus the fused ψ(y), the same seeded sample of positions in every run, at most 64 MB in all."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_dump_is_a_fixed_sample_of_each_output(tmp_path):
    n = 4 * bench.DUMP_SAMPLE
    outs = tuple(torch.arange(n, dtype=torch.float64) * k for k in (1, 2, 3))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs, 1.5, 0, 1)
    names = sorted(f"{op}.npy" for op in bench.OPS) + ["psi_prox_l0box.npy"]
    assert sorted(os.listdir(tmp_path / "a")) == sorted(names)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    got = {f: np.load(tmp_path / "a" / f) for f in names}
    assert all(a.dtype == np.float64 for a in got.values())
    assert all(np.array_equal(got[f], np.load(tmp_path / "b" / f)) for f in names)
    pos = got["prox_l0box.npy"]  # outs[0][i] == i: the sampled positions themselves
    assert bench.DUMP_SAMPLE // 2 <= pos.size <= bench.DUMP_SAMPLE and np.all(np.diff(pos) > 0) and pos[-1] < n
    assert np.array_equal(got["prox_lhalfbox.npy"], 2 * pos) and np.array_equal(got["iprox_l0box.npy"], 3 * pos)
    assert got["psi_prox_l0box.npy"].tolist() == [1.5]


def test_small_outputs_are_dumped_whole_and_per_rank(tmp_path):
    outs = tuple(torch.full((1000,), float(k), dtype=torch.float64) for k in (1, 2, 3))
    bench.dump_outputs(str(tmp_path), outs, 0.25, 1, 2)
    assert sorted(os.listdir(tmp_path)) == sorted(f"{op}_rank1.npy" for op in bench.OPS)  # ψ(y) from rank 0 only
    assert np.array_equal(np.load(tmp_path / "iprox_l0box_rank1.npy"), np.full(1000, 3.0))
