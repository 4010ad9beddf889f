"""bench.py --dump-outputs: every field of the result tables as float64 .npy, exact, and a fixed sample within the size budget."""
import os

import numpy as np

import bench
from grove_b200 import tables as T


def test_dump_writes_every_field_exactly(tmp_path):
    st = np.zeros(3, dtype=T.status_dt)
    st["n_pods"] = [1, 2, 0xFFFFFFFF]
    st["reserved1"][1] = [4, 5, 6]
    pl = np.zeros(2, dtype=T.placement_dt)
    pl["node"] = [7, 8]
    bench.dump_outputs(str(tmp_path), {"gang_status": st, "placements": pl})
    assert sorted(os.listdir(tmp_path)) == sorted([f"gang_status.{f}.npy" for f in T.status_dt.names] +
                                                  ["placements.clique.npy", "placements.node.npy"])
    for name, a in (("gang_status", st), ("placements", pl)):
        for f in a.dtype.names:
            d = np.load(tmp_path / f"{name}.{f}.npy")
            assert d.dtype == np.float64 and np.array_equal(d, a[f]), (name, f)


def test_dump_samples_a_table_over_budget(tmp_path):
    nodes = np.zeros(1_500_000, dtype=T.node_dt)
    nodes["free_cpu_milli"] = np.arange(len(nodes))
    rows = []
    for run in ("a", "b"):
        out = tmp_path / run
        bench.dump_outputs(str(out), {"nodes": nodes})
        assert sum(p.stat().st_size for p in out.iterdir()) <= 64 * 10**6
        rows.append(np.load(out / "nodes.rows.npy"))
        assert 0 < len(rows[-1]) < len(nodes)
        assert np.array_equal(np.load(out / "nodes.free_cpu_milli.npy"), rows[-1])
    assert np.array_equal(rows[0], rows[1])
