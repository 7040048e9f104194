"""bench.py --dump-outputs on the CPU arm: the last step's results land as float64 .npy files, the same arguments write the
same arrays, and results above the size limit are written as a fixed-seed sample with the kept positions."""
import os
import subprocess
import sys

import numpy as np

import bench
from kai_scheduler_b200 import synthetic
from oracle_lib import Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(d):
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cycle5-small",
                    "--steps", "2", "--warmup", "0", "--dump-outputs", str(d)], check=True, capture_output=True)
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_repeatable_and_holds_the_last_step(tmp_path):
    a, b = _bench_dump(tmp_path / "a"), _bench_dump(tmp_path / "b")
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k]), k
    o = Oracle()
    o.load(synthetic.config_snapshot("cycle5-small"))
    for action in synthetic.CONFIG_ACTIONS["cycle5-small"]:
        r = o.run(action)
        assert np.array_equal(a[f"{action}_task_node"], r.task_node)
        assert np.array_equal(a[f"{action}_task_status"], r.task_status)
        assert np.array_equal(a[f"{action}_node_idle"], r.node_idle)
        assert np.array_equal(a[f"{action}_visit_job"], r.visits[:, 0])
        assert list(a[f"{action}_pods_placed_evicted"]) == [r.pods_placed, r.pods_evicted]


def test_large_dump_is_a_fixed_sample(tmp_path, monkeypatch):
    snap = synthetic.config_snapshot("config3-cycle-small")
    o = Oracle()
    o.load(snap)
    results = [(a, o.run(a)) for a in ("allocate", "reclaim")]
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 40_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), results)
    names = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / f) - 128 for f in names) <= 40_000  # 128: .npy header
    for f in names:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    t = np.load(tmp_path / "a" / "reclaim_task_node_index.npy").astype(int)
    assert 0 < len(t) < snap.n_tasks
    assert np.array_equal(np.load(tmp_path / "a" / "reclaim_task_node.npy"), results[1][1].task_node[t])
    assert np.array_equal(np.load(tmp_path / "a" / "reclaim_task_status_index.npy"), t)
    n = np.load(tmp_path / "a" / "allocate_node_idle_index.npy").astype(int)
    assert np.array_equal(np.load(tmp_path / "a" / "allocate_node_idle.npy"), results[0][1].node_idle[:, n])
