"""The allocate action's keyed job order (default) against the replica job-order tree (KAI_JOB_ORDER=replica) on the GPU:
identical visits, bindings, statuses, node and queue tables on the config3-shaped cycle, where the keyed order is taken,
and on the seeded five-action fuzz cycles, where most snapshots fall back to the replica."""
import numpy as np
import pytest

import dsl
from kai_scheduler_b200 import abi, synthetic
from kai_scheduler_b200.engine import Engine
from test_engine_gpu import assert_same
from test_snapshot_io import _random_topology

pytestmark = pytest.mark.gpu


def _cycle(snap, actions, cfg=None):
    e = Engine(cfg)
    e.load(snap)
    out = [e.run(a) for a in actions]
    e.close()
    return out


def _both_orders(monkeypatch, snap, actions, cfg=None):
    monkeypatch.delenv("KAI_JOB_ORDER", raising=False)
    keyed = _cycle(snap, actions, cfg)
    monkeypatch.setenv("KAI_JOB_ORDER", "replica")
    replica = _cycle(snap, actions, cfg)
    monkeypatch.delenv("KAI_JOB_ORDER")
    return keyed, replica


@pytest.mark.parametrize("kw", [
    synthetic.CYCLE_CONFIGS["config3-cycle-small"],
    dict(n_nodes=4000, n_jobs=4000, tasks_per_job=4, n_queues=1000, gpus_per_node=4, running_nodes=8),  # 250 departments
])
def test_config3_cycle_keyed_equals_replica(kw, monkeypatch, capfd):
    snap = synthetic.cycle_snapshot(**kw)
    monkeypatch.setenv("KAI_PROFILE", "1")
    keyed, replica = _both_orders(monkeypatch, snap, ["allocate", "reclaim"])
    err = capfd.readouterr().err
    assert "[kai] job order: keyed" in err, err[-2000:]
    assert "[kai] job order: replica (KAI_JOB_ORDER=replica" in err
    for a, b in zip(keyed, replica):
        assert_same(a, b)
        assert a.pods_evicted == b.pods_evicted
    assert len(keyed[0].visits) == kw["n_jobs"]


@pytest.mark.parametrize("chunk", range(4))
def test_fuzz_cycles_keyed_equals_replica(chunk, monkeypatch):
    actions = ["allocate", "consolidation", "reclaim", "preempt", "stalegangeviction"]
    cfg = abi.make_config(allow_consolidating_reclaim=True, max_consolidation_preemptees=-1)
    for seed in range(chunk * 25, (chunk + 1) * 25):
        rng = np.random.default_rng(5000 + seed)
        snap, _meta = dsl.build_snapshot(_random_topology(rng))
        keyed, replica = _both_orders(monkeypatch, snap, actions, cfg)
        for act, a, b in zip(actions, keyed, replica):
            try:
                assert_same(a, b)
            except AssertionError as ex:
                raise AssertionError(f"seed {seed} action {act}: {ex}") from None
            assert a.pods_evicted == b.pods_evicted, f"seed {seed} action {act}"
