#!/usr/bin/env python
"""bench.py — one JSON line per run (driver contract).

A "step" is one scheduling cycle (proportion OnSessionOpen + the allocate and reclaim Actions) over one synthetic
cluster snapshot.  Default workload: the configuration BASELINE.json's metric is quoted on (configs[2]) — 50 000 nodes
("node-%d", 4 GPUs) / 200 000 pending 1-GPU pods in 50 000 gangs of 4 / 1 000 leaf queues under 250 departments, plus
8 nodes full of running over-quota pods: allocate fills the cluster, the gangs left over reclaim (synthetic.cycle_snapshot).
`--config config2` is BASELINE.json configs[1] (10 000 nodes / 40 000 pods, allocate).

After the timed loop the engine's outcome of the last step is compared with the CPU oracle on the same snapshot
(bindings, statuses, victim set, queue shares); the line carries bindings_match / victims_match / max_share_abs_err
and the process exits non-zero on a mismatch.

  value        pods placed per second, device time (CUDA events on the engine's stream) of the open-session
               kernels + the action kernel, snapshot already resident in HBM
  e2e          the same metric through the C-ABI call a Go shim makes: kai_engine_load_snapshot(HOST
               buffers) + kai_engine_run(), host->device and device->host copies inside the timed region
  roofline     dominant kernel k_action: algorithmic bytes = node rows swept x 76 B (SURVEY.md §8d)
  cpu_baseline the CPU oracle (port of the reference's Go path) on this box's host cores

  --impl reference   times the CPU oracle instead (the reference is Go; no Go toolchain exists here or on the
                     GPU box, so the "reference arm" is the restatement in oracle/, all host threads).
  --dump-outputs DIR writes the results of every action of the last timed step as DIR/<action>_<field>.npy (float64),
                     so that two builds run with the same arguments (same seeded inputs) can be compared array by array.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from kai_scheduler_b200 import abi, synthetic  # noqa: E402

METRIC = "pods_placed_per_sec"
UNIT = "pods/s"
BYTES_PER_NODE = (2 * 4 + 1) * 8 + 4  # SURVEY.md §8d: Idle[R]+Releasing[R]+Allocatable[1] f64 + 4 B flags, R=4


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


DUMP_LIMIT_BYTES = 60_000_000  # below 64 MB with the .npy headers


def dump_outputs(out_dir, results):
    """Writes the results of one step, [(action, abi.Result)] in run order, as out_dir/<action>_<field>.npy in float64
    (exact for the int32 fields).  Every array's last axis runs over tasks, visits, queues or nodes.  When the whole
    exceeds DUMP_LIMIT_BYTES, every array keeps the same fixed-seed sample of its last axis (arrays of equal length keep
    the same positions) and <action>_<field>_index.npy lists the kept positions."""
    names = [a for a, _ in results]
    arrays = {}
    for i, (action, r) in enumerate(results):
        tag = action if names.count(action) == 1 else f"{action}{i}"
        fields = {"task_node": r.task_node, "task_status": r.task_status,
                  "visit_job": r.visits[:, 0], "visit_outcome": r.visits[:, 1],
                  "queue_fair_share": r.queue_fair_share, "queue_allocated": r.queue_allocated,
                  "queue_allocated_non_preemptible": r.queue_allocated_non_preemptible,
                  "queue_request": r.queue_request, "total_resource": r.total_resource,
                  "node_idle": r.node_idle, "node_releasing": r.node_releasing,
                  "pods_placed_evicted": [r.pods_placed, r.pods_evicted]}
        arrays.update({f"{tag}_{k}": np.asarray(v, dtype=np.float64) for k, v in fields.items()})
    total = sum(a.nbytes for a in arrays.values())
    keep = 1.0 if total <= DUMP_LIMIT_BYTES else DUMP_LIMIT_BYTES / (2 * total)  # 2: room for the index arrays
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        n = a.shape[-1]
        if keep < 1.0 and n > 1:
            idx = np.sort(np.random.default_rng(0).choice(n, max(1, int(n * keep)), replace=False))
            a = a[..., idx]
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.sm_max = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def reference_sample(config, snap, actions):
    """Bounded sample of the workload for the CPU arm: same cluster (all nodes, all queues), the first gangs of the pending
    list, sized to a few seconds of oracle time per step so that --steps 20 --warmup 5 ends within minutes."""
    if config in synthetic.CYCLE_CONFIGS or config in ("config3", "config3-mixed"):
        kw = dict(synthetic.CYCLE_CONFIGS.get(config) or synthetic.CONFIGS[config])
        gangs = min(kw["n_jobs"], max(1, int(1.0e9 // (kw["n_nodes"] * kw.get("tasks_per_job", 1)))))
        kw["n_jobs"] = gangs
        if config in synthetic.CYCLE_CONFIGS:
            sample = synthetic.cycle_snapshot(**kw)
        else:
            sample = synthetic.benchmark_snapshot(**kw)
        note = (f"per step: the first {gangs} gangs ({gangs * kw.get('tasks_per_job', 1)} pods) of the pending list on the full "
                f"{kw['n_nodes']}-node / {int(sample.queue_parent.shape[0])}-queue cluster, allocate action"
                + (" (the sample leaves free GPUs, so reclaim has no work in it)" if "reclaim" in actions else ""))
        return sample, ["allocate"], note
    return snap, list(actions), "full workload per step"


def run_reference(args, snap, workload, actions=("allocate",), engine_kw=None):
    """--impl reference: the CPU restatement of the reference's Go path (oracle/, 'port': no Go toolchain here or on the
    GPU box) with a pool of host threads, same config / metric, bounded sample per step."""
    from oracle_lib import Oracle
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cores = min(os.cpu_count() or 1, int(os.environ.get("KAI_REF_THREADS", "16")))
    sample, s_actions, note = (snap, list(actions), "full recorded snapshot per step") if args.snapshot else \
        reference_sample(args.config, snap, actions)
    o = Oracle(abi.make_config(**(engine_kw or {})), threads=cores)
    times, placed = [], 0
    for i in range(args.warmup + args.steps):
        o.load(sample)
        t0 = time.perf_counter()
        moved, outputs = 0, []
        for a in s_actions:
            res = o.run(a)
            outputs.append((a, res))
            moved += res.pods_placed + res.pods_evicted
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
            placed += moved
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    total = sum(times)
    value = placed / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "recorded snapshot" if args.snapshot else "synthetic",
        "config": workload,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": note + "; oracle/kai_oracle.cpp, node sweep fanned out over a worker pool of KAI_REF_THREADS "
                                   "threads (default 16 of %d host cores)" % (os.cpu_count() or 1)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", default="config3-cycle", choices=sorted(synthetic.CONFIG_ACTIONS))
    ap.add_argument("--resident", default="on", choices=["on", "off"],
                    help="on: steps after the first refresh the per-cycle columns of a resident snapshot (structure_epoch); "
                         "off: every step is a full kai_engine_load_snapshot")
    ap.add_argument("--parity", default="auto", choices=["auto", "off"],
                    help="compare the last step's outcome with the CPU oracle (threaded) and exit 1 on a mismatch")
    ap.add_argument("--cpu-baseline", default="auto", choices=["auto", "off"])
    ap.add_argument("--snapshot", default=None,
                    help="time a recorded cluster instead of a synthetic config: a zip of the reference's snapshot "
                         "plugin (kai_scheduler_b200/snapshot_io.py); actions and plugin arguments come from the file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the results of every action of the last timed step to DIR/<action>_<field>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    rank, world, local = dist_env()

    actions = synthetic.CONFIG_ACTIONS[args.config]
    engine_kw = {}
    if args.snapshot:
        from kai_scheduler_b200 import snapshot_io
        snap, _meta, engine_kw, actions = snapshot_io.pack_cluster(snapshot_io.read_snapshot_zip(args.snapshot))
        desc = (f"snapshot {os.path.basename(args.snapshot)}: {snap.n_nodes} nodes, {snap.n_jobs} pod groups, "
                f"{int(snap.task_status.shape[0])} pods; actions {'+'.join(actions)}")
    else:
        snap = synthetic.config_snapshot(args.config)
    if args.snapshot:
        pass
    elif args.config in synthetic.CYCLE_CONFIGS:
        kw = synthetic.CYCLE_CONFIGS[args.config]
        desc = (f"{args.config}: {kw['n_nodes']} nodes x {kw['gpus_per_node']} GPUs, {kw['n_jobs']} pending gangs x {kw['tasks_per_job']} "
                f"1-GPU pods, {kw['n_queues']} leaf queues under {(kw['n_queues'] + 3) // 4} departments (DRF proportion), binpack, "
                f"{kw['running_nodes']} nodes full of running over-quota pods; actions allocate+reclaim (pods = placed + evicted)")
    elif args.config in synthetic.CONFIGS:
        kw = synthetic.CONFIGS[args.config]
        desc = (f"{args.config}: {kw['n_nodes']} nodes x {kw['n_jobs']} jobs x {kw.get('tasks_per_job', 1)} pods, "
                f"{kw.get('n_queues', 4)} leaf queues, binpack, allocate action")
    elif args.config in synthetic.TOPOLOGY_CONFIGS:
        kw = synthetic.TOPOLOGY_CONFIGS[args.config]
        desc = (f"{args.config}: {snap.n_nodes} nodes on 3 topology tiers (spine/leaf/rack), {kw['n_gangs']} gangs of 2-16 node-exclusive "
                f"8-GPU pods ({int(snap.task_status.shape[0])} pods), required level leaf|rack, preferred rack; allocate action")
    else:
        kw = synthetic.RECLAIM_CONFIGS[args.config]
        desc = (f"{args.config}: {snap.n_nodes} nodes x 8 GPUs, {int((snap.task_status == abi.POD_RUNNING).sum())} running 1-GPU pods "
                f"in over-quota queues, {int((snap.task_status == abi.POD_PENDING).sum())} pending reclaimer pods; actions {'+'.join(actions)}"
                " (pods = placed + evicted)")
    workload = {
        "workload": desc,
        "nodes": snap.n_nodes, "pods": int(snap.task_status.shape[0]), "queues": int(snap.queue_parent.shape[0]),
        "parallelism": f"nodes sharded by range over {args.gpus} GPUs, one sequencer replica per rank" if args.gpus > 1 else "1 GPU",
        "sequencer": os.environ.get("KAI_SEQUENCER", "host"), "transport": os.environ.get("KAI_TRANSPORT", "launch"),
        "l2_policy": "the whole snapshot is re-uploaded (H2D) before every timed step; within a step the node tiles "
                     "(76 B x nodes, 3.8 MB at 50 000 nodes) stay L2-resident between the sweep launches by design",
    }
    if args.impl == "reference":
        run_reference(args, snap, workload, actions, engine_kw)
        return

    import torch
    import torch.distributed as dist
    from kai_scheduler_b200.engine import Engine

    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    # N > 1: the node rows are striped by name rank over the GPUs (kai_shard_range(N, world, r)); every rank
    # runs the same deterministic sequencer, one reduced answer line per GPU per sweep is exchanged through a
    # shared host segment.  Total work is fixed => strong scaling.
    eng = Engine(abi.make_config(device=local, shard_rank=rank, shard_count=world, **engine_kw))
    if world > 1:
        handles = [eng.export_peer_handle() if rank == 0 else b""]
        dist.broadcast_object_list(handles, src=0)
        eng.wire_peers(handles * world)
    # steady-state cycle: the cluster's structure (queues, pod groups, requests, node identities) is unchanged between
    # cycles, the per-cycle columns (node idle / releasing / flags, task status / node) are refreshed from host buffers
    # every step (kai_snapshot.structure_epoch, ABI v7).  --resident off reloads the whole snapshot every step.
    snap.structure_epoch = 1 if args.resident == "on" else 0
    c_snap = snap.to_c()
    full_bytes = snap.host_bytes()
    dyn_bytes = int(snap.node_idle.nbytes + snap.node_releasing.nbytes + snap.node_flags.nbytes + snap.task_status.nbytes +
                    snap.task_node.nbytes)
    h2d = dyn_bytes if args.resident == "on" else full_bytes

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(keep=None):
        """returns (device_ms, e2e_s, pods, stats); `keep` (a list) receives a copy of every action's result, made off the
        e2e clock (the engine's result buffers only live until the next run)"""
        t0 = time.perf_counter()
        copy_s = 0.0
        eng.load_c(c_snap, snap.n_res)       # H2D of the whole snapshot + open-session kernels
        dev, moved, launches_, alg_, act_ = 0.0, 0, 0, 0, 0.0
        one_step.evicted, one_step.decisions = 0, 0
        for a in actions:
            r = eng.run(a, copy=False)       # action kernel + D2H of the results
            if keep is not None:
                tc = time.perf_counter()
                keep.append((a, abi.Result.from_c(r, snap.n_res)))
                copy_s += time.perf_counter() - tc
            st = eng.stats()
            dev += st.action_ms
            moved += int(r.pods_placed) + int(r.pods_evicted)
            one_step.evicted += int(r.pods_evicted)
            one_step.decisions += int(st.decisions)
            launches_ = int(st.kernel_launches)
            alg_ += int(st.algorithmic_bytes)
            act_ += st.action_ms
        e2e = time.perf_counter() - t0 - copy_s
        st.kernel_launches, st.algorithmic_bytes, st.action_ms = launches_, alg_, act_
        return st.open_session_ms + dev, e2e, moved, st, r

    for _ in range(max(args.warmup, 3) if args.steps > 0 else 0):
        one_step()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    dev_ms, e2e_s, pods, launches, alg_bytes, act_ms, d2h = 0.0, 0.0, 0, 0, 0, 0.0, 0
    phase_ms = {"upload": 0.0, "open_session": 0.0, "action": 0.0, "download": 0.0}
    t_wall0 = time.perf_counter()
    decisions = evicted_e = 0
    outputs = []
    for i in range(args.steps):
        d, e, p, st, r = one_step(outputs if args.dump_outputs and rank == 0 and i == args.steps - 1 else None)
        decisions, evicted_e = one_step.decisions, one_step.evicted
        dev_ms += d
        e2e_s += e
        pods += p
        launches += int(st.kernel_launches)
        alg_bytes += int(st.algorithmic_bytes)
        act_ms += st.action_ms
        phase_ms["upload"] += st.upload_ms
        phase_ms["open_session"] += st.open_session_ms
        phase_ms["action"] += st.action_ms
        phase_ms["download"] += st.download_ms  # of the last action of the step
        d2h = (r.n_tasks * 8 + r.n_visits * 8 + r.n_queues * 3 * 8 * 4 + r.n_nodes * snap.n_res * 8 * 2 + 24)
    barrier()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    if outputs:
        dump_outputs(args.dump_outputs, outputs)
    last = abi.Result.from_c(r, snap.n_res)  # outcome of the last timed step (copied out of the engine's buffers)
    ranks_agree = True
    if world > 1:  # every rank runs the same sequencer over its node stripe: the bindings must be identical everywhere
        import hashlib
        h = hashlib.sha256(last.task_node.tobytes() + last.task_status.tobytes()).digest()[:8]
        mine = torch.tensor([int.from_bytes(h, "little", signed=True)], dtype=torch.int64, device="cuda")
        lo, hi = mine.clone(), mine.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        ranks_agree = bool(lo.item() == hi.item())

    # max over ranks of the timed quantities
    if world > 1:
        t = torch.tensor([dev_ms, e2e_s, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s, wall = [float(x) for x in t.tolist()]
        pods_all = pods  # every rank places the same pods (replicated sequencer over sharded nodes)
    else:
        pods_all = pods
    # dominant kernel: k_record, one launch per node-table sweep.  Its duration is measured live: back-to-back launches of
    # one list sweep over this rank's node rows, CUDA events on the engine's stream (kai_engine_time_sweeps)
    sweep_ms, merge_ms, sweep_rows = eng.time_sweeps(200) if args.steps > 0 else (0.0, 0.0, 0)
    if rank == 0:
        peak, which = measured_peak_gbs()
        sweep_bytes = sweep_rows * BYTES_PER_NODE
        achieved = sweep_bytes / (sweep_ms * 1e-3) / 1e9 if sweep_ms > 0 else 0.0
        traffic, traffic_src = None, "no ncu --set full capture recorded for this build"
        tp = os.path.join(ROOT, "profiles", "r02_k_record_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
            except Exception:
                pass
        line = {
            "metric": METRIC, "value": pods_all / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "recorded snapshot" if args.snapshot else "synthetic",
            "config": workload,
            "e2e": {"value": pods_all / e2e_s, "unit": UNIT, "ms_per_step": 1e3 * e2e_s / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "snapshot": ("resident: per-cycle columns re-read from host buffers each step (structure_epoch); a full load is "
                                 f"{full_bytes} B" if args.resident == "on" else "full load every step"),
                    # engine-side phases of one step (kai_engine_stats); the rest of e2e is marshalling in the caller
                    "phases_ms": {k: v / max(args.steps, 1) for k, v in phase_ms.items()}},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_record (one node-table sweep per launch: node deltas, fit + score of every row, "
                                                   "per-scanner top-M; 74 % of the GPU time of a step, profiles/r02_launches_bench.csv)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)",
                         "algorithmic_bytes_per_launch": sweep_bytes, "rows_per_launch": sweep_rows,
                         "kernel_us_per_launch": 1e3 * sweep_ms,
                         "how": "200 back-to-back launches of one list sweep timed with CUDA events on the engine's stream, after the timed steps",
                         "merge_kernel_us_per_launch": 1e3 * merge_ms,
                         "sweeps_per_step": decisions, "sweep_share_of_step": (decisions * sweep_ms) / (act_ms / args.steps) if act_ms > 0 else None,
                         # SURVEY.md §8d: the naive path sweeps every node for every pod
                         "naive_equivalent_bytes_per_step": int(snap.n_nodes) * int(pods_all // max(args.steps, 1)) * BYTES_PER_NODE,
                         "traffic": traffic, "traffic_source": traffic_src},
            "clocks": clocks,
            "wall_ms_per_step": 1e3 * wall / args.steps,
        }
        line["decisions_executed"] = int(decisions)
        ok = True
        if args.parity != "off" and args.cpu_baseline != "off":
            # the engine's outcome of the last timed step against the oracle on the same snapshot, once, outside the
            # timed loop; the oracle run doubles as the CPU baseline (bounded: one cycle)
            from oracle_lib import Oracle
            cores = min(os.cpu_count() or 1, int(os.environ.get("KAI_REF_THREADS", "16")))
            o = Oracle(abi.make_config(**engine_kw), threads=cores)
            o.load(snap)
            t0 = time.perf_counter()
            moved, evicted_o = 0, 0
            for a in actions:
                ro = o.run(a)
                moved += ro.pods_placed + ro.pods_evicted
                evicted_o += ro.pods_evicted
            dt = time.perf_counter() - t0
            bindings = bool(np.array_equal(last.task_node, ro.task_node) and np.array_equal(last.task_status, ro.task_status))
            releasing = abi.POD_STATUS_NAMES["Releasing"]
            victims = bool(np.array_equal(np.flatnonzero(last.task_status == releasing), np.flatnonzero(ro.task_status == releasing))
                           and evicted_e == evicted_o)
            share_err = float(np.max(np.abs(last.queue_fair_share - ro.queue_fair_share))) if last.queue_fair_share.size else 0.0
            alloc_err = float(np.max(np.abs(last.queue_allocated - ro.queue_allocated))) if last.queue_allocated.size else 0.0
            if world > 1:  # a rank's result carries its own node stripe only
                own = (snap.node_name_rank % world) == rank
                nodes_eq = bool(np.array_equal(last.node_idle[:, own], ro.node_idle[:, own])
                                and np.array_equal(last.node_releasing[:, own], ro.node_releasing[:, own]))
            else:
                nodes_eq = bool(np.array_equal(last.node_idle, ro.node_idle) and np.array_equal(last.node_releasing, ro.node_releasing))
            line.update({"bindings_match": bindings, "victims_match": victims, "max_share_abs_err": max(share_err, alloc_err),
                         "node_tables_match": nodes_eq, "pods_moved": {"engine": int(pods_all // max(args.steps, 1)), "oracle": int(moved)}})
            ok = bindings and victims and nodes_eq and max(share_err, alloc_err) <= 1e-6 and pods_all // max(args.steps, 1) == moved
            if args.config in synthetic.REFERENCE_PUBLISHED_MS:
                line["reference_published_ms_per_op"] = synthetic.REFERENCE_PUBLISHED_MS[args.config]
            line["cpu_baseline"] = {"value": moved / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"one full {args.config} cycle ({'+'.join(actions)}), oracle/kai_oracle.cpp with a pool of "
                                              f"{cores} threads for the node sweep, {dt:.2f} s (also the parity check of this line)",
                                    "host_cores_available": os.cpu_count()}
        if world > 1:
            line["ranks_agree"] = bool(ranks_agree)
            ok = ok and bool(ranks_agree)
        print(json.dumps(line))
        if not ok:
            print("bench: PARITY MISMATCH against the oracle (see bindings_match / victims_match / node_tables_match)", file=sys.stderr)
    eng.close()
    if world > 1:
        flag = torch.tensor([0 if (rank != 0 or ok) else 1], device="cuda")
        dist.all_reduce(flag)
        dist.destroy_process_group()
        if int(flag.item()):
            sys.exit(1)
    elif rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
