#!/usr/bin/env python
"""bench.py — reconciles/sec of the batched RayCluster reconcile engine (BASELINE.json metric).

A "step" is one full pass of the hot path (spec hash + selector match + replica delta + status roll-up) over one synthetic
snapshot: workload C3 = 10 000 RayClusters x 100 pods per GPU (BASELINE.json configs[2], the headline; fits one GPU).
  value  : clusters decided / device time, inputs already resident in HBM (CUDA events on the engine stream, L2 flushed
           between steps, max over ranks).
  e2e    : same metric through the C ABI with HOST buffers: kr_snapshot_commit (H2D of the whole snapshot from the pinned
           arenas) + kr_reconcile_batch (kernels + D2H of every result record) per step, wall clock, max over ranks.  Two engines
           alternate so the next epoch's upload overlaps this epoch's kernels and download (double-buffered epochs);
           e2e_single_engine is the same loop on one engine (the latency of one epoch).
  roofline / cpu_baseline: see DESIGN.md §5.
`--impl reference` times the CPU arm instead (the oracle port with the reference's namespace-scan List cost structure, all
host threads): the Go controller cannot be built in this image (no Go toolchain), so the arm is a labelled restatement.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "reconciles/sec over 10k RayCluster x 100 pods (batched reconcilePods + status roll-up)"
UNIT = "reconciles/s"


def _ncu_traffic(kernel: str, workload: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed `ncu --set full` capture of
    this same command (profiles/r2_ncu_full_c3.json; C3 only) — None when no capture matches."""
    if workload != "C3":
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_full_c3.json")) as f:
            prof = json.load(f)
    except Exception:
        return None
    for name, d in prof.items():
        if name.startswith(kernel):
            return int((d["dram_rd_MB"] + d["dram_wr_MB"]) * 1e6)
    return None


def _ncu_inst(kernel: str, workload: str):
    """Warp instructions executed by one launch of `kernel` in the committed ncu capture (C3 only)."""
    if workload != "C3":
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_full_c3.json")) as f:
            prof = json.load(f)
    except Exception:
        return None
    for name, d in prof.items():
        if name.startswith(kernel):
            return int(d["inst"])
    return None


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons DURING the GPU legs (B200_PROFILING.md recipe).  Sampled through NVML (same counters as
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*`) every 2 ms from a thread, because the timed
    region lasts tens of milliseconds and nvidia-smi's own loop cannot tick faster than ~100 ms."""

    def __init__(self, device: int):
        self.device = device
        self.samples: list[tuple[int, int]] = []
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.device]) if vis and vis.split(",")[self.device].isdigit() else self.device
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def pump():
                while not self._stop.is_set():
                    try:
                        self.samples.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), int(reasons_fn(h))))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self._t = threading.Thread(target=pump, daemon=True)
            self._t.start()
        except Exception as ex:  # noqa: BLE001
            self.err = str(ex)

    def stop(self) -> dict:
        if self._t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self._stop.set()
        self._t.join(timeout=1)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        seen = set()
        for _, r in self.samples:
            for name, bit in bits.items():
                if r & bit:
                    seen.add(name)
        mhz = [m for m, _ in self.samples]
        # "under load" = samples at or above half the maximum clock (idle gaps between legs sit at the idle clock)
        load = [m for m in mhz if self.max_mhz and m >= 0.5 * self.max_mhz] or mhz
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(seen), "samples": len(mhz)}


def bind_to_gpu_numa_node(local_rank: int) -> str:
    """Pin this rank (and so the engine's pinned arenas, allocated after this call) to the CPUs of its GPU's NUMA node: eight
    ranks uploading 66 MB each out of remote memory were what bent the round-1 e2e scaling curve (GPUs 0-3 / 4-7 sit on
    different nodes).  Best effort: a restricted cgroup keeps what it allows."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa node unknown"
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = sorted(set(cpus) & allowed)
        if use:
            os.sched_setaffinity(0, use)
            return f"node {node}: {len(use)} cpus"
        return f"node {node}: no allowed cpu"
    except Exception as ex:  # noqa: BLE001
        return f"not bound ({type(ex).__name__})"


def build_workload(name: str, rank: int, world: int, strong: bool = False):
    """Global snapshot = world x (workload per GPU), sharded by cluster-UID hash (SURVEY §8(e)); weak scaling — or, with
    --scaling strong, the fixed workload split over the ranks (the literal BASELINE.json metric: one 10k x 100 snapshot at 1/2/4/8)."""
    from kuberay_b200 import synthetic
    params = synthetic.config(name)
    if world > 1 and not strong:
        params.n_clusters *= world
    snap, flags = synthetic.generate(params)
    if world > 1:
        snap = synthetic.shard_by_uid(snap, rank, world)
    return snap, flags, params


class CpuArm:
    """The CPU restatement (oracle port) as the reference arm: built here with -O3 -march=native (SHA-NI SHA-1 where the host
    has it, like Go's crypto/sha1), ONE shared index per snapshot (controller-runtime's informer cache keeps its namespace
    index between reconciles — building it is reported separately, never inside a timed reconcile), one preallocated result set,
    worker threads looping over a bounded sample of clusters."""

    def __init__(self, snap):
        from oracle import oracle
        self.oracle = oracle
        self._tmp = tempfile.TemporaryDirectory(prefix="kr_oracle_native_")  # the tree may be read-only
        self.L = oracle.load(oracle.build_native(self._tmp.name))
        t0 = time.perf_counter()
        self.cx = oracle.Context(snap, self.L)
        self.ctx_build_ms = 1e3 * (time.perf_counter() - t0)
        self.nc = snap.dims["clusters"]
        self.sha = "SHA-NI" if self.L.kr_oracle_sha1_impl() else "portable C"

    def run(self, flags, budget_s: float, threads: int, list_mode=None):
        """-> (reconciles/s, reconciles done, seconds).  A bounded sample: `sample` clusters x `reps` repetitions inside the
        worker threads (thread start-up amortised), sized from a probe so that the leg takes about budget_s."""
        o = self.oracle
        mode = o.NS_SCAN if list_mode is None else list_mode
        probe = min(self.nc, max(threads * 4, 32))
        self.cx.run_range(flags, 0, probe, list_mode=mode, threads=threads)  # first touch
        t0 = time.perf_counter()
        self.cx.run_range(flags, 0, probe, list_mode=mode, threads=threads)
        rate = probe / max(time.perf_counter() - t0, 1e-9)
        sample = int(min(self.nc, max(probe, rate * budget_s)))
        reps = max(1, int(rate * budget_s / sample))
        t0 = time.perf_counter()
        self.cx.run_range(flags, 0, sample, list_mode=mode, threads=threads, reps=reps)
        dt = time.perf_counter() - t0
        return sample * reps / dt, sample * reps, dt

    def close(self):
        self.cx.close()
        self._tmp.cleanup()


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(res, out_dir: str) -> None:
    """--dump-outputs: the records one pass hands its caller, one float array per field as out_dir/<name>.npy (8-bit fields as
    float32, wider ones as float64: both exact).  The two variable-length lists are written in owner order (each RayCluster's
    actions, each group's replica indices), without their arena offsets, which are layout rather than results.  An array with
    no rows is not written (a workload without RayJobs has no jobs.* records).  Above DUMP_CAP_BYTES in all, every array keeps
    the same fixed, seeded sample of the same fraction of its rows."""
    from kuberay_b200.abi import _gather_owned
    arrays = {}
    for rec in ("clusters", "groups", "jobs"):
        a = getattr(res, rec)
        for f in a.dtype.names:
            if f not in ("create_off", "reserved"):
                arrays[f"{rec}.{f}"] = a[f]
    arrays.update(hash=res.hash, wtd_pod_idx=res.wtd_pod_idx, act_cnt=res.act_cnt)
    acts = _gather_owned(res.act_start[:-1], res.act_cnt)
    arrays.update(act_pod_idx=res.act_pod_idx[acts], act_code=res.act_code[acts],
                  create_idx=res.create_idx[_gather_owned(res.groups["create_off"], res.groups["n_create"])])
    arrays = {k: v.astype(np.float32 if v.dtype.itemsize == 1 else np.float64) for k, v in arrays.items() if len(v)}
    frac = DUMP_CAP_BYTES / sum(v.nbytes for v in arrays.values())
    if frac < 1:
        for k, v in arrays.items():
            arrays[k] = v[np.sort(np.random.default_rng(0).choice(len(v), max(1, int(len(v) * frac)), replace=False))]
    arrays["totals"] = np.array([res.n_create_total, res.n_orphans, res.n_actions], dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    snap, flags, params = build_workload(args.workload, 0, 1)
    threads = os.cpu_count() or 1
    arm = CpuArm(snap)
    per_step = max(0.25, min(5.0, 100.0 / max(args.steps + args.warmup, 1)))
    for _ in range(args.warmup):
        arm.run(flags, per_step / 4, threads)
    tot_c, tot_t, sample = 0, 0.0, 0
    for _ in range(args.steps):
        _, sample, dt = arm.run(flags, per_step, threads)
        tot_c += sample; tot_t += dt
    v = tot_c / tot_t
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {params.n_clusters} RayClusters x {params.pods_per_cluster} pods, {params.groups} worker group(s), 100 clusters/namespace",
                   "note": "CPU restatement (C, -O3 -march=native, " + arm.sha + " SHA-1), NOT the Go controller: no Go toolchain in this image; namespace-scan cached List per "
                           "selector as in controller-runtime; the cache's namespace index is built once outside the timed region (" + f"{arm.ctx_build_ms:.1f} ms)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "index_build_ms_not_timed": arm.ctx_build_ms,
                         "sample": f"{sample} reconciles per step over the {snap.dims['clusters']}-cluster snapshot (each = G+4 namespace-scan Lists + SHA-1 of its spec JSON)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    arm.close()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU-baseline sample budget (rank 0, N=1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--allgather", action="store_true", help="also all-gather the per-group delta records over NCCL each step (N>1)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: the workload per GPU (default); strong: the workload once, split over the GPUs")
    ap.add_argument("--no-pack-leg", action="store_true", help="skip the e2e_with_pack leg (tools/pack_bench)")
    ap.add_argument("--no-next-rows", action="store_true", help="skip the f2-f4 extras (tools/f4_bench.py, tools/f3_bench.py --quick)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step of the value leg (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner, ...) goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from kuberay_b200.engine import Engine

    snap, flags, params = build_workload(args.workload, rank, world, strong=args.scaling == "strong")
    # the production configuration in every leg: the shim consumes the records + the compact action list + the replica indices,
    # not the full per-cluster pod lists (kr_flags.fetch_pod_lists = 0; they are a verification / debugging output)
    flags.fetch_pod_lists = 0
    nc_local = snap.dims["clusters"]
    eng = Engine.for_snapshot(snap, device=local_rank)
    eng.set_incremental(False)  # value / e2e / profile legs time the FULL pass; the incremental leg below turns the device-side incremental path on
    views = eng.load(snap)
    alg = eng.algorithmic_bytes()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def l2_flush():
        flush.zero_()
        torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gather = None
    if world > 1 and args.allgather:
        # optional exchange step (SURVEY §8(e)): every rank receives every shard's per-group delta records (32 B each)
        ng = torch.tensor([snap.dims["groups"]], device="cuda")
        dist.all_reduce(ng, op=dist.ReduceOp.MAX)
        cap = int(ng.item()) * 32
        gather = (torch.zeros(cap, dtype=torch.uint8, device="cuda"), torch.empty(cap * world, dtype=torch.uint8, device="cuda"))

    def step_device() -> float:
        eng.reconcile_device_only(flags)
        ms = eng.last_profile()["kernels_ms"]
        if gather is not None:
            eng.group_results_copy(gather[0].data_ptr(), gather[0].numel())
            t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
            t0.record()
            dist.all_gather_into_tensor(gather[1], gather[0])
            t1.record(); torch.cuda.synchronize()
            ms += t0.elapsed_time(t1)
        return ms

    # ---------------- value: device-resident leg
    sampler = ClockSampler(local_rank)  # nvidia-smi needs ~100 ms per sample: it runs across warm-up + every timed leg
    sampler.start()
    for _ in range(args.warmup):
        l2_flush(); step_device()
    barrier()
    wall0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        l2_flush()
        dev_ms += step_device()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - wall0)
    last_step = eng.fetch() if args.dump_outputs and rank == 0 else None
    n_kernels = eng.last_profile()["n_kernels"]
    # the same graph without the hash kernel: the match -> decide chain on its own (what pipeline_roofline is quoted on)
    flags.skip_hash = 1
    for _ in range(3):
        l2_flush(); step_device()
    chain_ms = 0.0
    for _ in range(args.steps):
        l2_flush()
        chain_ms += step_device()
    chain_ms /= args.steps
    flags.skip_hash = 0
    for _ in range(2):
        l2_flush(); step_device()

    # ---------------- e2e: host buffers through the C ABI (commit = H2D, reconcile_batch = kernels + D2H)
    # D2H = every cluster / group / RayJob record, the hashes, the workersToDelete resolutions, the compact action list and the
    # replica indices (kr_flags.fetch_pod_lists = 0, as in the value leg)
    for _ in range(2):
        eng.commit(); eng.reconcile(flags, copy=False)
    barrier()
    e2e_s = 0.0
    h2d = d2h = 0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        eng.commit()
        res = eng.reconcile(flags, copy=False)
        e2e_s += time.perf_counter() - t0
        p = eng.last_profile()
        h2d, d2h = p["h2d_bytes"], p["d2h_bytes"]
    barrier()
    e2e_parts = eng.last_profile()
    # ---------------- e2e, double-buffered epochs: two engines on this GPU used alternately.  kr_snapshot_commit is asynchronous, so
    # epoch k+1 crosses PCIe while kr_reconcile_batch of epoch k (kernels + D2H) runs.  Every step still uploads its whole
    # snapshot from the pinned arenas and downloads its records; the region is timed as one wall-clock interval.
    eng2 = Engine.for_snapshot(snap, device=local_rank)
    eng2.set_incremental(False)
    eng2.load(snap)
    pair = (eng, eng2)
    for i in range(4):
        pair[i & 1].commit(); pair[i & 1].reconcile(flags, copy=False)
    barrier()
    t0 = time.perf_counter()
    pair[0].commit()
    for i in range(args.steps):
        if i + 1 < args.steps:
            pair[(i + 1) & 1].commit()
        res2 = pair[i & 1].reconcile(flags, copy=False)
    pipe_s = time.perf_counter() - t0
    barrier()
    assert (res2.n_actions, res2.n_create_total, res2.n_orphans) == (res.n_actions, res.n_create_total, res.n_orphans)
    eng2.close()
    # additional figure (not the headline): an epoch in which no RayCluster spec changed — the spec-JSON arena stays
    # resident in HBM from the previous commit (kr_snapshot_commit_parts(KR_PART_COLUMNS)); the hash is still recomputed
    from kuberay_b200 import abi as _abi
    cols_s = 0.0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        eng.commit(_abi.PART_COLUMNS)
        eng.reconcile(flags, copy=False)
        cols_s += time.perf_counter() - t0
    cols_bytes = eng.last_profile()["h2d_bytes"]
    barrier()
    # additional figure: an incremental epoch (SURVEY §8(f) rank 1) — informer events touched 1 % of the pods: 0.8 % status
    # updates, 0.1 % deletions (their rows become KR_PP_TOMBSTONE rows), 0.1 % additions (into the rows freed one step earlier).
    # Uploaded: those rows (kr_snapshot_commit_pod_values) + every RayCluster / group / head / RayJob row (KR_PART_OBJECTS).
    # Rewriting the rows in the arenas is host packing and is not timed.
    rng_c = np.random.default_rng(5)
    npods = snap.dims["pods"]
    pod_cols = [name for name, _dt, _m, dim in _abi.COLUMNS if dim == "pods"]
    workers = np.nonzero(((snap.p_packed >> _abi.PP_NODE_TYPE_SHIFT) & 3) != _abi.NT_HEAD)[0].astype(np.uint32)
    n_upd, n_del = max(1, npods * 8 // 1000), max(1, npods // 1000)
    freed = np.zeros(0, dtype=np.uint32)
    inc_s, inc_bytes = 0.0, 0
    eng.set_incremental(True)
    eng.commit(); eng.reconcile(flags, copy=False)  # the full pass that leaves buckets, tables, digests and results resident (untimed)
    inc_changed, inc_kern, inc_host = [], {}, [0.0, 0.0, 0.0]
    for step_i in range(args.steps + 1):  # (+1: one extra epoch, untimed, through the profiled entry point for the kernel breakdown)
        timed = step_i < args.steps
        for c in pod_cols:  # Pods created since the last epoch take the rows freed one step earlier
            views[c][freed] = snap.cols[c][freed]
        gone = rng_c.choice(workers, n_del, replace=False)
        gone = gone[~np.isin(gone, freed)]
        for c in pod_cols:
            views[c][gone] = 0
        views["p_packed"][gone] = np.uint32(_abi.PP_TOMBSTONE)
        upd = rng_c.choice(npods, n_upd, replace=False).astype(np.uint32)
        upd = upd[~np.isin(upd, gone) & ~np.isin(upd, freed)]  # (kr_snapshot_commit_pod_values takes every row once)
        views["p_packed"][upd] ^= np.uint32(1 << 5)  # PodReady True <-> absent
        rows = np.concatenate([freed, gone, upd])
        vals = np.stack([views[c][rows].view(np.uint32) for c in pod_cols], axis=1)  # the handlers have the new rows in hand
        t0 = time.perf_counter()
        eng.commit(_abi.PART_OBJECTS)
        t1 = time.perf_counter()
        eng.commit_pod_values(rows, vals)
        t2 = time.perf_counter()
        if timed:
            res_i = eng.reconcile(flags, copy=False)
            t3 = time.perf_counter()
            inc_s += t3 - t0
            inc_host[0] += t1 - t0; inc_host[1] += t2 - t1; inc_host[2] += t3 - t2
            inc_prof = eng.last_profile()
            inc_bytes = inc_prof["h2d_bytes"]  # both commits of the epoch
            inc_changed.append(int(res_i.n_changed) if res_i.changed_clusters is not None or res_i.n_changed < nc_local else -1)
        else:
            inc_kern = {k: round(v, 5) for k, v in eng.reconcile_profiled(flags)["kernels"]}
        freed = gone
    # second variant: the same number of touched pods, but in 1 % of the RayClusters (a few clusters scaling / restarting — the usual
    # shape of informer traffic) instead of spread uniformly over all of them.  Object rows are not re-uploaded here (none changed).
    for c in pod_cols:
        views[c][:] = snap.cols[c]
    eng.commit(); eng.reconcile(flags, copy=False)
    key = snap.p_ns_id.astype(np.uint64) << np.uint64(32) | snap.p_cluster_name_id.astype(np.uint64)
    ckey = snap.c_ns_id.astype(np.uint64) << np.uint64(32) | snap.c_name_id.astype(np.uint64)
    n_hot = max(1, nc_local // 100)
    loc_s, loc_changed, loc_prof = 0.0, [], {"kernels_ms": 0.0, "d2h_ms": 0.0, "h2d_bytes": 0, "d2h_bytes": 0}
    for step_i in range(args.steps):
        hot = rng_c.choice(nc_local, n_hot, replace=False)
        rows = np.nonzero(np.isin(key, ckey[hot]))[0].astype(np.uint32)
        views["p_packed"][rows] ^= np.uint32(1 << 5)
        vals = np.stack([views[c][rows].view(np.uint32) for c in pod_cols], axis=1)
        t0 = time.perf_counter()
        eng.commit_pod_values(rows, vals)
        res_i = eng.reconcile(flags, copy=False)
        loc_s += time.perf_counter() - t0
        loc_prof = eng.last_profile()
        loc_changed.append(int(res_i.n_changed) if res_i.changed_clusters is not None or res_i.n_changed < nc_local else -1)
        loc_rows = int(rows.size)
    eng.set_incremental(False)
    for c in pod_cols:
        views[c][:] = snap.cols[c]
    barrier()
    # host packing stand-in (not in e2e): copying pre-packed columns into the pinned arenas
    t0 = time.perf_counter()
    eng.fill(views, snap)
    pack_ms = 1e3 * (time.perf_counter() - t0)

    # ---------------- per-kernel times (serialised, event-bracketed), L2 flushed: feeds the roofline block
    ksum: dict[str, float] = {}
    kcnt: dict[str, int] = {}
    nprof = max(3, min(args.steps, 10))
    for _ in range(nprof):
        l2_flush()
        for name, ms in eng.reconcile_profiled(flags)["kernels"]:
            ksum[name] = ksum.get(name, 0.0) + ms
            kcnt[name] = kcnt.get(name, 0) + 1
    kavg = {k: ksum[k] / nprof for k in ksum}  # per-step time of each kernel name (k_scatter etc. launch several times)
    clocks = sampler.stop()

    # ---------------- reduce over ranks
    t = torch.tensor([dev_ms, e2e_s * 1e3, float(nc_local), wall_ms, cols_s * 1e3, inc_s * 1e3, pipe_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, wall_ms, cols_ms, inc_ms, pipe_ms = float(mx[0]), float(mx[1]), float(mx[3]), float(mx[4]), float(mx[5]), float(mx[6])
        nc_total = float(sm[2])
    else:
        e2e_ms, nc_total, cols_ms, inc_ms, pipe_ms = e2e_s * 1e3, float(nc_local), cols_s * 1e3, inc_s * 1e3, pipe_s * 1e3

    if rank == 0:
        peak, peak_src = _peaks()
        value = nc_total * args.steps / (dev_ms / 1e3)
        e2e_v = nc_total * args.steps / (e2e_ms / 1e3)
        dom = max(kavg, key=kavg.get)
        non_hash_ms = sum(v for k, v in kavg.items() if k != "k_hash")
        dom_bytes = alg["hash"] if dom == "k_hash" else alg["match"]
        dom_ms = kavg[dom] if dom == "k_hash" else non_hash_ms
        ach = dom_bytes / (dom_ms / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": dom if dom == "k_hash" else "match->sort->decide pipeline", "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "traffic": _ncu_traffic("k_hash3" if dom == "k_hash" else dom, args.workload), "peak_source": peak_src, "algorithmic_bytes_per_launch": dom_bytes, "avg_ms": dom_ms,
                "note": "k_hash is INT32-issue/latency bound (SHA-1 is a serial chain per message; 80 rounds per 64 B), HBM is its secondary bound" if dom == "k_hash" else ""}
        kernels = {k: round(v, 5) for k, v in sorted(kavg.items(), key=lambda kv: -kv[1])}
        # The hash against the bound that actually holds it (SURVEY §8(d): "report ... and the ALU-bound ceiling"): warp instructions
        # of one launch (committed ncu capture) over its duration, against the ALU pipe's issue rate (one warp instruction per
        # 2 cycles per scheduler; ~all of SHA-1 is LOP3/SHF/IADD3/LEA on that pipe) — over all 4 x SMs schedulers, and over the
        # ceil(n/32) schedulers that have a warp at all when there are fewer one-lane-per-message warps than schedulers.
        hash_alu = None
        h_inst = _ncu_inst("k_hash3", args.workload)
        if h_inst and kavg.get("k_hash") and clocks.get("sm_mhz"):
            n_sched = 4 * torch.cuda.get_device_properties(local_rank).multi_processor_count
            rate = h_inst / (kavg["k_hash"] / 1e3)  # warp instr / s
            per_sched_peak = clocks["sm_mhz"] * 1e6 / 2
            busy = min(n_sched, 2 * ((nc_local + 31) // 32))  # k_hash3: a consumer and a producer warp per 32 messages
            hash_alu = {"warp_instr_per_launch": h_inst, "achieved_gwarp_instr_s": rate / 1e9, "alu_pipe_peak_gwarp_instr_s": n_sched * per_sched_peak / 1e9,
                        "frac_of_chip": rate / (n_sched * per_sched_peak), "schedulers_with_a_warp": busy, "frac_of_busy_schedulers": rate / (busy * per_sched_peak)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {params.n_clusters // world} RayClusters x {params.pods_per_cluster} pods per GPU ({int(nc_total)} clusters total), {params.groups} worker group(s), 100 clusters/namespace, pods in shuffled List order",
                       "sharding": "cluster-UID hash % n_gpus, no data-path collective" + (" + NCCL all-gather of the per-group delta records" if gather is not None else ""),
                       "numa": numa,
                       "l2": "flushed between timed steps (512 MiB memset, excluded)", "timing": "CUDA events on the engine stream per step, max over ranks",
                       "hash": "SHA-1+base32hex of every spec JSON recomputed every step (as the reference does)"},
            "e2e": {"value": nc_total * args.steps / (pipe_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": pipe_ms / args.steps,
                    "mode": "double-buffered epochs: two engines per GPU used alternately through the C ABI; kr_snapshot_commit (async H2D of the whole snapshot) of epoch k+1 "
                            "overlaps kr_reconcile_batch (kernels + D2H of the records) of epoch k; one wall-clock interval around all steps",
                    "host_pack_ms_not_included": pack_ms},
            "e2e_single_engine": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / args.steps,
                                  "h2d_ms": e2e_parts["h2d_ms"], "kernels_ms": e2e_parts["kernels_ms"], "d2h_ms": e2e_parts["d2h_ms"],
                                  "note": "one engine, commit then reconcile_batch back to back: the latency of one epoch"},
            "e2e_spec_json_resident": {"value": nc_total * args.steps / (cols_ms / 1e3), "unit": UNIT, "ms_per_step": cols_ms / args.steps, "h2d_bytes_per_step": int(cols_bytes),
                                       "note": "extra, not the headline: columns re-uploaded every step, spec-JSON arena kept in HBM from the previous epoch (no spec changed)"},
            "e2e_incremental_1pct_pod_churn": {"value": nc_total * args.steps / (inc_ms / 1e3), "unit": UNIT, "ms_per_step": inc_ms / args.steps, "h2d_bytes_per_step": int(inc_bytes), "patch_ms": inc_prof["h2d_ms"], "kernels_ms": inc_prof["kernels_ms"], "d2h_ms": inc_prof["d2h_ms"], "d2h_bytes_per_step": int(inc_prof["d2h_bytes"]),
                                               "device_incremental_steps": sum(1 for x in inc_changed if x >= 0), "changed_clusters_per_step": (int(np.mean([x for x in inc_changed if x >= 0])) if any(x >= 0 for x in inc_changed) else None),
                                               "kernels_ms_profiled_epoch": inc_kern,
                                               "host_call_ms": {"commit_parts_objects": 1e3 * inc_host[0] / args.steps, "commit_pod_values": 1e3 * inc_host[1] / args.steps, "reconcile_batch": 1e3 * inc_host[2] / args.steps},
                                               "note": "extra, not the headline: per step informer events touched 1 % of the pods (0.8 % status updates, 0.1 % deletions -> tombstone rows, 0.1 % additions into freed rows); "
                                                       "uploaded: those rows (kr_snapshot_commit_pod_values, 32 B each) + all RayCluster/group/head/RayJob rows (KR_PART_OBJECTS); the pass is incremental ON THE DEVICE "
                                                       "(kr_incr.cuh: only the touched rows are re-matched, only the RayClusters they belong to re-decided, digests stay resident) and bit-identical to a full pass"},
            "e2e_incremental_1pct_of_clusters": {"value": nc_local * world * args.steps / loc_s if world == 1 else None, "unit": UNIT, "ms_per_step": 1e3 * loc_s / args.steps,
                                                 "touched_pods_per_step": loc_rows, "changed_clusters_per_step": (int(np.mean([x for x in loc_changed if x >= 0])) if any(x >= 0 for x in loc_changed) else None),
                                                 "device_incremental_steps": sum(1 for x in loc_changed if x >= 0), "kernels_ms": loc_prof["kernels_ms"], "d2h_ms": loc_prof["d2h_ms"],
                                                 "h2d_bytes_per_step": int(loc_prof["h2d_bytes"]), "d2h_bytes_per_step": int(loc_prof["d2h_bytes"]),
                                                 "note": "extra, rank 0's own figure: every pod of 1 % of the RayClusters changed (kr_snapshot_commit_pod_values only); the pass re-decides just those clusters and returns just their records"},
            "gpu_launches": int(n_kernels) * args.steps,
            "clocks": clocks,
            "roofline": roof,
            "kernels_ms_per_step": kernels,
            "algorithmic_bytes": alg,
            "pass_roofline": {"achieved": alg["pass"] / (dev_ms / args.steps / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg["pass"] / (dev_ms / args.steps / 1e3) / 1e9 / peak,
                              "note": "all algorithmic bytes of one pass (hash + match/decide) over the graph replay time of the value leg"},
            "pipeline_roofline": {"achieved": alg["match"] / (chain_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg["match"] / (chain_ms / 1e3) / 1e9 / peak,
                                  "kernels": "clear+build_tables+match+decide as one graph replay with the hash kernel skipped (kr_flags.skip_hash), CUDA events, L2 flushed", "avg_ms": chain_ms,
                                  "serialised_sum_ms": non_hash_ms},
            "hash_roofline": {"achieved": alg["hash"] / (kavg.get("k_hash", float("nan")) / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                              "frac": alg["hash"] / (kavg.get("k_hash", float("nan")) / 1e3) / 1e9 / peak, "avg_ms": kavg.get("k_hash")},
            "hash_alu_view": hash_alu,
            "wall_ms_timed_region": wall_ms,
            "results_check": {"n_actions": int(res.n_actions), "n_create_total": int(res.n_create_total), "n_orphans": int(res.n_orphans)},
        }
        if world == 1 and not args.no_pack_leg and args.workload in ("C3", "C2"):
            # e2e THROUGH the native packer (tools/pack_bench.cpp: plain C++ on the C ABI, as the cgo shim would be): per epoch the
            # informer events of a 1 % pod churn + 2 % RayCluster updates are applied natively (interning, row placement),
            # kr_packer_flush uploads what changed, kr_reconcile_batch returns every record
            exe = os.path.join(ROOT, "tools", "pack_bench")
            try:
                out = subprocess.run([exe, str(params.n_clusters), str(params.pods_per_cluster), str(args.steps), "3"], capture_output=True, text=True, timeout=600)
                pb = json.loads(out.stdout.strip().splitlines()[-1])
                epoch = pb["flush_ms"] + pb["reconcile_ms"]
                line["e2e_with_pack"] = {
                    "value": params.n_clusters / (epoch / 1e3), "unit": UNIT, "ms_per_step": epoch, "flush_ms": pb["flush_ms"], "reconcile_ms": pb["reconcile_ms"],
                    "h2d_bytes_per_step": pb["h2d_bytes_per_epoch"], "d2h_bytes_per_step": pb["d2h_bytes_per_epoch"],
                    "events_per_step": pb["events_per_epoch"], "event_handling_ms_per_step": pb["events_ms"],
                    "value_with_event_handling_on_the_critical_path": pb["reconciles_per_s"], "initial_load_pod_upserts_per_s": pb["pod_upserts_per_s"],
                    "note": "native packer (kr_packer_*): the epoch = kr_packer_flush (changed pod rows + small object tables, filled natively from the event "
                            "stream) + kr_reconcile_batch; event handlers run as events arrive (off the epoch's critical path in the shim) — their cost is "
                            "given beside it, and the last figure puts it ON the critical path"}
            except Exception as ex:  # noqa: BLE001
                line["e2e_with_pack"] = {"unavailable": f"{type(ex).__name__}: {ex}"}
        if world == 1 and not args.no_next_rows:
            # the rows either side of the hot path (SURVEY §8 f2-f4), measured by their own tools on this box: the batched RayService hash
            # comparison (GPU SHA-1 behind a host thread pool) and the host-side builders (one thread)
            nxt = {}
            for key, cmd in (("f4_hash_compare", [sys.executable, os.path.join(ROOT, "tools", "f4_bench.py"), "2000"]),
                             ("f2_f3_host_builders", [sys.executable, os.path.join(ROOT, "tools", "f3_bench.py"), "--quick"])):
                try:
                    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
                    nxt[key] = json.loads(out.stdout.strip().splitlines()[-1])
                except Exception as ex:  # noqa: BLE001
                    nxt[key] = {"unavailable": f"{type(ex).__name__}: {ex}"}
            line["next_rows"] = nxt
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            arm = CpuArm(snap)
            v, sample, dt = arm.run(flags, args.cpu_seconds, threads)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "index_build_ms_not_timed": arm.ctx_build_ms,
                                    "sample": f"{sample} reconciles over the {nc_local}-cluster snapshot in {dt:.1f} s (CPU restatement in C, -O3 -march=native, {arm.sha} SHA-1, "
                                              "namespace-scan Lists against one prebuilt cache index; not the Go controller)"}
            # SURVEY §8(d): the same port on one thread (the reference's default ReconcileConcurrency = 1, apis/config/v1alpha1/defaults.go:11)
            # and with pods pre-bucketed by cluster, so the GPU/CPU ratio is not credited to removing the namespace scan alone
            from oracle import oracle as _o
            v1, s1, d1 = arm.run(flags, args.cpu_seconds / 4, 1)
            vi, si, di = arm.run(flags, args.cpu_seconds / 4, threads, list_mode=_o.INDEXED)
            line["cpu_baseline_variants"] = {
                "one_thread_namespace_scan": {"value": v1, "unit": UNIT, "cores": 1, "sample": f"{s1} reconciles in {d1:.1f} s"},
                "all_threads_indexed_lists": {"value": vi, "unit": UNIT, "cores": threads, "sample": f"{si} reconciles in {di:.1f} s (pods pre-bucketed by cluster: no namespace scan)"}}
            arm.close()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
        if last_step is not None:
            dump_outputs(last_step, args.dump_outputs)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
