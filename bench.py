#!/usr/bin/env python
"""bench.py — joined bindings/s of the 3-pattern BGP hot path (BASELINE.json metric) on B200.

A "step" = one pass of the hot path over the resident store = one evaluation of the BASELINE configs[1] query
(`?e foaf:title ?t . ?e ds:annual_salary ?s . ?e foaf:name ?n FILTER(?s > 100000)`) on the employee shape scaled to the size the
metric is quoted on: 16 666 667 employees = 100 000 002 dictionary-encoded triples PER GPU (weak scaling: with N GPUs the global
dataset has N x that, sharded by kb_shard_of(subject, N); a subject-star join needs no exchange, SURVEY.md §8e).

  value      protocol "index-resident": the store and its predicate index (kb_store_build_index = build_all_indexes, built once,
             untimed, as the reference's harnesses do) are resident in HBM; a step is ONE launch of probe_index_kernel through a
             prepared plan (kb_star_join_prepare / kb_plan_submit / kb_plan_collect): K steps run back to back on the device, the host
             stays a ring of launches ahead, every step's row count is read back. Bindings/s of the whole job over all ranks.
  sync_path  the same K steps through the synchronous operator kb_star_join (one host round trip per step): what round 1 quoted
  scan_path  protocol "SURVEY.md §8(d) scan+build+probe": the same K steps with the index switched off — every step scans the
             12-byte/triple store, builds the direct tables and probes
  e2e        same metric through the one-shot C-ABI call with HOST (pinned) buffers: upload of the triple columns, the join,
             and the download of the binding columns are all inside the timed region
  roofline   algorithmic bytes (SURVEY.md §8d formulas) / CUDA-event time of the dominant kernel family, vs the measured HBM peak
  multi_gpu  (N > 1) the legs that exercise the real multi-GPU path, each parity-asserted against closed-form digests of the generator:
             cfg3 = 4-pattern star + GROUP BY ?t COUNT with the cross-rank merge of the partial groups inside the prepared plan
             (peer-memory tables, device-side barrier, one merge kernel over NVLink), the NCCL all-gather + kb_groups_merge variant beside it;
             shuffle_join = a path join on a NON-subject key through the fused peer-memory shuffle (kb_shuffle_push over NVLink);
             strong = the 100 M-triple store of BASELINE configs[2] split over the N GPUs (strong scaling)
  cfg2_10M   (N = 1) the same query on BASELINE configs[1]'s own 10 M-triple store: the size the CPU arm runs
  cpu_baseline / --impl reference: the oracle's restatement of the reference's own algorithm, timed on the host cores

--dump-outputs DIR writes the binding rows the headline's last timed step returned (see write_outputs), so that two builds of the
project can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "joined bindings/sec on 3-pattern BGP over 100M triples"
UNIT = "bindings/s"
DEFAULT_EMPLOYEES = 16_666_667  # x6 = 100 000 002 triples


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--employees", type=int, default=DEFAULT_EMPLOYEES, help="employees per GPU (6 triples each)")
    ap.add_argument("--query", default="cfg2", choices=["cfg2", "star3", "cfg3", "cfg1"])
    ap.add_argument("--cpu-sample", type=int, default=300_000, help="employees in the bounded CPU sample of the GPU arm's own cpu_baseline leg")
    ap.add_argument("--cpu-employees", type=int, default=0, help="--impl reference: employees in the store (default: BASELINE configs[1]'s 10 M triples)")
    ap.add_argument("--ring", type=int, default=4, help="result buffers of the prepared plan = queries in flight + 1")
    ap.add_argument("--config", default="", choices=["", "cfg3", "cfg4", "cfg5"], help="run ONE of the other BASELINE configs instead (one GPU) and print its line")
    ap.add_argument("--no-configs", action="store_true", help="N = 1: skip the cfg3 / cfg4 / cfg5 legs of the default line")
    ap.add_argument("--cfg4-scale", type=float, default=1.0, help="shrink the cfg4 taxonomy (1.0 = 48.9 M instances)")
    ap.add_argument("--no-adversarial", action="store_true", help="N = 1: skip the permuted-dictionary / shuffled-store leg")
    ap.add_argument("--no-multi", action="store_true", help="N > 1: skip the cfg3-merge / shuffle-join / strong-scaling legs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--numa", action="store_true", help="bind the rank to its GPU's NUMA node (helps the e2e leg at 8 ranks: 28 vs 33 ms per "
                    "step; off by default: the one 8-rank run with it on also showed a 3x slower host side of the resident step)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-index", action="store_true", help="headline on the store-scanning path (no predicate-partitioned index)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="write the rows the headline's last timed step returned to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config or args.impl == "reference"):
        ap.error("--dump-outputs writes the headline's result: not with --config or --impl reference")
    return args


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons of the job's GPUs during the timed region (B200_PROFILING.md recipe). Rank 0 samples every GPU of
    the job through NVML in-process; one `nvidia-smi` subprocess per rank every 0.2 s (the first version) initialises NVML for all
    eight GPUs each time and takes driver locks next to the ranks' launches — at 8 ranks that alone tripled the host side of a
    0.1 ms step. Falls back to nvidia-smi when pynvml is missing."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, indices):
        super().__init__(daemon=True)
        self.indices = list(indices)
        self.samples = []  # (sm_mhz, max_mhz, [reasons])
        self.stop_flag = threading.Event()
        self.nvml = None
        try:
            if not self.indices:
                raise RuntimeError("nothing to sample")
            import pynvml

            pynvml.nvmlInit()
            self.handles = [self._handle(pynvml, i) for i in self.indices]
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    @staticmethod
    def _handle(n, cuda_index):
        """NVML handle of CUDA device `cuda_index`: by PCI bus id, so that a CUDA_VISIBLE_DEVICES remapping cannot make the sampler
        watch somebody else's (idle) GPU; by index when torch does not expose the bus id"""
        try:
            import torch

            pr = torch.cuda.get_device_properties(cuda_index)
            bus = "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            return n.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:
            return n.nvmlDeviceGetHandleByIndex(cuda_index)

    def _sample_nvml(self):
        # two queries per GPU and sample (the maximum clock is asked once): every NVML query takes driver locks next to the ranks'
        # stream synchronisations — legs that synchronise every step lost up to ~10 ms to one unlucky sample (0.65 instead of
        # 0.12 ms/step over 20 steps at N = 4), the launch-only headline loop does not notice
        n = self.nvml
        if not hasattr(self, "max_mhz"):
            self.max_mhz = [float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)) for h in self.handles]
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        for h, mx in zip(self.handles, self.max_mhz):
            sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
            mask = int(get(h))
            self.samples.append((float(sm), mx, [k for k, b in self.BITS.items() if mask & b]))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", ",".join(str(i) for i in self.indices)],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            self.samples.append((float(f[0]), float(f[1]), [k for k, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7])
                                                                 if v.lower().startswith("active")]))

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [s[0] for s in self.samples]
        mx = [s[1] for s in self.samples]
        reasons = sorted({r for s in self.samples for r in s[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm),
                "gpus_sampled": len(self.indices), "via": "nvml" if self.nvml else "nvidia-smi"}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_from_profiles(family):
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(family)
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------------------------
CFG2_10M_EMPLOYEES = 1_666_667  # BASELINE configs[1]: "scaled to 10M triples"


def cpu_reference_run(args, steps, warmup, employees, budget_s=120.0):
    """The reference's own algorithm for this query, restated (oracle 'faithful' mode): StarJoin plan (optimizer.rs:84-152) =
    index scan of the first pattern, then per binding one bound index lookup per remaining pattern in the reference's SEQUENTIAL
    mode (engine.rs:621-655: results > 10 000), rows of maps, then the FILTER. Indexes are built before timing, as the reference's
    harnesses do (n_triple_10M.rs:79-95). Result caps (quirk Q1) off. Also times the oracle's columnar OpenMP mode as the strong
    CPU competitor. `employees` = store size of the run; the timed loop stops after `budget_s` seconds."""
    from kolibrie_b200 import datagen
    from tests import oracle_api as O

    E = int(employees)
    d = datagen.employee_dataset(E)
    js, pats, filt = datagen.employee_queries(d)[args.query]
    db = O.Db(d.s, d.p, d.o, d.num_or0, d.is_num)
    t_i = time.perf_counter()
    db.build_index()
    t_i = time.perf_counter() - t_i
    O.set_threads(O.usable_cpus())  # the CPU arm gets every host thread this process may use (affinity mask and cgroup quota)
    cores = O.num_threads()
    rows = 0
    for _ in range(max(1, min(warmup, 1))):
        rows = db.bgp(pats, filt, mode=1).n_rows
    t0 = time.perf_counter()
    n_done = 0
    for _ in range(steps):
        rows = db.bgp(pats, filt, mode=1).n_rows
        n_done += 1
        if time.perf_counter() - t0 > budget_s:  # bounded: never more than ~2 minutes of CPU work
            break
    dt = (time.perf_counter() - t0) / n_done
    t1 = time.perf_counter()
    reps = 0
    while reps < 3:
        rows_c = db.bgp(pats, filt, mode=0).n_rows
        reps += 1
    dt_c = (time.perf_counter() - t1) / reps
    assert rows_c == rows
    return {
        "value": rows / dt, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"{E} employees = {6 * E} triples, query {args.query}, {n_done} timed steps; oracle faithful mode (reference StarJoin, sequential mode as engine.rs:621 "
                  f"dictates above 10 000 rows => 1 worker thread; FILTER stage on {cores} threads); indexes prebuilt ({t_i:.1f} s, untimed)",
        "ms_per_step": dt * 1e3, "rows_per_step": int(rows), "triples": 6 * E,
        "columnar_openmp": {"value": rows / dt_c, "unit": UNIT, "cores": cores, "ms_per_step": dt_c * 1e3,
                            "note": "oracle columnar mode (OpenMP scan + hash joins on u32 columns, no index), same store"},
    }, n_done


def run_reference(args):
    """--impl reference: the CPU arm. Store = BASELINE configs[1]'s own size (10 M triples) — the largest the faithful restatement
    (four nested hash-map indexes, rows of maps: ~0.4 KB of host memory per triple, ~3 s of index build per million triples) runs
    inside the bound; its throughput per row does not depend on the store size (hash lookups per binding)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    E = min(args.cpu_employees or CFG2_10M_EMPLOYEES, args.employees)
    base, n_done = cpu_reference_run(args, args.steps, args.warmup, E)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": n_done, "warmup": 1,
        "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": workload_name(args)},
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "columnar_openmp": base["columnar_openmp"],
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def bind_near_gpu(local):
    """Run this rank (and first-touch the pinned buffers it allocates) on the NUMA node its GPU hangs off: host<->device copies of the
    e2e leg then stay on one socket. Returns (previous affinity, node or None); placement only, no effect on results."""
    try:
        prev = os.sched_getaffinity(0)
    except (AttributeError, OSError):
        return None, None
    try:
        import torch

        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        try:
            import pynvml

            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
            bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()[-12:]
        except Exception:
            return prev, None
    try:
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return prev, None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= prev
        if not cpus:
            return prev, None
        os.sched_setaffinity(0, cpus)
        return prev, node
    except (OSError, ValueError):
        return prev, None


def workload_name(args):
    q = {"cfg2": "3-pattern star BGP (?e title ?t . ?e annual_salary ?s . ?e name ?n) + FILTER(?s > 100000)",
         "star3": "3-pattern star BGP (?e title ?t . ?e annual_salary ?s . ?e name ?n), no FILTER",
         "cfg3": "4-pattern star BGP", "cfg1": "2-pattern BGP (?p workplaceHomepage ?c . ?p name ?n)"}[args.query]
    return f"employee shape, {args.employees} employees = {6 * args.employees} triples per GPU, {q}"


def run_pipelined(plan, steps, keep=None):
    """K prepared queries back to back: submit, and collect the query submitted ring-1 steps earlier. Returns the last row count.
    With a list `keep`, the last query's rows are appended to it (a Relation view of the plan's ring slot)."""
    depth = max(1, plan.ring - 1)
    inflight = []
    rows = 0
    for _ in range(steps):
        inflight.append(plan.submit())
        if len(inflight) > depth:
            rows = plan.collect(inflight.pop(0))
    while inflight:
        if keep is not None and len(inflight) == 1:
            keep.append(plan.collect_rows(inflight.pop(0)))
            rows = keep[-1].n_rows
        else:
            rows = plan.collect(inflight.pop(0))
    return rows


DUMP_BYTES = 60_000_000  # --dump-outputs: at most this many bytes of rows in all (over all ranks)


def write_outputs(out_dir, rel, rank, world):
    """--dump-outputs: the rows `rel` holds, columns in ascending slot order, as DIR/bindings.npy (float64: u32 ids are exact in it),
    sorted lexicographically so that two builds compare row for row whatever order their kernels emit them in. Above the size bound a
    fixed seeded sample of the sorted rows is written; DIR/bindings_index.npy holds the positions of the written rows among the
    sorted ones, DIR/row_count.npy the number of rows. With several ranks every rank writes its own rows, suffixed _rank<r>."""
    from kolibrie_b200 import datagen

    rows = datagen.canonical_rows(rel.to_numpy(sorted(rel.slots)))
    cap = DUMP_BYTES // (8 * (rows.shape[1] + 1) * world)
    idx = np.arange(len(rows))
    if len(rows) > cap:
        idx = np.sort(np.random.default_rng(0).choice(len(rows), size=cap, replace=False))
    sfx = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"bindings{sfx}.npy"), rows[idx].astype(np.float64))
    np.save(os.path.join(out_dir, f"bindings_index{sfx}.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, f"row_count{sfx}.npy"), np.array([len(rows)], dtype=np.float64))


# ---------------------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    from kolibrie_b200 import capi as c
    from kolibrie_b200 import datagen
    from kolibrie_b200 import dist as kd

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: kolibrie_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    prev_affinity, numa_node = bind_near_gpu(local) if args.numa else (None, None)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def reduce_max(*xs):
        if world == 1:
            return [float(x) for x in xs]
        t = torch.tensor([float(x) for x in xs], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def reduce_sum(*xs):
        if world == 1:
            return [int(x) for x in xs]
        t = torch.tensor([int(x) for x in xs], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(v) for v in t]

    K = args.steps
    W = max(args.warmup, 3)
    if args.config:
        if rank == 0:
            ctx1 = c.Context(local)
            peak1, _ = measured_peak()
            res = other_configs(args, ctx1, c, datagen, torch, peak1, which=(args.config,), cpu=not args.no_cpu)[args.config]
            res.update({"metric": res["workload"], "n_gpus": 1, "steps": K, "warmup": W, "higher_is_better": True, "dtype": "u32", "data": "synthetic",
                        "config": {"workload": res["workload"]}, "vs_baseline": None, "gpu_launches": int(ctx1.get_stats()["kernel_launches"])})
            print(json.dumps(res))
            ctx1.close()
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- setup (untimed): this rank's shard of the global dataset, pinned on the host and resident on the device
    t_gen = time.perf_counter()
    d = datagen.employee_shard(args.employees * world, rank, world)
    n = d.n_triples
    hs, hp, ho = (torch.from_numpy(x).pin_memory() for x in (d.s, d.p, d.o))
    t_gen = time.perf_counter() - t_gen
    ctx = c.Context(local)
    ctx.set_sharding(rank, world)
    ctx.dict_numeric_load(d.num_or0, d.is_num)
    ctx.store_load(d.s, d.p, d.o)
    # SparqlDatabase::build_all_indexes, once, outside the timed region (the reference's harnesses do the same, n_triple_10M.rs:91-95).
    # Built twice: the first build also grows the stream-ordered memory pool from empty (cudaMalloc of ~3 GB of slices, tables and
    # scan scratch: hundreds of ms); the second is the steady-state cost of the operation, the one reported.
    n_pred, index_ms_first = (0, 0.0) if args.no_index else ctx.build_index()
    n_pred, index_ms = (0, 0.0) if args.no_index else ctx.build_index()
    js, pats, filt = datagen.employee_queries(d)[args.query]
    plan = None if args.no_index else ctx.prepare_star_join(js, pats, filt, ring=args.ring)

    def step_sync(keep=None):
        r = ctx.star_join(js, pats, filt)
        rows = r.n_rows
        if keep is not None:
            keep.append(r)
        else:
            r.free()
        return rows

    # rank 0 samples all GPUs of the job through warm-up, the timed region and the e2e leg (all of it is load)
    sampler = ClockSampler(range(world) if rank == 0 else [])
    if rank == 0:
        sampler.start()

    # ---- headline: K prepared queries back to back (protocol "index-resident"); without an index: the synchronous scanning step
    def timed(fn, k):
        """fn(k) runs k steps and returns the last row count; wall clock between barrier + synchronize on both sides"""
        ctx.get_stats(reset=True)
        barrier()
        t0 = time.perf_counter()
        rows = fn(k)
        ctx.synchronize()
        t1 = time.perf_counter()  # this rank's K steps are complete on its device; the MAX over ranks of these spans is reported
        barrier()
        return rows, t1 - t0, ctx.get_stats(reset=True)

    def sync_loop(k, keep=None):
        """k synchronous steps; with a list `keep`, the last step's rows are appended to it"""
        return [step_sync(keep if i == k - 1 else None) for i in range(k)][-1]

    head_fn = (lambda k, keep=None: run_pipelined(plan, k, keep)) if plan else sync_loop
    head_fn(W)
    ctx.set_timing(True)
    last = [] if args.dump_outputs else None
    rows_step, dt, st = timed(lambda k: head_fn(k, last), K)
    if last:
        write_outputs(args.dump_outputs, last[0], rank, world)
        last[0].free()
    # the same K steps through the synchronous operator (one host round trip per step)
    sync_leg = None
    def timed_best(fn, k, reps=3):
        """secondary legs that synchronise with the host every step: best of `reps` repetitions of k steps (a clock sample that lands
        inside a 2 ms leg costs it several ms; the headline leg is ONE k-step measurement as the contract says)"""
        best = None
        for _ in range(reps):
            r = timed(fn, k)
            if best is None or r[1] < best[1]:
                best = r
        return best

    if plan:
        sync_loop(3)
        rows_sync, dt_sync, st_sync = timed_best(sync_loop, K)
        assert rows_sync == rows_step
        sync_leg = (dt_sync, st_sync)
    # the same K steps on the store-SCANNING path (index switched off): the K_scan / K_build / K_probe numbers of SURVEY.md §8(d)
    scan_leg = None
    if not args.no_index:
        ctx.set_use_index(False)
        sync_loop(3)
        rows_scan, dts, st_scan = timed_best(sync_loop, K)
        assert rows_scan == rows_step
        scan_leg = (dts, st_scan)
        ctx.set_use_index(True)
    ctx.set_timing(False)

    # ---- multi-GPU legs (N > 1): the cross-rank GROUP BY merge, the non-subject-key join through the peer-memory shuffle, strong scaling
    multi = None
    if world > 1 and not args.no_multi:
        multi = multi_gpu_legs(args, ctx, d, rank, world, local, dev, K, barrier, reduce_max, reduce_sum, c, datagen, kd, torch)

    # ---- e2e: host (pinned) buffers in, host (pinned) buffers out, through kb_star_join_host_into. This call REPLACES the device store
    # (and drops the index and the plan with it), so it runs after every leg that needs them.
    if plan:
        plan.free()
    e2e = None
    if not args.no_e2e:
        n_out_cols = len({t.value for pt in pats for t in (pt.s, pt.p, pt.o) if t.is_var})
        outs = [torch.empty(max(rows_step, 1) + 16, dtype=torch.int32).pin_memory() for _ in range(n_out_cols)]

        def step_e2e():
            return c.star_join_host_raw(ctx, hs.data_ptr(), hp.data_ptr(), ho.data_ptr(), n, js, pats, filt, [o.data_ptr() for o in outs], outs[0].numel())

        for _ in range(max(1, min(args.warmup, 3))):
            rows_e, slots_e = step_e2e()
        barrier()
        t1 = time.perf_counter()
        for _ in range(K):
            rows_e, slots_e = step_e2e()
        ctx.synchronize()
        dt_e = time.perf_counter() - t1
        barrier()
        assert rows_e == rows_step, (rows_e, rows_step)
        e2e = {"dt": dt_e, "h2d": 3 * 4 * n, "d2h": len(slots_e) * 4 * rows_e}
        ctx.get_stats(reset=True)
    if args.no_e2e or K * 0.03 < 1.0:  # keep the GPU under the same load until the clock sampler has a few samples
        t_s = time.perf_counter()
        while time.perf_counter() - t_s < 1.2:
            step_sync() if args.no_e2e else step_e2e()
    sampler.stop_flag.set()
    if rank == 0:
        sampler.join(timeout=2)

    # ---- reduce over ranks: max time, sum of rows
    dt, dte, dt_sync_m, dts_m = reduce_max(dt, e2e["dt"] if e2e else 0.0, sync_leg[0] if sync_leg else 0.0, scan_leg[0] if scan_leg else 0.0)
    rows_all, n_all = reduce_sum(rows_step, n)
    dev_ms_step_max, = reduce_max(st["total_ms"] / K)

    # ---- N = 1: the NON-ideal case — the same 100 M-triple store with its dictionary ids randomly permuted and its triples shuffled
    # (subjects in no order, an employee's terms far apart in id space): direct tables still apply (dense ids, functional predicates)
    adversarial = None
    if world == 1 and not args.no_adversarial and not args.no_index and args.query == "cfg2":
        ps_, pp_, po_, pnum, pisn, pi = datagen.permuted_dataset(d)
        patsP = [c.pattern(c.V(0), c.K(int(pi[pt.p.value])), c.V(v)) for pt, v in zip(pats, (1, 2, 3))]
        ctx.dict_numeric_load(pnum, pisn)
        ctx.store_load(ps_, pp_, po_)
        del ps_, pp_, po_
        ctx.build_index()
        planP = ctx.prepare_star_join(js, patsP, filt, ring=args.ring)
        run_pipelined(planP, W)
        ctx.set_timing(True)
        rowsP, dtP, stP = timed(lambda k: run_pipelined(planP, k), K)
        ctx.set_timing(False)
        assert rowsP == rows_step, (rowsP, rows_step)
        # content parity: the digest of the relabelled closed-form answer
        tk = planP.submit()
        relP = planP.collect_rows(tk)
        keepP = d.salary_of_employee > 100000
        subjP = d.s[0::6][keepP]
        expectP = np.stack([pi[subjP], pi[d.o[1::6][keepP]], pi[d.o[5::6][keepP]], pi[subjP]], axis=1)
        assert datagen.row_checksums(relP.to_numpy([0, 1, 2, 3])) == datagen.row_checksums(expectP), "permuted store: rows differ from the closed form"
        relP.free()
        planP.free()
        ctx.set_use_index(False)
        sync_scanP = lambda k: [ctx.star_join(js, patsP, filt).n_rows for _ in range(k)][-1]
        sync_scanP(2)
        ctx.set_timing(True)
        rowsPs, dtPs, stPs = timed(sync_scanP, max(3, K // 4))
        ctx.set_timing(False)
        ctx.set_use_index(True)
        assert rowsPs == rows_step
        adversarial = {"workload": "the same 100 M-triple store, dictionary ids randomly permuted, triples shuffled; same query",
                       "index_path": {"value": rowsP / (dtP / K), "unit": UNIT, "ms_per_step": dtP / K * 1e3, "probe_ms": stP["probe_ms"] / K},
                       "scan_path": {"value": rowsPs / (dtPs / max(3, K // 4)), "unit": UNIT, "ms_per_step": dtPs / max(3, K // 4) * 1e3,
                                     "scan_ms": (stPs["scan_ms"] + stPs["build_ms"]) / max(3, K // 4), "probe_ms": stPs["probe_ms"] / max(3, K // 4)},
                       "parity": "digest of the result == relabelled closed form"}
    # ---- N = 1: BASELINE configs[1]'s own size (10 M triples) through the same prepared path — the size the CPU arm runs
    cfg2_10m = None
    if world == 1 and not args.no_cpu and args.employees > CFG2_10M_EMPLOYEES and args.query == "cfg2":
        d10 = datagen.employee_dataset(CFG2_10M_EMPLOYEES)
        ctx.dict_numeric_load(d10.num_or0, d10.is_num)
        ctx.store_load(d10.s, d10.p, d10.o)
        ctx.build_index()
        js10, pats10, filt10 = datagen.employee_queries(d10)["cfg2"]
        p10 = ctx.prepare_star_join(js10, pats10, filt10, ring=args.ring)
        run_pipelined(p10, W)
        rows10, dt10, st10 = timed(lambda k: run_pipelined(p10, k), K)
        p10.free()
        h10 = [torch.from_numpy(x).pin_memory() for x in (d10.s, d10.p, d10.o)]
        o10 = [torch.empty(rows10 + 16, dtype=torch.int32).pin_memory() for _ in range(4)]
        e10 = lambda: c.star_join_host_raw(ctx, h10[0].data_ptr(), h10[1].data_ptr(), h10[2].data_ptr(), d10.n_triples, js10, pats10, filt10, [o.data_ptr() for o in o10], o10[0].numel())
        e10()
        ctx.synchronize()
        t1 = time.perf_counter()
        for _ in range(K):
            re10, _ = e10()
        ctx.synchronize()
        dte10 = (time.perf_counter() - t1) / K
        assert re10 == rows10
        cfg2_10m = {"workload": f"BASELINE configs[1]: {CFG2_10M_EMPLOYEES} employees = {d10.n_triples} triples, same query, prepared index path",
                    "value": rows10 / (dt10 / K), "unit": UNIT, "ms_per_step": dt10 / K * 1e3, "bindings_per_step": int(rows10),
                    "e2e": {"value": rows10 / dte10, "unit": UNIT, "ms_per_step": dte10 * 1e3, "h2d_bytes_per_step": 12 * d10.n_triples, "d2h_bytes_per_step": 16 * int(rows10)}}
    configs = None
    if world == 1 and not args.no_configs and args.query == "cfg2":
        configs = other_configs(args, ctx, c, datagen, torch, measured_peak()[0], cpu=not args.no_cpu, d_full=d)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_step = dt / K * 1e3
    value = rows_all / (dt / K)
    peak, peak_src = measured_peak()

    # ---- roofline of each kernel family (rank 0's launches): algorithmic bytes per SURVEY.md §8(d)
    E_loc = d.n_employees
    n_pat = len(pats)
    m_rows = []
    for k in range(n_pat):
        filtered = bool(filt) and k == 1  # cfg2: the salary pattern carries the FILTER
        m_rows.append(rows_step if filtered else E_loc)
    probe_k = max((k for k in range(n_pat) if not (bool(filt) and k == 1)), key=lambda k: m_rows[k])
    builds = [k for k in range(n_pat) if k != probe_k]
    T = len(builds)
    b_probe = 4 * 2 * m_rows[probe_k] + 8 * T * m_rows[probe_k] + 4 * (n_pat + 1) * rows_step
    kernel_names = {"scan": "kb::scan_kernel<K>", "scan+build": "kb::scan_kernel<K> (fused scan + direct-table build) + table memsets",
                    "build": "kb::build_pairs_filtered_kernel / build_direct_pairs_kernel + table memsets", "probe": "kb::probe_fast_kernel<T>"}

    def families(stx, indexed):
        if indexed:
            # build sides are read from their predicate slices: 8 B per slice row in, (filtered) rows into the table: 8*M_slice + 8*M_b
            b_build = sum(8 * E_loc + 8 * m_rows[k] for k in builds)
            fam = {"probe": {"alg_bytes": b_probe, "ms": stx["probe_ms"] / K, "launches_per_step": stx["probe_launches"] / K,
                             "note": "probe rows = one predicate slice of the index (zero copy); lookups go to direct tables"}}
            if stx["build_launches"] > 0:  # a pattern without a persistent table in the index is built per query
                fam["build"] = {"alg_bytes": b_build, "ms": stx["build_ms"] / K, "launches_per_step": stx["build_launches"] / K,
                                "note": "index path: K_build reads the predicate slice (8 B/row) and evaluates the pushed-down FILTER itself"}
            else:
                fam["probe"]["note"] += "; all build sides are persistent per-predicate tables of the index (the reference's spo[s][P] lookup): no per-query build"
        else:
            b_scan = 12 * n + sum(4 * 2 * m for m in m_rows)
            b_build = sum(16 * m_rows[k] for k in builds)
            if stx.get("fused_scan_builds", 0) > 0:
                fam = {"scan+build": {"alg_bytes": b_scan + b_build, "ms": (stx["scan_ms"] + stx["build_ms"]) / K, "launches_per_step": stx["scan_launches"] / K,
                                      "note": "one kernel does K_scan and K_build of SURVEY.md 8(d): build-side patterns insert into their direct tables"},
                       "probe": {"alg_bytes": b_probe, "ms": stx["probe_ms"] / K, "launches_per_step": stx["probe_launches"] / K}}
            else:
                fam = {"scan": {"alg_bytes": b_scan, "ms": stx["scan_ms"] / K, "launches_per_step": stx["scan_launches"] / K},
                       "build": {"alg_bytes": b_build, "ms": stx["build_ms"] / K, "launches_per_step": stx["build_launches"] / K},
                       "probe": {"alg_bytes": b_probe, "ms": stx["probe_ms"] / K, "launches_per_step": stx["probe_launches"] / K}}
        for v in fam.values():
            v["achieved_gbs"] = v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else None
            v["frac"] = v["achieved_gbs"] / peak if v["achieved_gbs"] else None
        return fam

    def roof(fam, stx):
        dom = max(fam, key=lambda k: fam[k]["ms"])
        name = "kb::probe_index_kernel<T,PRE>" if (dom == "probe" and stx.get("index_joins", 0) and stx["build_launches"] == 0) else kernel_names[dom]
        return {"bound": "hbm", "kernel": name, "achieved": fam[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": fam[dom]["frac"],
                "traffic": traffic_from_profiles(dom.split("+")[0] + ("_index" if stx.get("index_joins", 0) else "")), "peak_source": peak_src,
                "alg_bytes_per_launch": fam[dom]["alg_bytes"], "ms_per_launch": fam[dom]["ms"], "families": fam, "device_ms_per_step": stx["total_ms"] / K}

    indexed = st.get("index_joins", 0) > 0
    roofline = roof(families(st, indexed), st)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "protocol": ("index-resident: store + predicate index resident in HBM, one probe_index_kernel launch per step through a prepared plan (ring of %d), "
                     "K steps back to back, every step's row count collected" % args.ring) if plan is not None or indexed else "SURVEY.md 8(d): scan + build + probe every step",
        "config": {"workload": workload_name(args)},
        "details": {"triples_total": n_all, "bindings_per_step": rows_all, "sharding": "kb_shard_of(subject) = (id >> 10) % n_gpus (block-cyclic on dense ids), no data-path collective",
                    "l2": "inputs per step (index path: 0.4 GB of predicate slices + 0.13 GB of tables; scan path: 1.2 GB of triple columns) exceed the 126 MB L2; no explicit flush",
                    "store": ("predicate-partitioned index built ONCE at load by kb_store_build_index (= SparqlDatabase::build_all_indexes), %d predicates, %.1f ms "
                              "(first build in a fresh process, which also grows the CUDA memory pool from empty: %.1f ms), outside the timed region"
                              % (n_pred, index_ms, index_ms_first)) if not args.no_index else "unindexed: every step scans the store",
                    "datagen_s": round(t_gen, 1), "host_numa_node": numa_node,
                    "timing": "per rank: wall clock from the opening barrier+synchronize to the synchronize that ends its K steps (a closing barrier follows); MAX over ranks",
                    "host_overhead_us_per_step": (ms_step - dev_ms_step_max) * 1e3, "device_ms_per_step_max_over_ranks": dev_ms_step_max},
        "roofline": roofline,
        "gpu_launches": int(st["kernel_launches"]),
        "clocks": sampler.summary(),
    }
    if sync_leg:
        line["sync_path"] = {"value": rows_all / (dt_sync_m / K), "unit": UNIT, "ms_per_step": dt_sync_m / K * 1e3, "gpu_launches": int(sync_leg[1]["kernel_launches"]),
                             "device_ms_per_step": sync_leg[1]["total_ms"] / K,
                             "note": "same K steps through the synchronous kb_star_join (result allocation + stream synchronisation every step); best of 3 repetitions of K steps"}
    if scan_leg:
        st_scan = scan_leg[1]
        line["scan_path"] = {"value": rows_all / (dts_m / K), "unit": UNIT, "ms_per_step": dts_m / K * 1e3, "gpu_launches": int(st_scan["kernel_launches"]),
                             "protocol": "SURVEY.md 8(d): R / (t_scan + t_build + t_probe), every step scans the 12-byte/triple store; best of 3 repetitions of K steps",
                             "roofline": roof(families(st_scan, False), st_scan)}
    if multi:
        line["multi_gpu"] = multi
    if cfg2_10m:
        line["cfg2_10M"] = cfg2_10m
    if configs:
        line["other_configs"] = configs
    if adversarial:
        b_tab = 4 * 3 * m_rows[probe_k] * 1 + 8 * m_rows[probe_k] + 4 * (n_pat + 1) * rows_step  # table mode: 3 tables x 4 B + 8 B typed value per slot, output
        adversarial["index_path"]["frac_of_peak"] = (b_probe / (adversarial["index_path"]["probe_ms"] * 1e-3) / 1e9) / peak
        adversarial["index_path"]["note"] = "fraction of the measured HBM peak with the SAME algorithmic bytes as the headline probe (B_probe = %d); table-mode bytes %d" % (b_probe, b_tab)
        line["adversarial"] = adversarial
    if e2e:
        line["e2e"] = {"value": rows_all / (dte / K), "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                       "ms_per_step": dte / K * 1e3, "api": "kb_star_join_host_into (pinned host columns in, pinned host binding columns out; chunked upload overlapped with the scan)"}
    if world == 1 and not args.no_cpu:
        if prev_affinity:
            os.sched_setaffinity(0, prev_affinity)  # the CPU arm gets every host thread back
        base, _ = cpu_reference_run(args, steps=3, warmup=1, employees=min(args.cpu_sample, args.employees), budget_s=20.0)
        line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_columnar_openmp"] = base["columnar_openmp"]
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def other_configs(args, ctx, c, datagen, torch, peak, which=("cfg3", "cfg4", "cfg5"), cpu=True, d_full=None):
    """The other BASELINE.json configs on one GPU, each with its roofline and a bounded CPU baseline (oracle). Returns {name: dict}."""
    import numpy as np
    from tests import oracle_api as O

    out = {}
    K = args.steps

    def frac(bytes_, ms):
        return (bytes_ / (ms * 1e-3) / 1e9) / peak if ms > 0 else None

    if "cfg3" in which:
        E = args.employees
        d = d_full if d_full is not None else datagen.employee_dataset(E)
        ctx.dict_numeric_load(d.num_or0, d.is_num)
        ctx.store_load(d.s, d.p, d.o)
        ctx.build_index()
        js, pats, _ = datagen.employee_queries(d)["cfg3"]
        plan = ctx.prepare_star_join(js, pats, None, group_slots=[1], aggs=[(c.AGG_COUNT, 0)], ring=args.ring)
        def run(k):
            inflight, res = [], None
            for _ in range(k):
                inflight.append(plan.submit())
                if len(inflight) >= plan.ring:
                    res = plan.collect_groups(inflight.pop(0))
            while inflight:
                res = plan.collect_groups(inflight.pop(0))
            return res
        run(5)
        ctx.get_stats(reset=True); ctx.set_timing(True); ctx.synchronize()
        t0 = time.perf_counter()
        g, rows = run(K)
        ctx.synchronize()
        dt = (time.perf_counter() - t0) / K
        st = ctx.get_stats(reset=True); ctx.set_timing(False)
        plan.free()
        counts = {int(k): int(n_) for k, n_ in zip(g["keys"][0], g["counts"])}
        want = {int(d.title_id_by_value[t]): int((d.title_of_employee == t).sum()) for t in range(3)}
        assert rows == E and counts == want, "cfg3 groups differ from the closed form"
        alg = 4 * E + 8 * E + 4 * 3 * E + 16 * 3  # table-mode probe: 4 B value + (no filter) + 3 lookups x 4 B per subject; 3 groups out
        line = {"workload": f"BASELINE configs[2] on one GPU: {6 * E} triples, 4-pattern star + GROUP BY ?t COUNT (join + grouping in ONE kernel, no joined row written)",
                "value": rows / dt, "unit": "bindings/s", "ms_per_step": dt * 1e3, "device_ms_per_step": st["total_ms"] / K,
                "roofline": {"bound": "hbm", "kernel": "kb::probe_index_kernel<3,0,AGG,TAB>", "alg_bytes_per_launch": alg, "ms_per_launch": st["probe_ms"] / K,
                             "frac": frac(alg, st["probe_ms"] / K), "peak": peak, "unit": "GB/s"},
                "parity": "groups == closed-form title histogram"}
        if cpu:
            Ec = min(args.cpu_sample, E)
            dc = datagen.employee_dataset(Ec)
            odb = O.Db(dc.s, dc.p, dc.o, dc.num_or0, dc.is_num)
            _, cp, _ = datagen.employee_queries(dc)["cfg3"]
            O.set_threads(O.usable_cpus())
            t1 = time.perf_counter()
            rel = odb.bgp(cp)
            odb.group(rel, [1], [(c.AGG_COUNT, 0)])
            dtc = time.perf_counter() - t1
            line["cpu_baseline"] = {"value": rel.n_rows / dtc, "unit": "bindings/s", "cores": O.num_threads(), "kind": "port",
                                    "sample": f"{Ec} employees, oracle columnar mode (OpenMP) join + group"}
        out["cfg3"] = line

    if "cfg4" in which:
        n_inst = int(48_888_890 * args.cfg4_scale)
        t = datagen.taxonomy_dataset(10, 6, n_inst, seed=43)
        rules = datagen.taxonomy_rules(t)
        times, st = [], None
        for rep in range(6):  # one warm-up closure, then five timed ones (median), each on a freshly loaded store
            ctx.store_load(t.s, t.p, t.o)
            ctx.synchronize()
            t0 = time.perf_counter()
            rel, st = ctx.datalog_fixpoint(rules)
            ctx.synchronize()
            if rep:
                times.append(time.perf_counter() - t0)
            rel.free()
        dt = sorted(times)[len(times) // 2]
        inferred, deriv = int(st.inferred), int(st.derivations)
        lvl = np.repeat(np.arange(7), [10 ** k for k in range(7)])
        cls = t.o[t.p == t.ids["rdf:type"]].astype(np.int64) - 2
        assert inferred == int(lvl[cls].sum()) + sum(10 ** k * (k - 1) for k in range(2, 7)), "cfg4 closure differs from the closed form"
        alg = 12 * deriv + 12 * inferred
        line = {"workload": f"BASELINE configs[3] shape on one GPU: Datalog R1 (subClassOf transitive) + R2 (type propagation) over {len(t.s)} triples "
                            "(10-ary class tree of depth 6 + rdf:type facts), semi-naive fixpoint",
                "value": inferred / dt, "unit": "inferred facts/s", "seconds": dt, "seconds_all": [round(x, 4) for x in times], "inferred": inferred,
                "derivations": deriv, "rounds": int(st.rounds), "device_ms": float(st.device_ms),
                "roofline": {"bound": "hbm", "kernel": "kb::derive_partition_kernel + kb::derive_probe_kernel (radix-partitioned candidate dedup) and the joins feeding them",
                             "alg_bytes_per_closure": alg, "frac": frac(alg, dt * 1e3), "peak": peak, "unit": "GB/s",
                             "note": "SURVEY 8(d): 12 B per derived candidate + 12 B per new fact, over the WHOLE closure time (joins, set rebuilds and appends included)"},
                "parity": "inferred == closed-form count; per-round counts checked against the oracle in tests/test_gpu_datalog.py"}
        # the textbook OLD/delta scheme beside it (KB_SEMI_NAIVE_OLD_DELTA): same facts, rounds and per-round counts, fewer candidates
        times2, st2 = [], None
        for rep in range(3):
            ctx.store_load(t.s, t.p, t.o)
            ctx.synchronize()
            t0 = time.perf_counter()
            rel, st2 = ctx.datalog_fixpoint(rules, c.SEMI_NAIVE_OLD_DELTA)
            ctx.synchronize()
            if rep:
                times2.append(time.perf_counter() - t0)
            rel.free()
        assert int(st2.inferred) == inferred and int(st2.rounds) == int(st.rounds), "old/delta scheme: closure differs"
        assert [int(x) for x in st2.round_new[:st.rounds]] == [int(x) for x in st.round_new[:st.rounds]], "old/delta scheme: per-round counts differ"
        line["old_delta_scheme"] = {"seconds": min(times2), "seconds_all": [round(x, 4) for x in times2], "value": inferred / min(times2), "unit": "inferred facts/s",
                                    "derivations": int(st2.derivations),
                                    "note": "opt-in strategy: premises before the delta premise read only OLD facts; the headline value above keeps the reference's delta-against-ALL scheme (derivation count == oracle's)"}
        if cpu:
            ts = datagen.taxonomy_dataset(10, 4, 200_000, seed=43)
            t1 = time.perf_counter()
            w = O.Db(ts.s, ts.p, ts.o).fixpoint(datagen.taxonomy_rules(ts))
            dtc = time.perf_counter() - t1
            line["cpu_baseline"] = {"value": len(w["facts"]) / dtc, "unit": "inferred facts/s", "cores": 1, "kind": "port",
                                    "sample": "10-ary tree depth 4 + 200 000 type facts, oracle restatement of the reference's semi-naive strategy"}
        out["cfg4"] = line

    if "cfg5" in which:
        per = 1_000_002
        n_slides, width = 16, 10
        d = datagen.employee_dataset(per * n_slides // 6)
        ctx.dict_numeric_load(d.num_or0, d.is_num)
        js, pats, filt = datagen.employee_queries(d)["cfg2"]
        hs, hp, ho = (torch.from_numpy(x).pin_memory().numpy() for x in (d.s, d.p, d.o))
        ctx.store_clear()
        live, rows_tot, t_acc, t_h2d, timed_n = [], 0, 0.0, 0.0, 0
        ctx.get_stats(reset=True)
        for t in range(n_slides):
            lo, hi = t * per, (t + 1) * per
            ctx.synchronize()
            t0 = time.perf_counter()
            if len(live) == width:
                ctx.store_evict(live.pop(0))
            ctx.store_append(hs[lo:hi], hp[lo:hi], ho[lo:hi], tag=100 + t)
            live.append(100 + t)
            if t == 0:
                ctx.build_index()  # once; every later slide MAINTAINS it (one chunk per segment, tables updated in place)
            n0 = ctx.get_stats()["index_joins"]
            r = ctx.star_join(js, pats, filt)
            rows = r.n_rows
            r.free()
            ctx.synchronize()
            assert ctx.get_stats()["index_joins"] == n0 + 1, "the slide left the index path"
            if t >= width:  # steady state: a full window, one eviction + one append per slide
                t_acc += time.perf_counter() - t0
                rows_tot += rows
                timed_n += 1
                a = (t - width + 1) * per // 6
                b = hi // 6
                assert rows == int((d.salary_of_employee[a:b] > 100000).sum()), "cfg5 rows differ from the closed form"
        ms_host = t_acc / timed_n * 1e3
        rows_host, n_host = rows_tot, timed_n
        # the same slides with the new slide already in HBM (kb_store_append_device: what a producer kernel or the receive side of
        # kb_shuffle_push hands over): the per-slide cost WITHOUT the 12 MB host-to-device copy
        ds, dp, do = (torch.from_numpy(x).cuda() for x in (d.s, d.p, d.o))
        ctx.store_clear()
        live, t_dev, n_dev = [], 0.0, 0
        for t in range(n_slides):
            lo, hi = t * per, (t + 1) * per
            ctx.synchronize()
            t0 = time.perf_counter()
            if len(live) == width:
                ctx.store_evict(live.pop(0))
            ctx.store_append_device(ds.data_ptr() + 4 * lo, dp.data_ptr() + 4 * lo, do.data_ptr() + 4 * lo, per, 100 + t)
            live.append(100 + t)
            if t == 0:
                ctx.build_index()
            n0 = ctx.get_stats()["index_joins"]
            r = ctx.star_join(js, pats, filt)
            rows = r.n_rows
            r.free()
            ctx.synchronize()
            assert ctx.get_stats()["index_joins"] == n0 + 1, "the slide left the index path"
            if t >= width:
                t_dev += time.perf_counter() - t0
                n_dev += 1
                assert rows == int((d.salary_of_employee[(t - width + 1) * per // 6:hi // 6] > 100000).sum()), "cfg5 rows differ from the closed form"
        # window maintenance alone (evict + append, no query), device-resident slide
        t_m = []
        for t in range(3):
            ctx.synchronize()
            t0 = time.perf_counter()
            ctx.store_evict(live.pop(0))
            ctx.store_append_device(ds.data_ptr(), dp.data_ptr(), do.data_ptr(), per, 900 + t)
            ctx.synchronize()
            t_m.append(time.perf_counter() - t0)
            live.append(900 + t)
        del ds, dp, do
        st5 = ctx.get_stats()
        line = {"workload": f"BASELINE configs[4]: RSP window of {width} slides x {per} triples (10 s of a 1 M triples/s stream), per slide: evict the oldest slide, "
                            "append the new one (H2D of 12 MB), index maintained in place, 3-pattern BGP + FILTER through the index path",
                "value": rows_host / t_acc, "unit": "bindings/s", "ms_per_slide": ms_host, "slides_per_s": n_host / t_acc,
                "ms_per_slide_excl_h2d": t_dev / n_dev * 1e3, "ms_window_maintenance_excl_h2d": min(t_m) * 1e3,
                "triples_per_s_sustained": per * n_host / t_acc,
                "roofline": {"bound": "pcie", "note": "a slide moves 12 MB host->device (12 B per triple) and touches ~1/10 of the window on the device: the slide is bound by "
                             "the copy and by host round trips, not by HBM. Maintenance per slide: 1 clear launch (evicted keys leave the tables), "
                             "1 profile pass + 1 split pass over the new segment (2 read-backs), then the query's one probe launch"},
                "parity": "rows per slide == closed form; every slide stayed on the index path"}
        if cpu:
            w0, w1 = 0, width * per
            odb = O.Db(d.s[w0:w1], d.p[w0:w1], d.o[w0:w1], d.num_or0, d.is_num)
            t1 = time.perf_counter()
            n_c = odb.bgp(pats, filt).n_rows
            dtc = time.perf_counter() - t1
            line["cpu_baseline"] = {"value": n_c / dtc, "unit": "bindings/s", "cores": O.num_threads(), "kind": "port",
                                    "sample": "one full window (10 M triples), oracle columnar mode (OpenMP), query only (no window maintenance)"}
        out["cfg5"] = line
    return out


def multi_gpu_legs(args, ctx, d, rank, world, local, dev, K, barrier, reduce_max, reduce_sum, c, datagen, kd, torch):
    """The legs that exercise the multi-GPU path proper. Every result is asserted against closed forms of the generator."""
    import numpy as np

    out = {}
    E_glob = args.employees * world
    # ---- cfg3: 4-pattern star + GROUP BY ?t COUNT, local fused join+group per rank, partial groups all-gathered (NCCL) and folded by
    # kb_groups_merge on every rank. Pipelined: query i+1 is on the device while the partials of query i are exchanged and merged.
    js3, pats3, _ = datagen.employee_queries(d)["cfg3"]
    idx = datagen.employee_indices_of_shard(d, rank, world)
    titles = datagen.employee_title_ids(d, idx)
    tids = [int(x) for x in d.title_id_by_value]
    want = reduce_sum(*[int((titles == t).sum()) for t in tids])  # closed form: the global title histogram

    def check_groups(groups):
        got = {int(k): int(n_) for k, n_ in zip(groups["keys"][0], groups["counts"])}
        assert got == {t: w for t, w in zip(tids, want) if w}, (got, want)
        return len(got)

    # (a) the merge INSIDE the plan: partial tables in peer-mapped memory, device-side barrier, one merge kernel reading the peers'
    #     tables over NVLink — a submit is asynchronous end to end, K queries run back to back
    plan_p = kd.attach_group_plan(ctx.prepare_star_join(js3, pats3, None, group_slots=[1], aggs=[(c.AGG_COUNT, 0)], ring=max(args.ring, 2)))

    def cfg3_peer_steps(k):
        depth, inflight, out_ = max(1, plan_p.ring - 1), [], (None, 0)
        for _ in range(k):
            inflight.append(plan_p.submit())
            if len(inflight) > depth:
                out_ = plan_p.collect_groups(inflight.pop(0))
        while inflight:
            out_ = plan_p.collect_groups(inflight.pop(0))
        return out_

    cfg3_peer_steps(5)
    ctx.get_stats(reset=True)
    ctx.set_timing(True)
    barrier()
    t0 = time.perf_counter()
    g_p, rows_p = cfg3_peer_steps(K)
    ctx.synchronize()
    dt_p = time.perf_counter() - t0
    barrier()
    st_p = ctx.get_stats(reset=True)
    ctx.set_timing(False)
    plan_p.free()
    n_groups = check_groups(g_p)
    rows_p_all, = reduce_sum(rows_p)
    assert rows_p_all == E_glob == sum(want)
    dt_pm, dev_p, dev_pg = reduce_max(dt_p, st_p["probe_ms"] / K, st_p["group_ms"] / K)
    table_bytes = 4096 * 92 + 16
    out["cfg3_group_by_merge"] = {
        "workload": f"BASELINE configs[2]: {6 * args.employees} triples per GPU x {world} GPUs, 4-pattern star + GROUP BY ?t COUNT, global groups on every rank",
        "value": rows_p_all / (dt_pm / K), "unit": "bindings/s", "ms_per_step": dt_pm / K * 1e3, "device_ms_per_step_join_group": dev_p,
        "device_ms_per_step_barrier_init_merge": dev_pg, "groups": n_groups,
        "exchange": "fused: per-rank join+group kernel -> device-side barrier over peer-memory flags -> one merge kernel per rank reading the %d partial tables over NVLink "
                    "(P2P loads, %d bytes each); no NCCL call and no host round trip per query" % (world, table_bytes),
        "nvlink_bytes_read_per_rank_per_step": (world - 1) * table_bytes, "parity": "groups == closed-form global title histogram on every rank"}
    # (b) the portable variant: partial groups all-gathered over NCCL, folded by kb_groups_merge
    plan3 = ctx.prepare_star_join(js3, pats3, None, group_slots=[1], aggs=[(c.AGG_COUNT, 0)], ring=args.ring)

    def cfg3_steps(k):
        prev, merged, rows = None, None, 0
        for _ in range(k):
            t = plan3.submit()
            if prev is not None:
                packed, rows = plan3.collect_groups(prev, packed=True)
                merged = ctx.groups_merge(kd.allgather_groups(packed, dev))
            prev = t
        packed, rows = plan3.collect_groups(prev, packed=True)
        merged = ctx.groups_merge(kd.allgather_groups(packed, dev))
        return rows, merged

    cfg3_steps(3)
    ctx.get_stats(reset=True)
    ctx.set_timing(True)
    barrier()
    t0 = time.perf_counter()
    rows3, merged = cfg3_steps(K)
    ctx.synchronize()
    dt3 = time.perf_counter() - t0
    barrier()
    st3 = ctx.get_stats(reset=True)
    ctx.set_timing(False)
    plan3.free()
    check_groups(merged)
    rows3_all, = reduce_sum(rows3)
    assert rows3_all == E_glob
    dt3m, dev3 = reduce_max(dt3, st3["probe_ms"] / K)
    out["cfg3_group_by_merge_nccl"] = {
        "workload": "same query; partial groups packed (kb_groups_pack), all-gathered over NCCL, folded on every rank by kb_groups_merge",
        "value": rows3_all / (dt3m / K), "unit": "bindings/s", "ms_per_step": dt3m / K * 1e3, "device_ms_per_step_join_group": dev3,
        "collective": "all_gather_into_tensor of one %d-byte slot per rank and step" % kd.GROUPS_SLOT_BYTES, "parity": "groups == closed-form global title histogram"}

    # ---- shuffle_join: (?e reports_to ?m) . (?m foaf:title ?t) — the first pattern's rows live with ?e, the join key ?m is not their
    # subject: they are re-sharded by ?m with ONE kernel per rank (kb_shuffle_push: peer stores over NVLink) and joined locally.
    E_, M_, T_ = 0, 5, 1
    e_ids, m_ids, t_of_m = datagen.reports_to_relation(d, rank, world)
    left = ctx.rel_from_host([E_, M_], [e_ids, m_ids])
    right_pat = c.pattern(c.V(M_), c.K(d.ids["foaf:title"]), c.V(T_))
    cap = int(reduce_max(len(e_ids))[0] * 1.25) + 65536  # symmetric memory: the same size on every rank
    ps = kd.PeerShuffle(ctx, n_cols=2, capacity_rows=cap)
    sh_times, join_times, rows_j = [], [], 0
    for rep in range(1 + max(3, min(K, 6))):
        barrier()
        t0 = time.perf_counter()
        sh = ps.shuffle(left, M_)
        t1 = time.perf_counter()
        j = ctx.bind_join(sh, right_pat)  # (?m foaf:title ?t): one lookup kernel against the index's persistent table
        rows_j = j.n_rows
        ctx.synchronize()
        t2 = time.perf_counter()
        if rep:
            sh_times.append(t1 - t0)
            join_times.append(t2 - t1)
        if rep == 0:  # parity (untimed): order-independent digest of the joined rows, summed over ranks == closed form summed over ranks
            got_d = datagen.row_checksums(j.to_numpy([E_, M_, T_]))
            want_d = datagen.row_checksums(np.stack([e_ids, m_ids, t_of_m], axis=1))
            owner_ok = bool((datagen.shard_of_np(sh.to_numpy([E_, M_])[:, 1], world) == rank).all())
        sh.free()
        j.free()
    # the 64-bit digests travel as two 32-bit halves (the all-reduce sums int64) and are recombined modulo 2^64
    n_got, lo_g, hi_g = reduce_sum(got_d[0], got_d[1] & 0xFFFFFFFF, got_d[1] >> 32)
    n_want, lo_w, hi_w = reduce_sum(want_d[0], want_d[1] & 0xFFFFFFFF, want_d[1] >> 32)
    ok_all, = reduce_sum(int(owner_ok))
    assert n_got == n_want == E_glob and ok_all == world, (n_got, n_want, ok_all)
    assert ((hi_g << 32) + lo_g) % (1 << 64) == ((hi_w << 32) + lo_w) % (1 << 64), "joined rows differ from the closed form"
    t_sh, t_j = reduce_max(float(np.median(sh_times)), float(np.median(join_times)))
    rows_j_all, sent = reduce_sum(rows_j, int((datagen.shard_of_np(m_ids, world) != rank).sum()))
    nv_bytes_rank = 8 * sent / world
    out["shuffle_join"] = {
        "workload": f"path join (?e reports_to ?m).(?m foaf:title ?t): {len(e_ids)} rows per rank x {world} ranks re-sharded by the non-subject key ?m, then joined locally",
        "value": rows_j_all / (t_sh + t_j), "unit": "bindings/s", "ms_shuffle": t_sh * 1e3, "ms_join": t_j * 1e3,
        "nvlink_bytes_sent_per_rank": nv_bytes_rank, "nvlink_gbs_per_rank": nv_bytes_rank / t_sh / 1e9,
        "exchange": "kb_shuffle_push: one kernel per rank sorts a tile by destination in shared memory, reserves its range on the receiver's own cursor "
                    "(peer atomic) and streams 128-byte-aligned runs into the receiver's buffer; two symmetric-memory barriers around it; no count exchange",
        "parity": "bag digest of the joined rows summed over ranks == closed form; every received row belongs to its rank"}
    left.free()
    del ps

    # ---- strong scaling: the 100 M-triple store of BASELINE configs[2] (args.employees in total) split over the N GPUs
    ctx2 = c.Context(local)
    ds = datagen.employee_shard(args.employees, rank, world)
    ctx2.set_sharding(rank, world)
    ctx2.dict_numeric_load(ds.num_or0, ds.is_num)
    ctx2.store_load(ds.s, ds.p, ds.o)
    ctx2.build_index()
    jss, patss, filts = datagen.employee_queries(ds)[args.query]
    plans = ctx2.prepare_star_join(jss, patss, filts, ring=args.ring)
    run_pipelined(plans, 5)
    ctx2.set_timing(True)
    ctx2.get_stats(reset=True)
    barrier()
    t0 = time.perf_counter()
    rows_s = run_pipelined(plans, K)
    ctx2.synchronize()
    dt_s = time.perf_counter() - t0
    barrier()
    sts = ctx2.get_stats(reset=True)
    plans.free()
    ctx2.close()
    rows_s_all, = reduce_sum(rows_s)
    dt_sm, dev_s = reduce_max(dt_s, sts["total_ms"] / K)
    out["strong"] = {"workload": f"{6 * args.employees} triples in TOTAL over {world} GPUs (BASELINE configs[2] store), same query and protocol as the headline",
                     "value": rows_s_all / (dt_sm / K), "unit": "bindings/s", "ms_per_step": dt_sm / K * 1e3, "device_ms_per_step": dev_s,
                     "bindings_per_step": rows_s_all, "scaling": "strong"}
    return out


if __name__ == "__main__":
    main()
