#!/usr/bin/env python
"""bench.py — pods scheduled/sec of the allocate hot path (BASELINE.json metric).

A "step" is ONE scheduling cycle of the workload (BASELINE configs[1]: 10k nodes x 100k pending tasks,
8 resource dims, gang + predicates + nodeorder + binpack) through the reference-facing C ABI:

  value  : placements / device time of vc_allocate_run's commit kernel, snapshot already resident in HBM
  e2e    : placements / wall time of vc_snapshot_upload (host SoA -> HBM, session-open) + vc_allocate_run +
           result fetch to host buffers — the call sequence the cgo shim makes every cycle
  roofline : the dense task x node mask + score kernel (K1, SURVEY §8d) timed in the same process with CUDA
             events; algorithmic bytes / time against the measured HBM peak of MEASURED_PEAKS.json
  cpu_baseline : the CPU restatement of the reference path (oracle/, "port") on this box's host cores

--impl reference times that CPU restatement alone (the Go reference cannot be built: no go toolchain).
N > 1 (torchrun): ONE cluster, the same session on every rank, strong scaling. The node axis is cut over the CTAs of all
GPUs: the exact allocate loop runs as one persistent kernel per GPU whose per-step records cross NVLink through
peer-mapped mailboxes (vc_comm_*), and the dense task x node pass (K1) is node-sharded with NCCL collectives
(MAX all-reduce of the group statistics, all-gather + fold of the per-task best). value = placements of the one
cluster / max-over-ranks kernel time. N scheduler replicas (one cluster per GPU) are reported as a labelled secondary number.

--dump-outputs DIR writes what the last timed step returned (decisions, visits, fit errors) as DIR/<name>.npy, so that two
builds can be compared output for output on the same seeded workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOAD = "cfg2"
METRIC = "pods scheduled/sec"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [ln.strip().split(", ") for ln in open(self.f.name) if ln.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for nm, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_oracle(snap, threads, want_results=False):
    from oracle.pyoracle import OracleSession
    o = OracleSession(snap, threads=threads)
    t0 = time.perf_counter()
    dec, vis, fe = o.allocate()
    dt = time.perf_counter() - t0
    o.close()
    if want_results:
        return len(dec), dt, (dec, vis, fe)
    return len(dec), dt


DUMP_BYTES = 60_000_000  # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(out_dir, decisions, visits, fit_errors, job_allocated_hypernodes=None):
    """One cycle's result as out_dir/<array>_<field>.npy in float64 (the int32 fields are exact there). Above DUMP_BYTES in
    all, every k-th row of each array is written: the same rows for outputs of the same lengths."""
    arrays = {f"decisions_{f}": decisions[f] for f in decisions.dtype.names}
    arrays.update({f"visits_{f}": visits[f] for f in visits.dtype.names})
    arrays["fit_errors"] = fit_errors
    if job_allocated_hypernodes is not None:
        arrays["job_allocated_hypernodes"] = job_allocated_hypernodes
    stride = max(1, -(-8 * sum(a.size for a in arrays.values()) // DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a[::stride], np.float64))


KERNEL_NAMES = {0: "k_commit (general)", 1: "k_commit_fast (incremental)"}
# session shapes other than the headline one, same size (10k nodes x 100k tasks): GPU cycle vs the CPU port in the same mode
MODE_WORKLOADS = [("Releasing resources (terminating pods: FutureIdle gradient, pipelining)", "cfg2_fut"),
                  ("PreferNoSchedule taints (normalising TaintToleration batch score)", "cfg2_soft")]


def mode_results(device, threads):
    from volcano_b200 import engine
    from volcano_b200.synth import CONFIGS, make_snapshot
    out = []
    for mode, name in MODE_WORKLOADS:
        try:
            msnap = make_snapshot(CONFIGS[name])
            e = engine.Engine(msnap, device=device)
            e.upload()
            e.allocate()
            r = e.allocate()
            e.close()
            n, dt, oracle_results = run_oracle(msnap, threads, want_results=True)
            gpu_v = len(r.decisions) / (r.stats["commit_ms"] * 1e-3)
            out.append({"mode": mode, "workload": name, "gpu_ms": r.stats["commit_ms"], "gpu_pods_per_s": gpu_v,
                        "cpu_pods_per_s": n / dt, "cpu_threads": threads, "speedup": gpu_v / (n / dt),
                        "placements_identical": compare_placements(r, oracle_results)["placements_identical"],
                        "kernel": KERNEL_NAMES.get(r.stats["commit_kernel"])})
        except Exception as ex:  # a mode's failure must not hide the headline line
            out.append({"mode": mode, "workload": name, "error": str(ex)})
    return out


def compare_placements(res, oracle_results):
    """GPU result vs the cpu_baseline leg's result on the SAME snapshot: identical placements (task, node, kind, visit,
    in order), visit outcomes and fit errors; fp64 scores within 1e-6 (north_star). -> dict for the JSON line."""
    dec, vis, fe = oracle_results
    out = {"placements_identical": False, "first_difference": None, "compared": int(len(dec)),
           "max_abs_score_diff": None}
    if len(res.decisions) != len(dec):
        out["first_difference"] = {"what": "number of decisions", "gpu": int(len(res.decisions)), "cpu": int(len(dec))}
        return out
    for f in ("task", "node", "kind", "visit"):
        ne = np.nonzero(res.decisions[f] != dec[f])[0]
        if len(ne):
            out["first_difference"] = {"what": f"decision.{f}", "index": int(ne[0])}
            return out
    if not np.array_equal(res.visits, vis):
        out["first_difference"] = {"what": "visits"}
        return out
    if not np.array_equal(res.fit_errors, fe):
        out["first_difference"] = {"what": "fit_errors"}
        return out
    diff = float(np.max(np.abs(res.decisions["score"] - dec["score"]))) if len(dec) else 0.0
    out["max_abs_score_diff"] = diff
    out["placements_identical"] = diff <= 1e-6
    return out


def config_dict(name, world):
    """The same keys in both arms (the driver compares the dicts)."""
    return {"workload": workload_desc(name),
            "parallelism": ("one cluster, node axis cut over %d GPUs (peer-mapped mailbox / ring over NVLink; K1 node-sharded "
                            "over NCCL)" % world) if world > 1 else "1 GPU",
            "l2": "256 MB buffer written between timed iterations (GPU arm)",
            "timed_region": "GPU arm: per-cycle resets + k_commit (CUDA events on its stream), e2e = upload + run + fetch "
                            "wall time; reference arm: the allocate action, wall time"}


def workload_desc(name):
    from volcano_b200.synth import CONFIGS
    cfg = CONFIGS[name]
    return (f"{name}: {cfg.n_nodes} nodes x {cfg.n_tasks} tasks, R=8, {cfg.plugins}, "
            "percentage-nodes-to-find=100 (parity mode)")


def reference_arm(args, rank, world):
    """The reference's CPU implementation of the path = oracle port (kind "port"), all usable host threads
    (the reference runs 16 workers per task: util/predicate_helper.go:133)."""
    if rank != 0:
        return
    from volcano_b200.synth import make_snapshot
    snap = make_snapshot(args.workload)
    threads = max(1, min(16, cpu_cores()))
    for _ in range(args.warmup if args.warmup < 2 else 1):  # warm-up is a CPU cache matter only; one pass
        run_oracle(snap, threads)
    placed, times = 0, []
    for _ in range(args.steps):
        n, dt, out = run_oracle(snap, threads, want_results=True)
        placed += n
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *out)
    total = sum(times)
    val = placed / total
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pods/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong" if max(world, args.gpus) > 1 else "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": config_dict(args.workload, max(world, args.gpus)),
        "cpu_baseline": {"value": val, "unit": "pods/s", "cores": threads, "kind": "port",
                         "sample": "full workload, one allocate cycle per step"},
        "e2e": {"value": val, "unit": "pods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def multi_gpu_arm(args, rank, world, local):
    """ONE cluster across `world` GPUs (SURVEY §8e): see the module docstring."""
    import torch
    import torch.distributed as dist
    from volcano_b200 import engine
    from volcano_b200.parallel import sharded_dense_best
    from volcano_b200.parallel_commit import MultiGpuSession
    from volcano_b200.synth import CONFIGS, make_snapshot

    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    cfg = CONFIGS[args.workload]
    snap = make_snapshot(cfg)  # the same cluster on every rank
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def tmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms = MultiGpuSession(snap, local)
    for _ in range(max(3, args.warmup)):
        res = ms.allocate()
    sampler = ClockSampler(local)
    sampler.start()
    # ---- device-timed value: the persistent kernels of all ranks on the resident session ----------
    dev_ms, placed, n_steps = [], 0, 0
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        res = ms.allocate()
        dev_ms.append(tmax(res.stats["commit_ms"]))  # max over ranks of each rank's CUDA-event time
        cnt = torch.tensor([len(res.decisions), res.stats["n_steps"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(cnt, op=dist.ReduceOp.MAX)  # rank 0 holds the decisions of the one cluster
        placed += int(cnt[0].item())
        n_steps += int(cnt[1].item())
    timed = res
    t_dev = sum(dev_ms) / 1e3
    # ---- e2e: host buffers -> upload on every rank -> one session -> decisions on rank 0's host ----
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    e2e_placed, h2d, d2h = 0, 0, 0
    for _ in range(args.steps):
        ms.upload()
        res = ms.allocate()
        e2e_placed += len(res.decisions)
        h2d, d2h = res.stats["h2d_bytes"], res.stats["d2h_bytes"]
    torch.cuda.synchronize()
    t_e2e = tmax(time.perf_counter() - t0)
    cnt = torch.tensor([e2e_placed], dtype=torch.float64, device="cuda")
    dist.all_reduce(cnt, op=dist.ReduceOp.MAX)
    e2e_placed = int(cnt.item())
    clocks = sampler.stop()
    last = res
    ms.close()
    # ---- K1 node-sharded: shard kernels + one MAX all-reduce + one all-gather / fold (NCCL) --------
    dense = None
    try:
        eng = engine.Engine(snap, device=local)
        eng.upload()
        times = []
        for _ in range(4):
            torch.cuda.synchronize(); dist.barrier()
            t1 = time.perf_counter()
            sharded_dense_best(eng, world, rank, dev, materialize=True)
            torch.cuda.synchronize()
            times.append(tmax(time.perf_counter() - t1))
        eng.set_shard(0, snap.N)
        _, _, nbytes = eng.score_matrix_device(repeats=1)
        eng.close()
        peak, how = _peaks()
        best = min(times[1:])
        dense = {"kernel": "K1 node-sharded (mask + f64 score matrix shard per GPU) + MAX all-reduce + all-gather/fold",
                 "ms": 1e3 * best, "algorithmic_bytes_all_gpus": nbytes, "achieved_gbs_all_gpus": nbytes / best / 1e9,
                 "frac_of_n_times_peak": nbytes / best / 1e9 / (peak * world), "peak_per_gpu": peak, "peak_source": how,
                 "includes": "host launch overhead and the two NCCL collectives (wall clock, max over ranks)"}
    except Exception as ex:
        dense = {"error": str(ex)}
    # ---- secondary: N scheduler replicas, one cluster per GPU (no exchange) ----------------------
    replicas = None
    try:
        snap_r = make_snapshot(cfg, seed=cfg.seed + rank)
        er = engine.Engine(snap_r, device=local)
        er.upload()
        er.allocate()
        torch.cuda.synchronize(); dist.barrier()
        rr = er.allocate()
        er.close()
        tr = tmax(rr.stats["commit_ms"])
        c2 = torch.tensor([len(rr.decisions)], dtype=torch.float64, device="cuda")
        dist.all_reduce(c2, op=dist.ReduceOp.SUM)
        replicas = {"value": float(c2.item()) / (tr * 1e-3), "unit": "pods/s", "ms": tr,
                    "note": "N independent clusters, one per GPU (weak scaling, no data-path exchange) - not the headline"}
    except Exception as ex:
        replicas = {"error": str(ex)}
    # ---- parity of the multi-GPU session: rank 0 runs the SAME cluster on its GPU alone (the arm bench.py checks against the
    #      CPU port at N=1) and compares every decision, visit and fit error ---------------------------------------------------
    same = None
    if rank == 0:
        try:
            e1 = engine.Engine(snap, device=local)
            e1.upload()
            r1 = e1.allocate()
            e1.close()
            same = bool(np.array_equal(r1.decisions, last.decisions) and np.array_equal(r1.visits, last.visits) and
                        np.array_equal(r1.fit_errors, last.fit_errors))
        except Exception as ex:
            same = "error: %s" % ex
    if rank == 0:
        line = {
            "metric": METRIC, "value": placed / t_dev, "unit": "pods/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": 1e3 * t_dev / args.steps,
            "cycle_ms_p50": statistics.median(dev_ms), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.workload, world),
            "sweeps_per_step": n_steps / args.steps,
            "placements_identical": same,
            "parity": {"placements_identical": same, "against": "the same session on one GPU (decisions, scores, visits, fit errors "
                       "bit-equal); that arm is compared with the CPU port by the N=1 run"},
            "e2e": {"value": e2e_placed / t_e2e, "unit": "pods/s", "h2d_bytes_per_step": int(h2d) * world,
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * t_e2e / args.steps,
                    "note": "the snapshot is uploaded to every rank (h2d counts all of them); decisions come back from rank 0"},
            "gpu_launches": 2 * args.steps * world,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "K1 node-sharded over the ranks (wall clock incl. its two NCCL collectives)",
                         "achieved": (dense or {}).get("achieved_gbs_all_gpus"),
                         "peak": ((dense or {}).get("peak_per_gpu") or 0) * world or None, "unit": "GB/s",
                         "frac": (dense or {}).get("frac_of_n_times_peak"), "traffic": None, "sharded": dense},
            "cpu_baseline": None,
            "commit_kernel": {"kernel": "k_commit_fast, one persistent kernel per GPU, node axis cut over all their CTAs",
                              "bound": "latency (one NVLink round trip whenever the winning node moves to another GPU)",
                              "ms": 1e3 * t_dev / args.steps, "us_per_placement_attempt": 1e6 * t_dev / max(1, n_steps),
                              "exchange": "16-byte records stored into every rank's peer-mapped mailbox / publication ring "
                                          "(CUDA IPC), polled locally; no host or NCCL call inside the cycle"},
            "replicas_secondary": replicas,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, timed.decisions, timed.visits, timed.fit_errors, timed.job_allocated_hypernodes)
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default=WORKLOAD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    from volcano_b200 import engine
    from volcano_b200.synth import CONFIGS, make_snapshot

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libvcalloc has no CPU path")
    if world > 1:
        multi_gpu_arm(args, rank, world, local)
        return
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = CONFIGS[args.workload]
    snap = make_snapshot(cfg, seed=cfg.seed + rank)  # every rank its own cluster shard of the same shape
    eng = engine.Engine(snap, device=local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also allocates every device buffer) ----
    for _ in range(max(3, args.warmup)):
        eng.upload()
        res = eng.allocate()
    # ---- device-timed value: commit kernel on a resident snapshot -------------------------------
    eng.upload()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    dev_ms, placed = [], 0
    n_steps = 0
    for _ in range(args.steps):
        flush.fill_(1)  # L2 flush between timed iterations
        torch.cuda.synchronize()
        res = eng.allocate()
        dev_ms.append(res.stats["commit_ms"])  # CUDA events on the launching stream around k_commit
        placed += len(res.decisions)
        n_steps += res.stats["n_steps"]
    timed = res
    barrier()
    t_dev = sum(dev_ms) / 1e3
    # ---- e2e: host buffers -> upload -> allocate -> decisions on the host ------------------------
    barrier()
    t0 = time.perf_counter()
    e2e_placed, h2d, d2h = 0, 0, 0
    for _ in range(args.steps):
        eng.upload()
        res = eng.allocate()
        e2e_placed += len(res.decisions)
        h2d, d2h = res.stats["h2d_bytes"], res.stats["d2h_bytes"]
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    barrier()
    # ---- steady state of a cluster whose pending set did not change: only the accounting rows of the nodes whose
    #      NodeInfo.Generation moved go up (vc_snapshot_update_nodes; 5 % of the nodes here, same values) ----------
    inc = None
    try:
        dirty = np.sort(np.random.default_rng(1).choice(snap.N, size=max(1, snap.N // 20), replace=False)).astype(np.int32)
        rows = (snap.n_idle[:, dirty], snap.n_used[:, dirty], snap.n_releasing[:, dirty], snap.n_pipelined[:, dirty],
                snap.n_k8s_requested[:, dirty], snap.n_k8s_nonzero_requested[:, dirty], snap.n_pod_count[dirty])
        eng.update_nodes(dirty, *rows)
        eng.allocate()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        inc_placed, inc_h2d = 0, 0
        for _ in range(args.steps):
            eng.update_nodes(dirty, *rows)
            r_inc = eng.allocate()
            inc_placed += len(r_inc.decisions)
            inc_h2d = r_inc.stats["h2d_bytes"]
        torch.cuda.synchronize()
        t_inc = time.perf_counter() - t1
        inc = {"value": inc_placed / t_inc, "unit": "pods/s", "ms_per_step": 1e3 * t_inc / args.steps,
               "h2d_bytes_per_step": int(inc_h2d), "dirty_nodes": int(len(dirty)),
               "same_placements_as_full_upload": bool(np.array_equal(r_inc.decisions, res.decisions)),
               "note": "pending set unchanged since the last full upload; rows of 5 % of the nodes re-sent"}
        eng.upload()
    except Exception as ex:
        inc = {"error": str(ex)}
    clocks = sampler.stop()
    # ---- roofline kernel: dense task x node mask + score matrix ---------------------------------
    roof = None
    if rank == 0:
        try:
            dense_ms, expand_ms, nbytes = eng.score_matrix_device(repeats=4)
            peak, how = _peaks()
            ach = nbytes / (expand_ms * 1e-3) / 1e9
            traffic = None
            tp = os.path.join(ROOT, "profiles", "r01_k1_expand_ncu.json")
            if os.path.exists(tp) and args.workload == WORKLOAD:
                traffic = json.load(open(tp)).get("traffic_bytes_per_launch")  # dram read+write, ncu --set full
            # the kernel is ~99.8 % stores: next to the (read+write) copy peak of MEASURED_PEAKS.json also measure a
            # write-only stream in this run (SURVEY §8d): cudaMemset-class fill of an 8 GB f64 buffer, best of 5
            wpeak = None
            try:
                buf = torch.empty(2 ** 30, dtype=torch.float64, device="cuda")
                best = 1e9
                for _ in range(5):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); buf.fill_(1.5); b.record(); torch.cuda.synchronize()
                    best = min(best, a.elapsed_time(b))
                wpeak = buf.numel() * 8 / (best * 1e-3) / 1e9
                del buf
            except Exception:
                pass
            roof = {"bound": "hbm", "kernel": "k_group_expand_bulk (task x node mask + f64 score matrix, K1b)",
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                    "share_of_step": 0.0,
                    "peak_source": how, "algorithmic_bytes": nbytes, "kernel_ms": expand_ms,
                    "write_only_peak": wpeak, "frac_of_write_only_peak": (ach / wpeak) if wpeak else None,
                    "dense_pass_ms": dense_ms, "achieved_whole_pass": nbytes / (dense_ms * 1e-3) / 1e9}
        except Exception as ex:  # e.g. not enough memory for the matrix
            roof = {"bound": "hbm", "error": str(ex)}
    # ---- aggregate over ranks: max time, sum of units ---------------------------------------------
    if dist is not None:
        tt = torch.tensor([t_dev, t_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        cc = torch.tensor([placed, e2e_placed], dtype=torch.float64, device="cuda")
        dist.all_reduce(cc, op=dist.ReduceOp.SUM)
        t_dev, t_e2e = tt.tolist()
        placed, e2e_placed = cc.tolist()
    value = placed / t_dev
    e2e_value = e2e_placed / t_e2e
    cpu = None
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        threads = max(1, min(16, cpu_cores()))
        n, dt, oracle_results = run_oracle(snap, threads, want_results=True)
        parity = compare_placements(res, oracle_results)  # `res`: the last e2e cycle of the GPU arm, same snapshot
        cpu = {"value": n / dt, "unit": "pods/s", "cores": threads, "kind": "port",
               "sample": "full workload, one allocate cycle (%.1f s), percentage-nodes-to-find=100; its decisions are "
                         "compared with the GPU arm's (placements_identical)" % dt}
        # the reference's DEFAULT search-space reduction (adaptive 5 %% of 10k nodes = 500 feasible nodes per task,
        # util/scheduler_helper.go:54-73) makes its CPU path ~20x cheaper per task and yields different placements;
        # reported so that the parity-mode ratio is not mistaken for the production-default ratio (BASELINE.md §2)
        try:
            snap.conf.percentage_nodes_to_find = 0
            n2, dt2, samp_results = run_oracle(snap, threads, want_results=True)
            cpu["reference_defaults"] = {"value": n2 / dt2, "unit": "pods/s", "placed": n2, "seconds": dt2,
                                         "note": "adaptive feasible-node sampling (deterministic single-worker reading); "
                                                 "different placements than parity mode"}
            # the same mode on the device (general commit kernel with the selection pass), informational
            eng.upload()
            eng.allocate()
            r2 = eng.allocate()
            cpu["reference_defaults"]["gpu_same_mode"] = {
                "value": len(r2.decisions) / (r2.stats["commit_ms"] * 1e-3), "unit": "pods/s", "placed": len(r2.decisions),
                "ms": r2.stats["commit_ms"], "kernel": KERNEL_NAMES.get(r2.stats["commit_kernel"]),
                "placements_identical": compare_placements(r2, samp_results)["placements_identical"]}
        finally:
            snap.conf.percentage_nodes_to_find = 100
    modes = None
    if rank == 0 and not args.no_cpu_baseline and args.workload == WORKLOAD:
        modes = mode_results(local, max(1, min(16, cpu_cores())))
        if cpu and "reference_defaults" in cpu and "gpu_same_mode" in cpu["reference_defaults"]:
            rd = cpu["reference_defaults"]
            modes.insert(0, {"mode": "feasible-node sampling (the reference's defaults)", "workload": args.workload,
                             "gpu_ms": rd["gpu_same_mode"]["ms"], "gpu_pods_per_s": rd["gpu_same_mode"]["value"],
                             "cpu_pods_per_s": rd["value"], "cpu_threads": cpu["cores"],
                             "speedup": rd["gpu_same_mode"]["value"] / rd["value"],
                             "placements_identical": rd["gpu_same_mode"].get("placements_identical"),
                             "kernel": rd["gpu_same_mode"].get("kernel")})
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "pods/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": 1e3 * t_dev / args.steps,
            "cycle_ms_p50": statistics.median(dev_ms), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args.workload, world),
            "sweeps_per_step": n_steps / args.steps,
            "placements_identical": parity["placements_identical"] if parity else None,
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": "pods/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * t_e2e / args.steps},
            "e2e_incremental": inc,
            "gpu_launches": 2 * args.steps,  # k_class_static + k_commit per e2e step (1 per device-timed step)
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "modes": modes,
            "commit_kernel": {"kernel": "k_commit_fast (persistent cooperative, exact greedy loop)", "bound": "latency",
                              "share_of_step": 0.9999, "ms": 1e3 * t_dev / args.steps,
                              "us_per_placement_attempt": 1e6 * t_dev / max(1, n_steps),
                              "hbm_traffic": "inputs once (17 MB); node state is shared-memory resident"},
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, timed.decisions, timed.visits, timed.fit_errors, timed.job_allocated_hypernodes)
        print(json.dumps(line), flush=True)
        if parity is not None and not parity["placements_identical"]:
            eng.close()
            raise SystemExit("bench.py: GPU placements differ from the cpu_baseline leg's: %s" % json.dumps(parity))
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
