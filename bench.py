#!/usr/bin/env python
"""bench.py — pose-opt iterations/s (bodies x corr_iters) of the M3T pose-optimisation hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                      (the CPU arm: the oracle port on the host cores)
  python bench.py ... --dump-outputs DIR                    (also writes the poses of the last timed step, DIR/poses.npy)

A "step" is one Tracker::ExecuteTrackingStep pass (n_corr correspondence iterations x n_update update
iterations, tracker.cpp:344-361) over this GPU's batch of bodies = ONE launch of the fused kernel k_track.
Default workload: the per-GPU shard of BASELINE.json configs[3] ("1024 bodies Region+Depth, 512 lines each,
640x480 RGB-D, sharded 8xB200" -> 128 bodies per GPU, weak scaling), the configuration the metric's
1/2/4/8-GPU numbers are quoted on; `--workload c2|c3` selects the other configs.

value : whole-job throughput, frames already resident in HBM, timed with CUDA events around each step on the
        launching stream, L2 flushed between steps (untimed), max over ranks.
e2e   : the same through the C ABI with HOST buffers: per step the pinned-host -> device copy of every body's
        RGB-D frame + start poses, the step, the device -> host read of the solved poses (+ the pose all-gather
        at N>1); wall clock around synchronised regions, max over ranks.
"""
from __future__ import annotations

import os
import sys

# Before anything can load an OpenMP runtime (numpy / torch do): pin the CPU arm's threads to cores. Unbound, a
# 128-thread team on this host alternates between 2.4 ms and 95 ms per step (measured, tests/diag/cpu_arm_threads.py); bound it
# is stable and fastest, which is the honest baseline. ONLY in processes that run the CPU arm (single-process runs and
# --impl reference): OMP_PROC_BIND also pins the initial thread to the first place, so under torchrun every rank's host
# thread would land on the same core - at 4 and 8 ranks that made every other end-to-end step wait ~19 ms for a
# time slice (scripts/e2e_scaling_diag.py). stdout carries exactly one JSON line: keep NCCL's banner out.
if int(os.environ.get("WORLD_SIZE", "1")) == 1 or "reference" in sys.argv:
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

import argparse  # noqa: E402
import importlib  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pose-opt iterations/sec (bodies x corr_iters)"
UNIT = "pose-opt iterations/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--variant", default="projected", choices=["projected", "constrained"],
                    help="c5 only: joints as projected unknowns or as 6-DoF links + constraints (optimization_time.cpp)")
    ap.add_argument("--bodies", type=int, default=None, help="bodies per GPU (default: the preset's)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the poses the last timed step solved (every body of the job, float32) to DIR/poses.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 path computed; it does not apply to --impl reference")
    return args


def workload_description(wl, args, per_gpu=None):
    r = f"{wl.lines_per_body} lines" if wl.region else ""
    d = f"{wl.points_per_body} depth points" if wl.depth else ""
    both = " + ".join(x for x in (r, d) if x)
    if args.workload == "c5":
        st = wl.structures[0]
        n_chains = (per_gpu or wl.n_bodies) // len(st.links)
        return (f"configs[4] per-GPU shard (256 chains / 8 GPUs): {n_chains} chains/GPU x {len(st.links)} links x ({both}), "
                f"{wl.notes['variant']} joints ({st.dof} unknowns + {st.n_constraint_rows} constraint rows per chain), "
                f"one 640x480 RGB-D pair per link, {wl.n_corr_iterations} corr x {wl.n_update_iterations} update iterations")
    preset = {"c2": "configs[1]", "c3": "configs[2]", "c4": "configs[3] per-GPU shard (1024 bodies / 8 GPUs)"}[args.workload]
    return (f"{preset}: {per_gpu or wl.n_bodies} bodies/GPU x ({both}), one 640x480 "
            f"{'RGB-D pair' if wl.depth and wl.region else 'frame'} per body, "
            f"{wl.n_corr_iterations} corr x {wl.n_update_iterations} update iterations")


def config_dict(wl, args, world, per_gpu):
    """The `config` both arms print (identical dicts, so that the driver's same_config check reads true)."""
    frame_mib = 0.0
    if wl.color_frames is not None:
        frame_mib += wl.color_frames[0].nbytes * per_gpu / 2 ** 20
    if wl.depth_frames is not None:
        frame_mib += wl.depth_frames[0].nbytes * per_gpu / 2 ** 20
    return {"workload": workload_description(wl, args, per_gpu=per_gpu), "bodies_per_gpu": int(per_gpu),
            "l2": f"flushed (256 MiB memset) between timed steps; each step's frames are {frame_mib:.0f} MiB/GPU (> L2)",
            "timing": "GPU arm: CUDA events around each step on the launching stream, summed over K steps, max over ranks; "
                      "CPU arm: steady_clock around each full step",
            "parallelism": f"bodies sharded x{world}, no data-path collective"}


def source_sha():
    """sha256 over the CUDA sources: ties profiles/traffic.json (an ncu capture) to the kernel it was captured from."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "3dobjecttracking_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def parity_check(ctx, wl, n_sample=4):
    """What was just timed, checked: the first n_sample bodies of the benchmarked batch against the CPU oracle
    (reference-faithful mode: polar rotation(), Pade exp). (i) per correspondence iteration on identical inputs (both
    sides enter every iteration with the oracle's pose) - the north_star gate of 1e-4 m / 1e-4 rad; (ii) the fused
    whole-step launch free-running from the start poses. The oracle is the checker here, never the thing measured."""
    if getattr(wl, "structures", None):
        return {"skipped": "kinematic structures: covered by tests/test_gpu_structures.py"}
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    n = min(n_sample, wl.n_bodies)
    orc = oracle_py.OracleTracker(wl, rotation_mode=oracle_py.ROTATION_POLAR, exp_mode=oracle_py.EXP_PADE, n_threads=n)
    # second realisation of the same algorithm (linear rotation block, Rodrigues): where the two oracle modes end an
    # iteration more than the tolerance apart, a 1e-7 difference has flipped an integer decision of the algorithm (an
    # int() of a line coordinate, a histogram bin pair, a template view) and the pair says nothing about the CUDA path
    alt = oracle_py.OracleTracker(wl, rotation_mode=oracle_py.ROTATION_LINEAR, exp_mode=oracle_py.EXP_RODRIGUES, n_threads=n)
    orc.start_modalities(0)
    alt.start_modalities(0)

    def err(p, q):
        p, q = np.asarray(p, np.float64).reshape(-1, 3, 4), np.asarray(q, np.float64).reshape(-1, 3, 4)
        dt = np.linalg.norm(p[:, :, 3] - q[:, :, 3], axis=1)
        R = np.einsum("bij,bkj->bik", p[:, :, :3], q[:, :, :3])
        c = np.clip((np.trace(R, axis1=1, axis2=2) - 1.0) / 2.0, -1.0, 1.0)
        sk = 0.5 * np.sqrt((R[:, 2, 1] - R[:, 1, 2]) ** 2 + (R[:, 0, 2] - R[:, 2, 0]) ** 2 + (R[:, 1, 0] - R[:, 0, 1]) ** 2)
        return dt, np.arctan2(sk, c)

    worst_m = worst_rad = 0.0
    compared = excluded = 0
    orc.set_poses(wl.start_body2world)
    for corr in range(wl.n_corr_iterations):
        start = orc.get_poses()
        alt.set_poses(start)
        ctx.set_poses(start)
        ctx.corr_iteration(0, corr, wl.n_update_iterations)
        orc.tracking_step(0, n_corr=corr + 1, corr_begin=corr, first=0, count=n)
        alt.tracking_step(0, n_corr=corr + 1, corr_begin=corr, first=0, count=n)
        st, sr = err(alt.get_poses()[:n], orc.get_poses()[:n])
        ok = (st < 1e-4) & (sr < 1e-4)
        dt, dr = err(ctx.get_poses(0, n), orc.get_poses()[:n])
        compared += int(ok.sum())
        excluded += int((~ok).sum())
        if ok.any():
            worst_m, worst_rad = max(worst_m, float(dt[ok].max())), max(worst_rad, float(dr[ok].max()))
    ctx.set_poses(wl.start_body2world)
    ctx.tracking_step(0, wl.n_corr_iterations, wl.n_update_iterations)
    orc.set_poses(wl.start_body2world)
    orc.tracking_step(0, first=0, count=n)
    dt, dr = err(ctx.get_poses(0, n), orc.get_poses()[:n])
    moved, _ = err(ctx.get_poses(0, n), wl.start_body2world[:n])
    return {"bodies": int(n), "oracle": "CPU restatement, reference-faithful mode (polar rotation, Pade exp)",
            "per_iteration_max_m": worst_m, "per_iteration_max_rad": worst_rad, "tolerance": 1e-4,
            "body_iterations_compared": compared, "body_iterations_excluded_oracle_modes_disagree": excluded,
            "ok": bool(compared > 0 and worst_m < 1e-4 and worst_rad < 1e-4),
            "free_running_step_max_m": float(dt.max()), "free_running_step_max_rad": float(dr.max()),
            "pose_change_of_the_step_m": float(moved.min())}


def bind_to_gpu_numa_node(torch, local_rank):
    """Pin this rank's host threads (and therefore, by first touch, the pinned frame buffers it allocates next) to the
    NUMA node its GPU hangs off. Unbound, the 8 ranks' zero-copy frame reads cross the socket interconnect for half of
    the GPUs (GPUs 0-3 on node 0, 4-7 on node 1 on the 8-GPU boxes) and the end-to-end step time rose from 0.71 to
    0.99 ms at N = 8 (SCALE_r01). Returns a description for the JSON line."""
    try:
        prop = torch.cuda.get_device_properties(local_rank)
        bdf = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return {"numa_node": None, "note": "single NUMA node / not reported"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_node": node, "note": "no allowed CPU on that node"}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "pci": bdf}
    except Exception as e:  # no sysfs, no permission: run unbound
        return {"numa_node": None, "note": f"unbound ({type(e).__name__})"}


def secondary_measurements(args, torch, dist, dev, stream, flush, rank, world):
    """Device-resident step time of the OTHER BASELINE.json configurations, measured exactly like `value` (CUDA events per
    step, L2 flushed in between, max over ranks), so that the driver's record carries them next to the headline workload.
    One GPU: configs[1], configs[2] and the per-GPU shard of configs[4] in both joint formulations. N GPUs: configs[4]
    weak-scaled like the headline (32 chains x 8 links per GPU; at N = 8 that is BASELINE's "256 instances sharded
    8 x B200"; whole chains per rank, no collective on the data path). Short runs: 10 steps each. Called by ALL ranks."""
    import copy
    pkg = importlib.import_module("3dobjecttracking_b200")
    capi = importlib.import_module("3dobjecttracking_b200.capi")
    out = {}
    todo = (("configs[4] projected", "c5", "projected"), ("configs[4] constrained", "c5", "constrained"))
    if world == 1:
        todo = (("configs[1]", "c2", None), ("configs[2]", "c3", None)) + todo
    for key, wname, variant in todo:
        a = copy.copy(args)
        a.workload, a.bodies = wname, None
        if variant:
            a.variant = variant
        try:
            _, wl = build_workload(a, rank)
            ctx = capi.context_from_workload(wl, device=dev.index, stream=stream.cuda_stream)
            ctx.start_modalities(0)
            poses = np.ascontiguousarray(wl.start_body2world.reshape(wl.n_bodies, 12))
            for _ in range(3):
                ctx.set_poses(poses); ctx.reset_joint_poses(); ctx.tracking_step(0, wl.n_corr_iterations, wl.n_update_iterations)
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier(device_ids=[dev.index])
            l0, evs = ctx.launch_count, []
            for _ in range(10):
                flush.zero_()
                ctx.set_poses(poses); ctx.reset_joint_poses()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                ctx.tracking_step(0, wl.n_corr_iterations, wl.n_update_iterations)
                e1.record(stream)
                evs.append((e0, e1))
            torch.cuda.synchronize(dev)
            ms = sum(x.elapsed_time(y) for x, y in evs) / len(evs)
            if world > 1:
                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            total_b = pkg.roofline.algorithmic_bytes_per_step(wl)[0]
            peak, _ = measured_peak_gbs()
            out[key] = {"workload": workload_description(wl, a), "n_gpus": world, "ms_per_step": ms,
                        "value": world * wl.n_bodies * wl.n_corr_iterations / (ms * 1e-3), "unit": UNIT,
                        "launches_per_step": (ctx.launch_count - l0) // 10,
                        "roofline_frac": total_b / (ms * 1e-3) / 1e9 / peak}
            ctx.close()
        except Exception as e:  # a secondary line must never take the headline down
            out[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
            if world > 1:
                raise  # ... except that ranks must not diverge inside collectives
    return out


def build_workload(args, rank, n_shards=1):
    """Bodies [rank*nb, (rank+n_shards)*nb) of the weak-scaled job (nb bodies per GPU)."""
    pkg = importlib.import_module("3dobjecttracking_b200")
    if args.workload == "c5":  # 8-link chains; --bodies counts links per GPU
        n_chains = (args.bodies or 256) // 8
        wl = pkg.synth.make_chain_workload(n_chains=n_chains * n_shards, n_links=8, n_lines=300, n_points=300,
                                           variant=args.variant, n_divides=4, seed=args.seed,
                                           first_chain=rank * n_chains)
        return pkg, wl
    nb = args.bodies or pkg.synth.PRESETS[args.workload]["n_bodies"]
    wl = pkg.synth.make_workload(args.workload, n_bodies=nb * n_shards, n_divides=4, seed=args.seed,
                                 first_body=rank * nb)
    return pkg, wl


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under load (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        if self.idx is None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


_THREADS = {}


def calibrate_threads(oracle_py, wl):
    """"All the host threads it can use": the OpenMP thread count that is fastest on this box among
    {affinity mask size, half of it (physical cores), cgroup CPU quota}; oversubscribing a cgroup-limited
    container makes the CPU arm slower, which would flatter the GPU arm."""
    if "n" in _THREADS:
        return _THREADS["n"]
    cands = set()
    try:
        n_aff = len(os.sched_getaffinity(0))
    except Exception:
        n_aff = os.cpu_count() or 1
    cands.update({n_aff, max(1, n_aff // 2)})
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            cands.add(max(1, int(float(q) / float(p))))
    except Exception:
        pass
    cands.add(oracle_py.lib(native=True).orc_max_threads())
    cands = sorted(c for c in cands if c >= 1)
    best, best_t = cands[0], None
    for c in cands:
        if c > max(1, len(wl.structures) if getattr(wl, "structures", None) else wl.n_bodies):
            continue
        trk = oracle_py.OracleTracker(wl, n_threads=c, native=True)
        trk.tracking_step(0)  # warm-up (thread pool)
        # sustained rate over >= 0.3 s of wall clock: this container has a cgroup CPU quota (cpu.max), so a thread count
        # that wins a single burst step can lose once the quota throttles it
        n, t_start = 0, time.perf_counter()
        while n < 2 or time.perf_counter() - t_start < 0.3:
            trk.set_poses(wl.start_body2world)
            trk.reset_joint_poses()
            trk.tracking_step(0)
            n += 1
        dt = (time.perf_counter() - t_start) / n
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    _THREADS["n"] = best
    return best


def cpu_reference_run(args, wl, steps, warmup, threads=None):
    """Times the oracle port (the reference's CPU algorithm; -O3 -march=native like M3T/CMakeLists.txt) on
    the host cores, OpenMP over bodies (how the reference parallelises independent runs,
    examples/rbot_evaluator.cpp:144). One step = the same full-batch tracking step the GPU arm times."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    if threads is None:
        threads = calibrate_threads(oracle_py, wl)
    trk = oracle_py.OracleTracker(wl, rotation_mode=oracle_py.ROTATION_POLAR, exp_mode=oracle_py.EXP_PADE,
                                  n_threads=threads, native=True)
    trk.start_modalities(0)
    phases = np.zeros(3)
    for _ in range(warmup):
        trk.set_poses(wl.start_body2world)
        trk.reset_joint_poses()
        trk.tracking_step(0)
    t_total, t_best = 0.0, None
    for _ in range(steps):
        trk.set_poses(wl.start_body2world)
        trk.reset_joint_poses()
        t0 = time.perf_counter()
        ph = trk.tracking_step(0)
        t = time.perf_counter() - t0
        t_total += t
        t_best = t if t_best is None else min(t_best, t)
        phases += np.array(ph[:3])
    its = wl.n_bodies * wl.n_corr_iterations * steps
    return {"value": its / t_total, "ms_per_step": 1e3 * t_total / steps, "cores": int(threads),
            "best_step_value": wl.n_bodies * wl.n_corr_iterations / t_best,
            "phase_split_cpu_seconds": {"correspondences": phases[0], "gradient_hessian": phases[1],
                                        "optimization": phases[2]}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # under torchrun only rank 0 runs the CPU arm
    pkg, wl = build_workload(args, 0, n_shards=args.gpus)  # the whole N-GPU job on this host's cores
    r = cpu_reference_run(args, wl, args.steps, args.warmup)
    total_b, *_ = pkg.roofline.algorithmic_bytes_per_step(wl)
    sample = f"{args.steps} full steps of the workload ({wl.n_bodies} bodies x {wl.n_corr_iterations} corr iterations each)"
    out = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(wl, args, args.gpus, wl.n_bodies // args.gpus),
        "arm_note": f"CPU arm: the whole {args.gpus}-GPU job ({wl.n_bodies} bodies) on this host's cores, OpenMP over bodies",
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample,
                         "best_step_value": r["best_step_value"],
                         "phase_split_cpu_seconds": r["phase_split_cpu_seconds"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(out))


def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank) if world > 1 else {"numa_node": None, "note": "single rank: unbound"}

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])

    pkg, wl = build_workload(args, rank)
    capi = importlib.import_module("3dobjecttracking_b200.capi")
    stream = torch.cuda.current_stream(dev)
    ctx = capi.context_from_workload(wl, device=local_rank, stream=stream.cuda_stream)
    ctx.start_modalities(0)  # histogram initialisation (once; not part of the timed step)
    ctx.synchronize()

    nb, n_corr, n_upd = wl.n_bodies, wl.n_corr_iterations, wl.n_update_iterations
    its_per_step = nb * n_corr
    start_poses = torch.from_numpy(np.ascontiguousarray(wl.start_body2world.reshape(nb, 12))).pin_memory()
    poses_np = start_poses.numpy()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step():
        ctx.tracking_step(0, n_corr, n_upd)

    # one sampler for the job (rank 0's GPU): a polling nvidia-smi per rank makes the ranks queue on the driver's
    # locks - at 8 ranks that stalled the host-side calls of the end-to-end loop to 33 ms per step
    sampler = ClockSampler(local_rank if rank == 0 and not os.environ.get("BENCH_NO_SAMPLER") else None)
    sampler.start()

    # ---------------- value: device-resident frames, CUDA events per step, L2 flushed between steps --------
    for _ in range(max(args.warmup, 3)):
        ctx.set_poses(poses_np)
        ctx.reset_joint_poses()
        step()
    torch.cuda.synchronize(dev)
    barrier()
    launches0 = ctx.launch_count
    evs = []
    for _ in range(args.steps):
        flush.zero_()
        ctx.set_poses(poses_np)
        ctx.reset_joint_poses()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step()
        e1.record(stream)
        evs.append((e0, e1))
    torch.cuda.synchronize(dev)
    launches = ctx.launch_count - launches0
    barrier()
    if args.dump_outputs:  # before the e2e and clock loops below move the poses on
        poses_out = torch.from_numpy(ctx.get_poses()).to(dev)
        if world > 1:  # equal shards in rank order: the whole job's bodies
            gathered_out = torch.empty((world * nb, 3, 4), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(gathered_out, poses_out)
            poses_out = gathered_out
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "poses.npy"), poses_out.cpu().numpy())
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * its_per_step / (ms_per_step * 1e-3)

    # ---------------- e2e: host buffers through the C ABI ------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        h_color = h_depth = None
        h2d = nb * 48
        if wl.region:
            h_color = torch.from_numpy(wl.color_frames).pin_memory()
            h2d += h_color.numel()
        if wl.depth:
            h_depth = torch.from_numpy(wl.depth_frames.view(np.uint8).reshape(nb, wl.depth_frames.shape[1], -1)).pin_memory()
            h2d += h_depth.numel()
        full_frame_bytes = h2d - nb * 48
        d2h = nb * 48
        out_poses = torch.empty((nb, 12), dtype=torch.float32).pin_memory()
        gathered = None
        if world > 1:  # persistent buffers of the per-frame pose all-gather (SURVEY §8e), on its own stream: the
            # tracking stream never queues behind the collective (r01: it was enqueued on the compute stream)
            poses_dev = torch.empty((nb, 12), dtype=torch.float32, device=dev)
            gathered = torch.empty((world * nb, 12), dtype=torch.float32, device=dev)
            gather_stream = torch.cuda.Stream(device=dev)

        def hand_over_frames():
            # Camera::UpdateImage for every camera (pinned frames: pointers only) + the optional prefetch: the ROI
            # ingest of these frames runs on a side stream while the step launched before is still tracking
            if h_color is not None:
                ctx.upload_batch_ptr(True, 0, nb, h_color.data_ptr(), h_color.stride(0), h_color.stride(1))
            if h_depth is not None:
                ctx.upload_batch_ptr(False, 0, nb, h_depth.data_ptr(), h_depth.stride(0), h_depth.stride(1))
            ctx.prefetch_frames()

        def e2e_step():
            # software pipeline, one frame deep: step t tracks the frames handed over during step t-1; the frames of
            # step t+1 are handed over (and start crossing PCIe) right after step t has been launched
            ctx.set_poses(poses_np)
            ctx.reset_joint_poses()
            step()
            hand_over_frames()
            ctx._ck(ctx.L.m3tb_get_poses(ctx.h, 0, nb, capi._p(out_poses.numpy())))  # synchronises the stream
            if world > 1:  # publish: NCCL all-gather of the solved poses, once per frame, not waited for by the next step
                with torch.cuda.stream(gather_stream):
                    poses_dev.copy_(out_poses, non_blocking=True)  # out_poses is complete: m3tb_get_poses synchronised
                    dist.all_gather_into_tensor(gathered, poses_dev)

        hand_over_frames()  # frame 0
        for _ in range(max(args.warmup, 3)):
            e2e_step()
        torch.cuda.synchronize(dev)
        barrier()
        t0 = time.perf_counter()
        step_ms = []
        for _ in range(args.steps):
            ts = time.perf_counter()
            e2e_step()
            step_ms.append(1e3 * (time.perf_counter() - ts))
        ctx.synchronize()  # includes the side stream: K steps tracked, K frame sets ingested inside the timed region
        if world > 1:
            gather_stream.synchronize()  # ... and K pose all-gathers completed
        if os.environ.get("BENCH_DEBUG_E2E"):
            print(f"[e2e debug] rank {rank}: per-step ms " + " ".join(f"{v:.2f}" for v in step_ms), file=sys.stderr, flush=True)
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        barrier()
        t = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item()) / args.steps
        moved = ctx.last_ingest_bytes()  # bytes the ROI frame ingest actually fetched in the last step
        if moved > 0:
            h2d = moved + nb * 48
        e2e = {"value": world * its_per_step / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s,
               "host_frame_bytes_per_step": int(full_frame_bytes), "host_binding": numa,
               "ingest": ("pinned frames, ROI-only zero-copy fetch (k_ingest): only the rectangle each body can touch "
                          "crosses PCIe; prefetched one frame ahead on a side stream (m3tb_prefetch_frames), so the copy "
                          "of step t+1's frames overlaps the tracking of step t" if moved > 0 else "full-frame copies")}

    # ---------------- clocks: keep the GPU under the same load for a while so nvidia-smi sees it ----------------
    t_end = time.perf_counter() + 1.5
    while time.perf_counter() < t_end:
        for _ in range(50):
            step()
        torch.cuda.synchronize(dev)
    clocks = sampler.stop()
    clocks["note"] = "sampled every 100 ms from before the timed region to the end of a 1.5 s repeat of the timed step"

    secondary = None
    if args.workload == "c4" and not args.bodies and not args.no_secondary:
        secondary = secondary_measurements(args, torch, dist, dev, stream, flush, rank, world)  # every rank takes part

    if rank == 0:
        total_b, region_b, depth_b, line_evals, point_evals = pkg.roofline.algorithmic_bytes_per_step(wl)
        peak, peak_src = measured_peak_gbs()
        kernel_s = ms_per_step * 1e-3  # rigid bodies: one k_track launch per step, the events bracket exactly that launch
        # (kinematic structures: k_track + k_structure per update iteration; the roofline is then quoted on the whole step)
        achieved = total_b / kernel_s / 1e9
        # DRAM traffic needs hardware counters (ncu); the capture is tied to the kernel sources it was taken from, so a
        # number measured on an older kernel is reported as null instead of silently going stale
        traffic, traffic_note = None, "no ncu capture on record for this workload"
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            key = args.workload if not args.bodies else f"{args.workload}-{args.bodies}"
            if key in tj:
                if tj.get("source_sha") == source_sha():
                    traffic, traffic_note = tj[key], tj.get("note", "")
                else:
                    traffic_note = (f"stale: profiles/traffic.json was captured from sources {tj.get('source_sha')}, "
                                    f"this build is {source_sha()} (last captured value {tj[key]:.4g} B/launch)")
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(wl, args, world, nb),
            "line_evals_per_s": world * line_evals / kernel_s,
            "depth_point_evals_per_s": world * point_evals / kernel_s,
            "roofline": {"bound": "hbm", "kernel": "k_track2<1024, true> (one fused launch per step; k_track serves what k_track2 does not take)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": total_b, "region_bytes": region_b, "depth_bytes": depth_b,
                         "launch_ms": ms_per_step},
            "clocks": clocks, "gpu_launches": int(launches),
        }
        if e2e:
            out["e2e"] = e2e
        if not args.no_parity_check:
            out["parity_check"] = parity_check(ctx, wl)
        if secondary is not None:
            out["secondary"] = secondary
        if world == 1 and not args.no_cpu_baseline:
            n_cpu_steps = max(3, min(50, int(0.5 / max(1e-4, ms_per_step * 1e-3 * 20))))  # ~0.5 s of sustained CPU work
            r = cpu_reference_run(args, wl, steps=n_cpu_steps, warmup=1)
            r1 = cpu_reference_run(args, wl, steps=1, warmup=0, threads=1)
            out["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                   "sample": f"{n_cpu_steps} full steps of the same workload ({nb} bodies x {n_corr} corr iterations), OpenMP over bodies, thread count chosen by sustained rate",
                                   "best_step_value": r["best_step_value"], "single_thread_value": r1["value"],
                                   "phase_split_cpu_seconds": r["phase_split_cpu_seconds"]}
        emit(json.dumps(out))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


_RESULT_OUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the result. Libraries write there too (NCCL prints its version banner on stdout at
    every debug level but NONE, OpenMP runtimes their warnings): keep a private handle on the real stdout for the result
    and point file descriptor 1 at stderr for everything else, in this process and its children."""
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
