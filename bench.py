#!/usr/bin/env python
"""bench.py — stereo pose solves/sec on KITTI-shaped synthetic input (BASELINE.json metric).

One *solve* = StereoFrameHandler::insertStereoPair's f2fTracking (4 matchNNR problems: points and lines,
both directions, + mutual filter) followed by optimizePose (stage-1 GN -> gate -> removeOutliers -> stage-2 GN
or robust fallback -> gate -> finalisation) on pre-extracted features (SURVEY.md 8(d)).
One *step* = one pass of that hot path over one batch of independent frame pairs.

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N ...            the reference's CPU implementation of the path
                                                           (the oracle port, all host threads), rank 0 only

Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM, CUDA events on the launching stream, max
over ranks.  `e2e`: the same metric through the C-ABI call with pinned HOST buffers, H2D and D2H inside the
timed region.  Weak scaling: every rank processes its own --pairs frame pairs, no data-path collective.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark writes nothing into the tree it runs from (which may be read-only)

from stvo_pl_b200 import synth, types as T  # noqa: E402

METRIC = "stereo pose solves/sec (KITTI-shape, 2k pts+500 lines)"
UNIT = "solves/s"
WORKLOAD = ("C2: synthetic KITTI-shape 1241x376, 2000 ORB pts + 500 LBD lines per frame, "
            "match (4 x matchNNR + mutual) + optimizePose to convergence")


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cgroup_cpu_quota():
    """CPUs the cgroup lets this process use (cpu.max of cgroup v2 / cfs_quota of v1), or None when unlimited or
    unreadable.  sched_getaffinity does not see such a quota: a 128-thread box can be leased with a fraction of it."""
    paths = []
    try:
        with open("/proc/self/cgroup") as f:
            for line in f:
                parts = line.strip().split(":", 2)
                if len(parts) == 3 and parts[0] == "0":
                    rel = parts[2].lstrip("/")
                    while True:
                        paths.append(os.path.join("/sys/fs/cgroup", rel, "cpu.max"))
                        if not rel:
                            break
                        rel = os.path.dirname(rel)
    except OSError:
        pass
    paths.append("/sys/fs/cgroup/cpu.max")
    best = None
    for p in paths:
        try:
            q, per = open(p).read().split()[:2]
            if q != "max":
                v = float(q) / float(per)
                best = v if best is None else min(best, v)
        except (OSError, ValueError):
            continue
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            best = q / per if best is None else min(best, q / per)
    except (OSError, ValueError):
        pass
    return best


def cpu_threads_to_use():
    """(threads, cores_visible, cores_quota): never more worker threads than the quota can run."""
    vis = host_threads()
    quota = cgroup_cpu_quota()
    use = vis if quota is None else max(1, min(vis, int(quota + 0.5)))
    return use, vis, quota


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# BASELINE.json configs that run through the same match + optimizePose pipeline (C4 = C2 sharded over ranks)
WORKLOADS = {
    "c2": ("kitti", T.kitti_config, 0, WORKLOAD),
    "c1": ("kitti_points", T.kitti_config, 0,
           "C1: KITTI-calibrated plumbing pairs, 2000 ORB points, no lines (synthetic: no KITTI images on the box)"),
    "c3": ("euroc", T.euroc_config, 1,
           "C3: synthetic EuRoC-shape 752x480, 1000 pts + 300 lines, robust weights on (MAD-scaled Cauchy, solver_mode 1)"),
}
ACTIVE = "c2"


def workload_config():
    shape, cfgf, mode, _ = WORKLOADS[ACTIVE]
    cfg = cfgf()
    cfg.solver_mode = mode
    if ACTIVE == "c1":
        cfg.has_lines = 0
    return cfg


def make_workload(pairs: int, first_pair: int):
    """The bench workload: every prev feature is re-observed in curr (overlap 1.0) so that the solver sees the
    named feature counts (C2: 2000 points + 500 lines); 10 % of the observations are gross outliers; descriptors of
    true correspondences differ in 10 % of their bits."""
    return synth.make_batch(WORKLOADS[ACTIVE][0], pairs, first_pair=first_pair, overlap=1.0)


class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (pynvml, ~4 ms period: a default run's timed region is
    only ~65 ms long)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.004)

    def __enter__(self):
        if self.ok:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.ok:
            self.t.join(timeout=1.0)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def measured_tensor_peak():
    """fp8 (e4m3) dense peak for the tensor roofline: MEASURED_PEAKS.json holds the cuBLAS bf16 burst figure; the 8-bit kinds
    run at twice the 16-bit rate on this part (nominal 4.5 vs 2.25 PFLOP/s), so 2 x the measured bf16 number is used."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return 2.0 * float(json.load(open(p))["bf16_tflops"]), "2 x measured cuBLAS bf16 burst (fp8 runs at twice the bf16 rate)"
        except Exception:
            pass
    return 2.0 * 1590.0, "2 x fallback bf16"


def ncu_traffic(name="k1_traffic.json"):
    """dram bytes per launch of a kernel from the committed ncu capture (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def cpu_leg(sample: int, budget_s: float = 25.0, min_reps: int = 5, max_reps: int = 20, first_pair: int = 0):
    """The reference's CPU implementation of the path on the box's host cores: the oracle (C restatement, built
    -O3 -march=native like the reference's CMakeLists.txt:18), one independent frame pair per worker thread.
    Protocol of SURVEY 8(d): warm-up, then up to `max_reps` timed repetitions of the same bounded sample (at least
    `min_reps`, stopping once `budget_s` of wall clock is spent); median and minimum reported.  The thread count is
    calibrated: a 1-thread run of the same work gives the per-core rate, and `cores_effective` = all-thread rate /
    1-thread rate says how many cores the lease really delivered (sched_getaffinity alone over-states a quota'd box).
    Also times the library the reference actually calls for matching, cv2.BFMatcher.knnMatch (src/matching.cpp:47-48),
    beside the oracle's own popcount loop on one 2000 x 2000 problem."""
    from oracle.oracle import Oracle
    orc = Oracle(native=True)
    threads, vis, quota = cpu_threads_to_use()
    prev, curr, _, cam = make_workload(sample, first_pair)
    cfg = workload_config()
    k1 = min(4, sample)
    one_p, one_c = prev.select(range(k1)), curr.select(range(k1))
    orc.track_batch(cam, cfg, one_p, one_c, threads=1)                               # warm-up, 1 thread
    t1 = []
    for _ in range(3):
        t0 = time.perf_counter()
        orc.track_batch(cam, cfg, one_p, one_c, threads=1)
        t1.append((time.perf_counter() - t0) / k1)
    per_pair_1t = float(np.median(t1))
    orc.track_batch(cam, cfg, prev, curr, threads=threads)                           # warm-up, all threads
    times, stage = [], np.zeros(2)
    t_start = time.perf_counter()
    while len(times) < max_reps and (len(times) < min_reps or time.perf_counter() - t_start < budget_s):
        t0 = time.perf_counter()
        r = orc.track_batch(cam, cfg, prev, curr, threads=threads)
        times.append(time.perf_counter() - t0)
        stage += r["stage_ms"]
    med, best = float(np.median(times)), float(np.min(times))
    rate = sample / med
    cpu_s = stage / 1e3 / len(times)                                                 # CPU seconds per repetition: [match, GN]
    eff = rate * per_pair_1t
    out = {"value": rate, "unit": UNIT, "kind": "port", "cores": threads, "cores_visible": vis,
           "cores_quota": quota, "cores_effective": eff, "cpu": cpu_model(),
           "reps": len(times), "value_median": rate, "value_best": sample / best,
           "ms_per_rep": {"median": med * 1e3, "min": best * 1e3, "max": float(np.max(times)) * 1e3},
           "one_thread_ms_per_pair": per_pair_1t * 1e3,
           "match_share": float(stage[0] / max(stage.sum(), 1e-9)),
           "rates": {"unit": UNIT, "match_only": sample / max(cpu_s[0] / max(eff, 1e-9), 1e-12),
                     "gn_only": sample / max(cpu_s[1] / max(eff, 1e-9), 1e-12),
                     "note": "stage CPU time of the same repetitions divided over cores_effective"},
           "sample": f"{sample} frame pairs of the same workload, one pair per thread on {threads} threads, "
                     f"{len(times)} repetitions of {med:.2f} s (median); {stage.sum() / 1e3 / len(times):.1f} s of CPU work each"}
    # matching alone, one thread, one points-sized problem: OpenCV's BFMatcher (what the reference calls) vs the oracle's loop
    a = prev.pdesc[int(prev.pt_off[0]):int(prev.pt_off[1])]
    b = curr.pdesc[int(curr.pt_off[0]):int(curr.pt_off[1])]
    if len(a) and len(b):
        tt = []
        for _ in range(23):
            t0 = time.perf_counter()
            orc.match_nnr(a, b, 0.75)
            tt.append(time.perf_counter() - t0)
        out["match_nnr_ms"] = {"shape": [int(len(a)), int(len(b))], "oracle_popcount_loop": {"median": float(np.median(tt[3:])) * 1e3,
                                                                                              "min": float(np.min(tt[3:])) * 1e3}}
        try:
            import cv2
            cv2.setNumThreads(1)
            bf = cv2.BFMatcher(cv2.NORM_HAMMING, False)
            tt = []
            for _ in range(23):
                t0 = time.perf_counter()
                bf.knnMatch(a, b, 2)
                tt.append(time.perf_counter() - t0)
            out["match_nnr_ms"]["cv2_bfmatcher_knnmatch"] = {"median": float(np.median(tt[3:])) * 1e3, "min": float(np.min(tt[3:])) * 1e3,
                                                             "version": cv2.__version__}
        except Exception as e:   # cv2 absent on the box: say so, keep the oracle's figure
            out["match_nnr_ms"]["cv2_bfmatcher_knnmatch"] = {"unavailable": str(e)[:80]}
    # one pair with the reference's own threading inside a pair (points || lines, 1->2 || 2->1)
    lat = []
    for k in range(min(5, sample)):
        t0 = time.perf_counter()
        orc.track_batch(cam, cfg, prev.select([k]), curr.select([k]), faithful=True)
        lat.append((time.perf_counter() - t0) * 1e3)
    out["single_pair_latency_ms"] = float(np.median(lat))
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores.  The
    reference project cannot be built here (Eigen / OpenCV C++ / Boost / yaml-cpp absent), so this is the oracle
    port (oracle/plstvo_oracle.c; pinned against the reference's compiled pose code, tests/test_oracle_ref.py),
    all usable host threads, one independent pair per thread.  --steps bounds the repetitions."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads, _, _ = cpu_threads_to_use()
    sample = max(32, 2 * threads)
    cb = cpu_leg(sample, budget_s=40.0, min_reps=3, max_reps=max(3, min(args.steps, 20)))
    value = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": cb["reps"], "warmup": 1, "ms_per_step": cb["ms_per_rep"]["median"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
        "config": {"workload": WORKLOADS[ACTIVE][3], "pairs_per_gpu": args.pairs, "pairs_per_step_cpu_sample": sample,
                   "note": "CPU oracle port of the reference path on a bounded sample of the same workload; N GPUs are not used by this arm"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def run_ours(args):
    import torch
    import torch.distributed as dist
    from stvo_pl_b200.engine import Engine, bind_to_gpu_numa

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL writes its version banner to stdout when NCCL_DEBUG is set on the box; stdout carries exactly one JSON
        # line, so the communicator is set up with fd 1 pointed at stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # pinned buffers are allocated with the process bound to the GPU's NUMA node (at N = 1 too: the 1-GPU lease may sit on
    # either socket); the affinity is restored afterwards so that the cpu_baseline leg still sees every usable core
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local)
    eng = Engine(local)
    cfg = workload_config()
    B = args.pairs
    prev, curr, Tgt, cam = make_workload(B, first_pair=rank * B)   # weak scaling: own pairs per rank

    # ---------------- value: inputs resident in HBM ----------------
    db = eng.upload(cam, cfg, prev, curr)
    if args.kernels_only:
        db.kernel_times(iters=1)      # first launches pay module load / local-memory setup: keep them out
        print(json.dumps(db.kernel_times(iters=2)), flush=True)
        db.free()
        eng.close()
        return 0
    for _ in range(max(args.warmup, 3)):
        db.run()
    eng.synchronize()
    launches0 = eng.launches
    barrier()
    with ClockSampler(local) as clk:
        ms = db.run_timed(args.steps, flush_l2=False)
    barrier()
    launches = eng.launches - launches0
    ms = max_over_ranks(ms)
    value = world * B * args.steps / (ms * 1e-3)
    out = db.download()
    good = int(out["results"]["good"].sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, prev)

    # ---------------- per-kernel times and the roofline of the dominant kernel, rank 0 ----------------
    st = db.stage_times(iters=max(5, min(args.steps, 20)))
    kt = {"ms_match": st["ms_expand"] + st["ms_distance"] + st["ms_resolve"], "ms_solve": st["ms_solve"], "n_tiles": st["n_items"]}
    n1p = int(prev.pt_off[-1]); n1l = int(prev.ls_off[-1]); n2p = int(curr.pt_off[-1]); n2l = int(curr.ls_off[-1])
    k1_bytes = 32 * (n1p + n2p + n1l + n2l) + 4 * (n1p + n1l)          # descriptors in + match indices out
    n_mp, n_ml = int(out["results"]["n_matched_pt"].sum()), int(out["results"]["n_matched_ls"].sum())
    k2_bytes = 32 * n_mp + 64 * n_ml + 632 * B                          # matched records in (fp32-packed size) + results out
    step_bytes = k1_bytes + k2_bytes                                    # SURVEY 8(d) compulsory bytes per solve, summed
    peak, peak_kind = measured_peak()
    tpeak, tpeak_kind = measured_tensor_peak()
    pair_dists = sum(int((prev.pt_off[p + 1] - prev.pt_off[p])) * int((curr.pt_off[p + 1] - curr.pt_off[p])) +
                     int((prev.ls_off[p + 1] - prev.ls_off[p])) * int((curr.ls_off[p + 1] - curr.ls_off[p]))
                     for p in range(B))
    step_ms = sum(st[k] for k in ("ms_expand", "ms_distance", "ms_resolve", "ms_solve"))
    tc_flops = 2.0 * 256 * pair_dists
    kernels = {
        "tc_expand_kernel": {"ms": st["ms_expand"], "bound": "hbm", "algorithmic_bytes": 9 * 32 * (n1p + n2p + n1l + n2l),
                             "note": "32 B descriptor in, 256 B e4m3 operand row out"},
        ("tc_hamming_kernel" if st["tensor_core_form"] else "hamming_knn2_kernel"):
            {"ms": st["ms_distance"], "bound": "tensor" if st["tensor_core_form"] else "alu", "flops": tc_flops,
             "pair_distances": pair_dists, "work_items": st["n_items"]},
        "tc_resolve_kernel": {"ms": st["ms_resolve"], "bound": "latency"},
    }
    if st["streamed_solver"]:
        evals = int(out["results"]["iters_stage1"].sum() + out["results"]["iters_stage2"].sum())
        rec = 32 * n_mp + 64 * n_ml
        kernels["stream_prepare_kernel"] = {
            "ms": st["ms_lists"], "bound": "latency (block-wide compaction steps)", "ctas": B,
            "algorithmic_bytes": 8 * (n1p + n1l) + 56 * n_mp + 136 * n_ml + rec,
            "note": "match finish (partials in, m12 out) + f2fTracking lists (fp64) + fp32 records"}
        gn_ms = st["ms_gn_stage1"] + st["ms_gn_stage2"]
        kernels["gn_loop_stream_kernel"] = {
            "ms": gn_ms, "launches": 2, "bound": "fp32 issue / latency (records resident in shared memory at this size)", "ctas": B,
            "evaluations": evals, "algorithmic_bytes": 2 * rec,
            "note": "stage 1 + stage 2 launches; the records of a KITTI-size problem (4 + 2 tiles of 16 KB) are loaded once per "
                    "launch and stay in shared memory for its iterations"}
        kernels["stream_outlier_kernel"] = {"ms": st["ms_outliers"], "bound": "latency (block-wide selection steps)", "ctas": B,
                                            "algorithmic_bytes": 56 * n_mp + 136 * n_ml}
        kernels["stream_finalize_kernel + handed-back problems"] = {
            "ms": max(st["ms_optimize_pose"] - gn_ms - st["ms_outliers"], 0.0), "bound": "latency", "algorithmic_bytes": 632 * B,
            "delegated_to_fp64": st["delegated_to_fp64"]}
    else:
        kernels["track_solve_kernel"] = {"ms": st["ms_solve"], "bound": "latency (fp64 pipe in its evaluations)",
                                         "algorithmic_bytes": k2_bytes, "ctas": B}
    for k in kernels.values():
        k["share_of_step"] = k["ms"] / step_ms if step_ms > 0 else 0.0
    dom_name = max(kernels, key=lambda n: kernels[n]["ms"])
    dom = kernels[dom_name]
    traffic = ncu_traffic("k_traffic.json") or {}
    if dom["bound"] == "tensor":
        achieved = tc_flops / (dom["ms"] * 1e-3) / 1e12
        roofline = {"kernel": dom_name, "bound": "tensor", "achieved": achieved, "peak": tpeak, "unit": "TFLOP/s",
                    "frac": achieved / tpeak, "peak_kind": tpeak_kind,
                    "traffic": (traffic.get(dom_name) or {}).get("dram_bytes_per_launch"),
                    "algorithmic_flops_per_launch": tc_flops, "ms_per_launch": dom["ms"],
                    "note": "2 x 256 flop per 256-bit pair distance (the +-1 contraction); the kernel is bound by its top-2 epilogue "
                            "on the ALU pipe (3 packed min/max per two distances and direction), not by the tensor pipe: see `pipes`"}
    else:
        alg = dom.get("algorithmic_bytes", k2_bytes)
        achieved = alg / (dom["ms"] * 1e-3) / 1e9
        roofline = {"kernel": dom_name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_kind": f"of {peak_kind}", "traffic": (traffic.get(dom_name) or {}).get("dram_bytes_per_launch"),
                    "algorithmic_bytes_per_launch": alg, "ms_per_launch": dom["ms"],
                    "note": "one persistent CTA per pair: ~16 dependent evaluate -> reduce -> 6x6 solve rounds; latency-bound, far from "
                            "the HBM roofline by construction (features are read once into shared memory)"}
    roofline["share_of_step"] = dom["share_of_step"]
    roofline["kernels"] = kernels
    roofline["pipes"] = traffic.get("pipes")
    roofline["tensor"] = {"kernel": "tc_hamming_kernel", "achieved": tc_flops / (st["ms_distance"] * 1e-3) / 1e12, "peak": tpeak,
                          "unit": "TFLOP/s", "frac": tc_flops / (st["ms_distance"] * 1e-3) / 1e12 / tpeak, "peak_kind": tpeak_kind,
                          "pair_distances_per_s": pair_dists / (st["ms_distance"] * 1e-3)} if st["tensor_core_form"] else None
    roofline["rates"] = {"unit": UNIT, "match_only": B / (kt["ms_match"] * 1e-3), "gn_only": B / (kt["ms_solve"] * 1e-3),
                         "note": "resident inputs, each stage's kernels timed alone over the whole batch"}
    roofline["step"] = {"algorithmic_bytes": step_bytes, "achieved": step_bytes * args.steps / (ms * 1e-3) / 1e9,
                        "frac": step_bytes * args.steps / (ms * 1e-3) / 1e9 / peak}
    # spread of single steps (the contract's `value` is the mean over the K timed steps above)
    singles = sorted(db.run_timed(1, flush_l2=False) for _ in range(20))
    spread = {"single_step_ms": {"min": singles[0], "median": singles[len(singles) // 2], "max": singles[-1]}, "reps": len(singles)}
    db.free()

    # ---------------- e2e: host buffers through the C-ABI, H2D + D2H inside the timed region ----------------
    pprev, pcurr = eng.pinned.pin_frames(prev), eng.pinned.pin_frames(curr)
    # PCIe probe: one copy of the step's input byte count out of the library's own pinned allocator (same NUMA node as the
    # frames above), best of 6 — the floor of any e2e step
    nbytes_in = int(prev.input_bytes("prev") + curr.input_bytes("curr"))
    psrc = torch.from_numpy(eng.pinned.empty((nbytes_in,), np.uint8))
    pdst = torch.empty(nbytes_in, dtype=torch.uint8, device=f"cuda:{local}")
    h2d_ms = 1e9
    for _ in range(6):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        pdst.copy_(psrc, non_blocking=True)
        ev1.record()
        torch.cuda.synchronize()
        h2d_ms = min(h2d_ms, ev0.elapsed_time(ev1))
    del pdst
    pouts = [eng.pinned_outputs(prev), eng.pinned_outputs(prev)]
    pout = pouts[0]
    # (a) the synchronous call, one batch at a time: returns when the results are in host memory
    for _ in range(max(args.warmup, 3)):
        eng.track_batch(cam, cfg, pprev, pcurr, out=pout)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.track_batch(cam, cfg, pprev, pcurr, out=pout)
    torch.cuda.synchronize()
    sync_s = time.perf_counter() - t0
    barrier()
    sync_s = max_over_ranks(sync_s)
    same = (pout["results"].tobytes() == out["results"].tobytes())
    # (a') latency of one blocking call on ONE frame pair: what a per-frame caller of insertStereoPair() / optimizePose() sees
    one_p, one_c = eng.pinned.pin_frames(prev.select([0])), eng.pinned.pin_frames(curr.select([0]))
    one_out = eng.pinned_outputs(prev.select([0]))
    os.sched_setaffinity(0, affinity0)          # every pinned buffer exists now: give the cores back
    lat = []
    for k in range(60):
        t1 = time.perf_counter()
        eng.track_batch(cam, cfg, one_p, one_c, out=one_out)
        lat.append((time.perf_counter() - t1) * 1e3)
    single_ms = float(np.median(lat[10:]))
    # (b) the streaming call (plstvo_track_batch_async / plstvo_wait), two batches in flight: step k+1's H2D overlaps
    # step k's kernels.  Every step still uploads its inputs and reads back its results inside the timed region.
    for k in range(max(args.warmup, 3)):
        eng.wait(eng.track_batch_async(cam, cfg, pprev, pcurr, pouts[k & 1]))
    barrier()
    t0 = time.perf_counter()
    pending = None
    for k in range(args.steps):
        tk = eng.track_batch_async(cam, cfg, pprev, pcurr, pouts[k & 1])
        if pending is not None:
            eng.wait(pending)
        pending = tk
    eng.wait(pending)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_s = max_over_ranks(e2e_s)
    e2e_value = world * B * args.steps / e2e_s
    same = same and all(po["results"].tobytes() == out["results"].tobytes() for po in pouts)
    h2d = prev.input_bytes("prev") + curr.input_bytes("curr")
    d2h = B * T.POSE_RESULT_DTYPE.itemsize + 4 * (n1p + n1l) + (n1p + n1l)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("u8 matching (as e4m3 +-1 on the tensor cores, f16 accumulators: exact); solve: f32 per feature, f64 sums / 6x6 algebra / "
                  "SE(3) / outlier statistics (streamed solver)") if st["streamed_solver"] else "u8 matching (e4m3 +-1, f16 accumulators: exact); solve: f64",
        "data": "synthetic",
        "config": {"workload": WORKLOADS[ACTIVE][3], "pairs_per_gpu": B, "solver": "streamed" if st["streamed_solver"] else "K2 (fp64)", "global_pairs_per_step": world * B,
                   "parallelism": f"independent pairs sharded over {world} GPU(s), no collective",
                   "l2": f"inputs larger than L2: {(h2d + kt['n_tiles'] * 0) / 1e6:.0f} MB of inputs + "
                         f"{B * 140000 / 1e6:.0f} MB of tile partials per pass vs 126 MB L2",
                   "overlap": 1.0, "outlier_frac": 0.10, "solved_ok": good, "e2e_equals_resident": bool(same),
                   "numa_bound": numa},
        "clocks": clk.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_s / args.steps * 1e3,
                "mode": "plstvo_track_batch_async + plstvo_wait, 2 batches in flight (pinned host buffers)",
                "sync_value": world * B * args.steps / sync_s, "sync_ms_per_step": sync_s / args.steps * 1e3,
                "sync_mode": "plstvo_track_batch, one blocking call per step",
                "single_pair_latency_ms": single_ms,
                "h2d_only_ms_per_step": h2d_ms, "h2d_only_gbs": h2d / (h2d_ms * 1e-3) / 1e9,
                "h2d_gbs_inside_pipelined_loop": h2d / (e2e_s / args.steps) / 1e9,
                "bound": "PCIe" if h2d_ms > 0.8 * (e2e_s / args.steps * 1e3) else "kernels",
                "note": "h2d_only_*: one pinned cudaMemcpy of the step's input bytes alone (the PCIe floor of a step); "
                        "h2d_gbs_inside_pipelined_loop: the same bytes over the pipelined step time (a lower bound of the link rate)"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "spread": spread,
    }
    # ---------------- C4 as BASELINE.json states it: 512 pairs IN TOTAL cut into 512 / N per GPU (strong scaling) ----------------
    STRONG_TOTAL = 512
    Bs = max(1, STRONG_TOTAL // world)
    if world == 1 and B == STRONG_TOTAL:
        line["strong"] = {"pairs_total": STRONG_TOTAL, "pairs_per_gpu": B, "value": value, "ms_per_step": ms / args.steps,
                          "e2e_value": e2e_value, "e2e_ms_per_step": e2e_s / args.steps * 1e3, "note": "N = 1: the run above"}
    else:
        sp, sc = prev.select(range(min(Bs, B))), curr.select(range(min(Bs, B)))
        sdb = eng.upload(cam, cfg, sp, sc)
        for _ in range(5):
            sdb.run()
        eng.synchronize()
        ssteps = max(args.steps, 50)
        barrier()
        sms = sdb.run_timed(ssteps, flush_l2=False)
        barrier()
        sms = max_over_ranks(sms)
        sst = sdb.stage_times(iters=5)
        sdb.free()
        spp, spc = eng.pinned.pin_frames(sp), eng.pinned.pin_frames(sc)
        spo = [eng.pinned_outputs(sp), eng.pinned_outputs(sp)]
        for k in range(4):
            eng.wait(eng.track_batch_async(cam, cfg, spp, spc, spo[k & 1]))
        barrier()
        t0 = time.perf_counter()
        pending = None
        for k in range(ssteps):
            tk = eng.track_batch_async(cam, cfg, spp, spc, spo[k & 1])
            if pending is not None:
                eng.wait(pending)
            pending = tk
        eng.wait(pending)
        torch.cuda.synchronize()
        se2e = time.perf_counter() - t0
        barrier()
        se2e = max_over_ranks(se2e)
        nb = sp.B
        line["strong"] = {"pairs_total": nb * world, "pairs_per_gpu": nb, "steps": ssteps,
                          "value": world * nb * ssteps / (sms * 1e-3), "ms_per_step": sms / ssteps,
                          "e2e_value": world * nb * ssteps / se2e, "e2e_ms_per_step": se2e / ssteps * 1e3,
                          "stage_ms": {k: sst[k] for k in ("ms_expand", "ms_distance", "ms_resolve", "ms_solve")},
                          "note": "strong scaling of the named config: the same 512 pairs in total, 512 / N per GPU; compare with the "
                                  "N = 1 line's value / e2e.value (efficiency = value(N) / (N x value(1)) is the driver's to compute)"}
    if world == 1 and rank == 0 and not args.no_cpu:
        threads, _, _ = cpu_threads_to_use()
        line["cpu_baseline"] = cpu_leg(max(32, 2 * threads), budget_s=20.0)
    if world == 1 and rank == 0 and not args.no_hbm_run and ACTIVE == "c2":
        # the HBM-bound part of the path measured in the same run, THROUGH THE PRODUCT ENTRY POINTS: BASELINE config C5
        # (8000 + 2000 features per frame) matched and solved; its solve stage streams the matched records from HBM
        line["c5_pipeline"] = c5_pipeline(eng, 384)
        # ... and the sweep kernel alone (1024 problems resident, 20 back-to-back sweeps)
        _, roof, _, _ = c5_sweeps(eng, 1024)
        line["roofline_hbm_kernel"] = roof
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_LIMIT = 64 << 20


def dump_outputs(path, out, prev):
    """Writes what the caller of the timed path receives after its last step (plstvo_batch_download: the pose results and the
    match / inlier arrays) as float64 .npy files, one per array and per field of the results.  Beyond DUMP_LIMIT bytes only a
    fixed, seeded sample of the frame pairs is written; pairs.npy names them."""
    res = out["results"]
    B = len(res)
    pairs = np.arange(B)
    values = sum(int(np.prod(res.dtype[k].shape)) for k in res.dtype.names) + 2 * (len(out["m12_pt"]) + len(out["m12_ls"])) / B
    per_pair = 8 * values
    if B * per_pair > DUMP_LIMIT:
        keep = int((DUMP_LIMIT - (1 << 20)) // per_pair)      # 1 MB left for the .npy headers and pairs.npy
        pairs = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    arrays = {f"results_{k}": res[k][pairs] for k in res.dtype.names}
    for kind, off in (("pt", prev.pt_off), ("ls", prev.ls_off)):
        idx = np.concatenate([np.arange(off[p], off[p + 1]) for p in pairs] + [np.zeros(0, np.int64)])
        arrays[f"m12_{kind}"], arrays[f"inlier_{kind}"] = out[f"m12_{kind}"][idx], out[f"inlier_{kind}"][idx]
    arrays["pairs"] = pairs
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(a, np.float64))


def c5_sweeps(eng, B, iters=20):
    """BASELINE config C5: high-density 1920x1080 synthetic, 8000 pts + 2000 lines per problem, `iters` GN evaluations with
    the packed matched lists of B >= 1024 problems resident in HBM (393 MB per sweep, far beyond the 126 MB L2) so that every
    evaluation streams from HBM.  Returns (seconds per sweep, roofline object, mean error, clocks)."""
    mb, Ts, cam = synth.make_matched_batch("hd", B)
    cfg = T.kitti_config()
    eng.gn_eval_stream(cam, cfg, mb, Ts, iters=2)                      # warm-up (uploads, packing, first launches)
    with ClockSampler(0) as clk:
        H, g, e, ms = eng.gn_eval_stream(cam, cfg, mb, Ts, iters=iters)
    n, m = int(mb.pt_off[-1]), int(mb.ls_off[-1])
    alg = 32 * n + 64 * m                                              # SURVEY 8(d): 32 N_p + 64 N_l per evaluation
    peak, kind = measured_peak()
    per = ms / iters * 1e-3
    tr = ncu_traffic("gn_traffic.json")
    roof = {"kernel": "gn_eval_stream_kernel", "bound": "hbm", "achieved": alg / per / 1e9, "peak": peak, "unit": "GB/s",
            "frac": alg / per / 1e9 / peak, "peak_kind": f"{kind}, burst (kernel timed alone, {iters} back-to-back sweeps, each = the streaming kernel + the per-problem reduce launch)", "traffic": tr["dram_bytes_per_launch"] if tr and tr.get("problems") == B else None,
            "algorithmic_bytes_per_launch": alg, "problems_resident": B, "ms_per_sweep": ms / iters}
    return per, roof, float(np.mean(e)), clk.summary()


def tile_batch(fb, reps):
    """reps copies of a FrameBatch one after the other (timing workloads only: cuts the synthetic-data generation time)."""
    if reps <= 1:
        return fb
    B = fb.B
    return fb.select([i % B for i in range(B * reps)])


def c5_pipeline(eng, B, steps=3, distinct=128):
    """BASELINE config C5 through the PRODUCT path (plstvo_batch_upload / plstvo_batch_run): 1920x1080, 8000 points + 2000 lines per
    frame, f2fTracking (8000 x 8000 and 2000 x 2000 Hamming problems, both directions) + optimizePose with the KITTI solver
    parameters.  Lists of this size do not fit K2's shared memory: the solve runs as evaluation sweeps streamed from HBM
    (gn_eval_stream_kernel) with a per-problem step kernel in between.  Returns the bench object: stage times, solves/s, and the
    HBM roofline of the solve computed from THIS run: bytes = sum over problems of evaluations x (32 n_pt + 64 n_ls)."""
    cfg = T.kitti_config()
    reps = max(1, B // distinct)
    prev, curr, Tgt, cam = synth.make_batch("hd", min(B, distinct), overlap=1.0)
    prev, curr = tile_batch(prev, reps), tile_batch(curr, reps)
    B = prev.B
    db = eng.upload(cam, cfg, prev, curr)
    for _ in range(2):
        db.run()
    eng.synchronize()
    with ClockSampler(0) as clk:
        ms = db.run_timed(steps, flush_l2=False) / steps
    st = db.stage_times(iters=steps)
    out = db.download()
    db.free()
    res = out["results"]
    evals = res["iters_stage1"].astype(np.int64) + res["iters_stage2"].astype(np.int64)
    per_eval = 32 * res["n_matched_pt"].astype(np.int64) + 64 * res["n_matched_ls"].astype(np.int64)
    alg = int((evals * per_eval).sum())                       # bytes the sweeps of one step have to stream
    sweep_bytes = int(per_eval.sum())                         # one sweep over every problem
    peak, kind = measured_peak()
    tr = ncu_traffic("c5_traffic.json") or {}
    solve_s = st["ms_optimize_pose"] * 1e-3
    gn_s = (st["ms_gn_stage1"] + st["ms_gn_stage2"]) * 1e-3
    return {"workload": "C5: 1920x1080, 8000 pts + 2000 lines per frame, match + optimizePose (KITTI solver parameters), "
                        f"{B} pairs resident ({min(B, distinct)} distinct, repeated)",
            "pairs": B, "ms_per_step": ms, "value": B / (ms * 1e-3), "unit": UNIT, "solved_ok": int(res["good"].sum()),
            "stage_ms": {k: st[k] for k in ("ms_expand", "ms_distance", "ms_resolve", "ms_lists", "ms_optimize_pose", "ms_gn_stage1",
                                          "ms_outliers", "ms_gn_stage2")},
            "streamed_solver": st["streamed_solver"],
            "evaluations_per_solve": {"mean": float(evals.mean()), "min": int(evals.min()), "max": int(evals.max())},
            "clocks": clk.summary(),
            "roofline": {"kernel": "gn_loop_stream_kernel (the two GN launches of optimizePose)",
                         "bound": "hbm", "achieved": alg / gn_s / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / gn_s / 1e9 / peak, "peak_kind": f"of {kind}",
                         "algorithmic_bytes_per_step": alg, "bytes_per_sweep": sweep_bytes,
                         "l2": f"{sweep_bytes / 1e6:.0f} MB per sweep vs 126 MB L2",
                         "traffic": tr.get("dram_bytes_per_launch"),
                         "traffic_of": "one stage-2 launch over the first half of the batch (ncu --set full, profiles/c5_traffic.json); "
                                       f"its algorithmic bytes: {int((res['iters_stage2'][:B // 2].astype(np.int64) * per_eval[:B // 2]).sum())}",
                         "ms_gn_loops": gn_s * 1e3,
                         "ms_optimize_pose": st["ms_optimize_pose"], "ms_outliers": st["ms_outliers"],
                         "frac_of_optimize_pose": alg / solve_s / 1e9 / peak,
                         "frac_including_list_building": alg / ((st["ms_lists"] + st["ms_optimize_pose"]) * 1e-3) / 1e9 / peak,
                         "traffic_note": "DRAM traffic below the algorithmic bytes = L2 reuse: the records of one 256-pair chunk (98 MB) stay "
                                         "in the 126 MB L2 from one iteration to the next",
                         "note": "bytes = evaluations that actually ran x record bytes (32 B / point, 64 B / line); time = the two "
                                 "gn_loop_stream_kernel launches (CUDA events around each).  frac_of_optimize_pose divides the same bytes "
                                 "by everything after matched_pt / matched_ls exist (GN loops, gate + removeOutliers, finalisation); "
                                 "ms_lists (f2fTracking's list building + record packing) is reported separately"}}


def run_c5_pipeline(args):
    """BASELINE config C5 through the product path, as its own bench line."""
    from stvo_pl_b200.engine import Engine
    eng = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    obj = c5_pipeline(eng, max(args.pairs, 384), steps=max(3, min(args.steps, 10)))
    line = {"metric": "stereo pose solves/sec (C5 shape, 8000 pts + 2000 lines)", "value": obj["value"], "unit": UNIT, "n_gpus": 1,
            "steps": max(3, min(args.steps, 10)), "warmup": 2, "ms_per_step": obj["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 matching; f32 per-feature / f64 sums and 6x6 in the solve",
            "data": "synthetic", "config": {"workload": obj["workload"], "pairs_per_gpu": obj["pairs"]},
            "clocks": obj["clocks"], "stage_ms": obj["stage_ms"], "evaluations_per_solve": obj["evaluations_per_solve"],
            "roofline": obj["roofline"]}
    print(json.dumps(line), flush=True)
    eng.close()
    return 0


def run_c5(args):
    """The HBM-roofline run of the streamed GN evaluation alone (the sweep kernel of config C5) as its own bench line."""
    from stvo_pl_b200.engine import Engine
    eng = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    B = max(args.pairs, 1024)
    iters = 20
    per, roof, mean_err, clocks = c5_sweeps(eng, B, iters)
    line = {"metric": "GN evaluation sweeps (C5: 8000 pts + 2000 lines per problem)", "value": B / per, "unit": "problem-evaluations/s",
            "n_gpus": 1, "steps": iters, "warmup": 2, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 per feature, f64 reduction", "data": "synthetic",
            "config": {"workload": "C5: 1920x1080, 8000 pts + 2000 lines, 20 GN evaluations streamed from HBM",
                       "problems_resident": B, "l2": f"{roof['algorithmic_bytes_per_launch'] * 1e-6:.0f} MB streamed per sweep vs 126 MB L2"},
            "clocks": clocks, "gpu_launches": 2 * iters, "roofline": dict(roof, mean_err=mean_err)}
    print(json.dumps(line), flush=True)
    eng.close()
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# --workload stereo: the widened rows (SURVEY 8(f)-1, -2) measured to the same bar: StereoFrame::matchStereoPoints +
# matchStereoLines (grid cells -> matchGrid -> 3-D lifting) for a batch of KITTI-shape frames, host buffers in and out.
def stereo_frames(B, first=0):
    from stvo_pl_b200 import stereo_synth as SS
    pts = [SS.make_stereo_frame_points(2000, 2000, seed=9000 + first + i) for i in range(B)]
    lns = [SS.make_stereo_frame_lines(500, 500, seed=19000 + first + i) for i in range(B)]
    return pts, lns


def stereo_cpu_rate(pts, lns, threads):
    """The oracle (orc_stereo_batch: cells as the reference's caller forms them, matchGrid, lifting), one frame per host thread."""
    from oracle.oracle import Oracle
    orc = Oracle(native=True)
    cam, mc, sc = T.kitti_camera(), T.default_stereo_match_config(), T.default_stereo_config()
    B = len(pts)
    pl_off = np.concatenate([[0], np.cumsum([len(f[0]) for f in pts])]).astype(np.int32)
    pr_off = np.concatenate([[0], np.cumsum([len(f[3]) for f in pts])]).astype(np.int32)
    ll_off = np.concatenate([[0], np.cumsum([len(f[0]) for f in lns])]).astype(np.int32)
    lr_off = np.concatenate([[0], np.cumsum([len(f[4]) for f in lns])]).astype(np.int32)
    P = [np.concatenate([f[j] for f in pts]) for j in range(5)]
    L = [np.concatenate([f[j] for f in lns]) for j in range(6)]
    args = (cam, mc, sc, pl_off, P[0], P[1], P[2], pr_off, P[3], P[4], ll_off, L[0], L[1], L[2], L[3], lr_off, L[4], L[5])
    orc.stereo_batch(*args, threads=threads)                    # warm-up
    best, n = 1e9, 0
    for _ in range(3):
        t0 = time.perf_counter()
        n = int(orc.stereo_batch(*args, threads=threads).sum())
        best = min(best, time.perf_counter() - t0)
    return B / best, best, n


def run_stereo(args):
    import torch
    from stvo_pl_b200.engine import Engine
    metric, unit = "stereo frames matched + lifted/sec (KITTI-shape, 2k+2k pts, 500+500 lines)", "frames/s"
    threads = host_threads()
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        pts, lns = stereo_frames(max(256, 8 * threads))
        rate, dt, _ = stereo_cpu_rate(pts, lns, threads)
        line = {"impl": "reference", "metric": metric, "value": rate, "unit": unit, "n_gpus": args.gpus, "steps": 1, "warmup": 1,
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64",
                "data": "synthetic", "config": {"workload": "stereo: matchStereoPoints + matchStereoLines", "frames_per_step": len(pts)},
                "cpu_baseline": {"value": rate, "unit": unit, "cores": threads, "kind": "port", "cpu": cpu_model(),
                                 "sample": f"{len(pts)} frames, one frame per thread (oracle composition)"},
                "e2e": {"value": rate, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return 0
    eng = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    B = args.pairs
    pts, lns = stereo_frames(B)
    cam, mc, sc = T.kitti_camera(), T.default_stereo_match_config(), T.default_stereo_config()
    off_p = np.arange(B + 1, dtype=np.int32) * 2000
    off_l = np.arange(B + 1, dtype=np.int32) * 500
    P = [eng.pinned.copy(np.concatenate([f[j] for f in pts])) for j in range(5)]      # pinned host buffers in and out
    L = [eng.pinned.copy(np.concatenate([f[j] for f in lns])) for j in range(6)]
    out_p, out_l = eng.stereo_outputs(2000 * B, B, lines=False, pinned=True), eng.stereo_outputs(500 * B, B, lines=True, pinned=True)
    launches0 = eng.launches

    def step():
        tp, _ = eng.match_stereo_points(cam, mc, sc, off_p, P[0], P[1], P[2], off_p, P[3], P[4], out=out_p)
        tl, _ = eng.match_stereo_lines(cam, mc, sc, off_l, L[0], L[1], L[2], L[3], off_l, L[4], L[5], out=out_l)
        return tp, tl
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    with ClockSampler(0) as clk:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            tp, tl = step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    launches = eng.launches - launches0
    h2d = sum(a.nbytes for a in P) + sum(a.nbytes for a in L)
    d2h = 2000 * B * (4 + 16 + 8 + 24 + 8 + 4 + 32 + 4) + 500 * B * (4 + 16 * 2 + 8 * 2 + 24 * 3 + 8 * 2 + 4 + 32 + 4)
    line = {"metric": metric, "value": B * args.steps / dt, "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/f64", "data": "synthetic",
            "config": {"workload": "stereo: matchStereoPoints + matchStereoLines (grid cells -> matchGrid -> lifting), host buffers in / out",
                       "frames_per_step": B, "lifted_points_per_step": int(tp), "lifted_lines_per_step": int(tl),
                       "note": "value IS the end-to-end figure here: every step uploads the raw key points / key lines and "
                               "descriptors and reads the records back (pinned host arrays)"},
            "clocks": clk.summary(), "gpu_launches": int(launches),
            "e2e": {"value": B * args.steps / dt, "unit": unit, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "roofline": None}
    if not args.no_cpu:
        sp, sl = stereo_frames(max(256, 8 * threads), first=B)
        rate, secs, _ = stereo_cpu_rate(sp, sl, threads)
        line["cpu_baseline"] = {"value": rate, "unit": unit, "cores": threads, "kind": "port", "cpu": cpu_model(),
                                "sample": f"{len(sp)} frames of the same workload, one frame per thread, {secs:.2f} s wall"}
    print(json.dumps(line), flush=True)
    eng.close()
    return 0


# --workload stereo_track: raw stereo features of (prev, curr) frame pairs in, poses out (plstvo_track_stereo_batch): the whole
# of insertStereoPair() + optimizePose() behind feature detection, the lifted records never leaving HBM.
def run_stereo_track(args):
    import torch
    from stvo_pl_b200 import stereo_synth as SS
    from stvo_pl_b200.engine import Engine
    metric, unit = "stereo pose solves/sec from raw stereo features (KITTI-shape, 2k key points + 500 key lines per image)", "solves/s"
    threads = host_threads()
    mc, sc, cfg = T.default_stereo_match_config(), T.default_stereo_config(), T.kitti_config()

    def cpu_rate(n_pairs):
        """CPU arm: the oracle's stereo step for both frames (C, one frame per thread) + its f2fTracking / optimizePose on
        records of the same sizes (C, one pair per thread); the two legs are timed one after the other and their times added."""
        from oracle.oracle import Oracle
        orc = Oracle(native=True)
        prev, curr, _, cam = SS.make_stereo_pairs(n_pairs, n_pt=1740, n_ls=500, seed=777)
        t_st = 0.0
        for d in (prev, curr):
            a = (cam, mc, sc, d["pl_off"], d["kp_l"], d["poct_l"], d["pdesc_l"], d["pr_off"], d["kp_r"], d["pdesc_r"], d["ll_off"],
                 d["seg_l"], d["angle_l"], d["loct_l"], d["ldesc_l"], d["lr_off"], d["seg_r"], d["ldesc_r"])
            orc.stereo_batch(*a, threads=threads)
            t0 = time.perf_counter()
            orc.stereo_batch(*a, threads=threads)
            t_st += time.perf_counter() - t0
        pv, cv, _, cam2 = synth.make_batch("kitti", n_pairs, n_pt=1740, n_ls=500, overlap=1.0)
        orc.track_batch(cam2, cfg, pv, cv, threads=threads)
        t0 = time.perf_counter()
        orc.track_batch(cam2, cfg, pv, cv, threads=threads)
        t_tr = time.perf_counter() - t0
        return n_pairs / (t_st + t_tr), t_st, t_tr

    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        n = max(64, 2 * threads)
        rate, t_st, t_tr = cpu_rate(n)
        line = {"impl": "reference", "metric": metric, "value": rate, "unit": unit, "n_gpus": args.gpus, "steps": 1, "warmup": 1,
                "ms_per_step": (t_st + t_tr) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8/f64", "data": "synthetic", "config": {"workload": "stereo_track", "pairs_per_step": n},
                "cpu_baseline": {"value": rate, "unit": unit, "cores": threads, "kind": "port", "cpu": cpu_model(),
                                 "sample": f"{n} pairs: stereo step {t_st:.3f} s + tracking {t_tr:.3f} s, all host threads"},
                "e2e": {"value": rate, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return 0
    eng = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    B = args.pairs
    prev, curr, Tgt, cam = SS.make_stereo_pairs(B, n_pt=1740, n_ls=500, seed=4242)     # 1740 + 15 % clutter = 2001 key points
    pin = lambda d: {k: eng.pinned.copy(np.ascontiguousarray(v, T.STEREO_FEATURE_DTYPES[k])) for k, v in d.items()}
    prev, curr = pin(prev), pin(curr)
    res = eng.pinned.empty((B,), T.POSE_RESULT_DTYPE)
    for _ in range(max(args.warmup, 3)):
        eng.track_stereo_batch(cam, cfg, mc, sc, prev, curr, results=res)
    torch.cuda.synchronize()
    launches0 = eng.launches
    with ClockSampler(0) as clk:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            _, n_st = eng.track_stereo_batch(cam, cfg, mc, sc, prev, curr, results=res)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    launches = eng.launches - launches0
    h2d = sum(v.nbytes for v in prev.values()) + sum(v.nbytes for v in curr.values())
    err = [float(np.linalg.norm(res["DT_opt"][p][:3, 3] - Tgt[p][:3, 3])) for p in range(B)]
    line = {"metric": metric, "value": B * args.steps / dt, "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64",
            "data": "synthetic",
            "config": {"workload": "stereo_track: matchStereoPoints + matchStereoLines of both frames -> f2fTracking -> optimizePose, "
                                   "raw key points / key lines and descriptors in (pinned host buffers), poses out",
                       "pairs_per_step": B, "mean_lifted": [float(x) for x in n_st.mean(0)], "solved_ok": int(res["good"].sum()),
                       "median_translation_error_m": float(np.median(err)),
                       "note": "value IS the end-to-end figure: every step uploads both frames' raw features and reads the poses back"},
            "clocks": clk.summary(), "gpu_launches": int(launches),
            "e2e": {"value": B * args.steps / dt, "unit": unit, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(res.nbytes + 16 * B)},
            "roofline": None}
    # the streaming form, two batches in flight (uploads of batch k + 1 under the kernels of batch k)
    pc, keep_p = T.stereo_features_as_c(prev)
    cc, keep_c = T.stereo_features_as_c(curr)
    pres = [eng.pinned.empty((B,), T.POSE_RESULT_DTYPE) for _ in range(2)]
    pns = [eng.pinned.empty((B, 4), np.int32) for _ in range(2)]
    for k in range(3):
        eng.wait(eng.track_stereo_batch_async(cam, cfg, mc, sc, pc, cc, pres[k & 1], pns[k & 1]))
    t0 = time.perf_counter()
    pend = None
    for k in range(args.steps):
        tk = eng.track_stereo_batch_async(cam, cfg, mc, sc, pc, cc, pres[k & 1], pns[k & 1])
        if pend is not None:
            eng.wait(pend)
        pend = tk
    eng.wait(pend)
    torch.cuda.synchronize()
    dtp = time.perf_counter() - t0
    line["e2e"]["pipelined_value"] = B * args.steps / dtp
    line["e2e"]["pipelined_ms_per_step"] = dtp / args.steps * 1e3
    line["e2e"]["pipelined_equals_blocking"] = bool(pres[(args.steps - 1) & 1].tobytes() == res.tobytes())
    # sequence mode: B + 1 consecutive frames -> B poses, every frame through the stereo step once (plstvo_track_stereo_sequence)
    seq, _, scam = SS.make_stereo_sequence(B + 1, n_pt=1740, n_ls=500, seed=99)
    seq = pin(seq)
    sres = eng.pinned.empty((B,), T.POSE_RESULT_DTYPE)
    for _ in range(3):
        eng.track_stereo_sequence(scam, cfg, mc, sc, seq, results=sres)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.track_stereo_sequence(scam, cfg, mc, sc, seq, results=sres)
    torch.cuda.synchronize()
    dts = time.perf_counter() - t0
    line["sequence_mode"] = {"value": B * args.steps / dts, "unit": "poses/s", "ms_per_step": dts / args.steps * 1e3,
                             "frames_per_step": B + 1, "solved_ok": int(sres["good"].sum()),
                             "h2d_bytes_per_step": int(sum(v.nbytes for v in seq.values())),
                             "note": "plstvo_track_stereo_sequence: consecutive frames of one camera, each frame uploaded and "
                                     "stereo-matched once; the Tfw chaining is a host-side scan (plstvo.hpp chainPoses)"}
    if not args.no_cpu:
        n = max(64, 2 * threads)
        rate, t_st, t_tr = cpu_rate(n)
        line["cpu_baseline"] = {"value": rate, "unit": unit, "cores": threads, "kind": "port", "cpu": cpu_model(),
                                "sample": f"{n} pairs: stereo step {t_st:.3f} s + tracking {t_tr:.3f} s, all host threads"}
    print(json.dumps(line), flush=True)
    eng.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=512, help="frame pairs per GPU per step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-hbm-run", action="store_true", help="skip the C5 streamed-evaluation sweeps appended at N=1")
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c5", "c5_sweep", "stereo", "stereo_track"],
                    help="c2: the headline solves/s bench (default); c1 / c3: the same pipeline on the points-only and the "
                         "EuRoC-shape robust configurations; c5: HBM-roofline run of the streamed GN evaluation "
                         "(1920x1080, 8000 points + 2000 lines, >= 1024 problems resident, 20 evaluations)")
    ap.add_argument("--kernels-only", action="store_true",
                    help="profiling aid: upload, launch K1 and K2 over the whole batch twice, exit (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs (rank 0) as DIR/<name>.npy (c1 / c2 / c3)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS or args.kernels_only):
        ap.error("--dump-outputs applies to the c1 / c2 / c3 workloads of --impl ours")
    global ACTIVE
    if args.workload in WORKLOADS:
        ACTIVE = args.workload
    if args.workload == "stereo":
        return run_stereo(args)
    if args.workload == "stereo_track":
        return run_stereo_track(args)
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "c5":
        return run_c5_pipeline(args)
    if args.workload == "c5_sweep":
        return run_c5(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
