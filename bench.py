#!/usr/bin/env python
"""bench.py — pose-graph windows/sec (10 keyframes x 2000 correspondences, 640x480 synthetic RGB-D) on N B200s.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` (torchrun for N>1) prints ONE JSON
line on rank 0.  One "step" = one pass of the hot path over one batch of `--windows` independent tracking windows per GPU
(BASELINE.json configs[1] replicated; configs[3] is 32 windows/GPU x 8 GPUs), i.e. weak scaling.  Every timed region runs
exactly K steps between CUDA events (max over ranks).  --min-seconds S repeats that K-step block back to back until S seconds have
passed and reports the median block, so that the clocks sampled during the region mean something.  --dump-outputs DIR writes the
poses the timed paths returned in their last step (value: poses.npy, e2e: e2e_poses.npy, [windows, frames, 4, 4] float32); the
inputs are seeded, so two builds run with the same arguments can be compared output for output.

  value     windows/s, whole job, inputs (keyframe maps, correspondences, poses, tables) already resident in HBM: per step
            ONE new frame per window is stored into the keyframe cache (k_frame_cache_store: its quarter-resolution maps are
            built inside the timed region), the other N-1 keyframes are reused - what a tracker does per frame
            (Bundler::processNewFrame -> selectKeyFramesForBA -> optimizeGPU) - then k_prep_frames (poses) + k_solve.
  e2e       the same through the reference-facing calls (bt_frame_cache_store + bt_solve_windows): per step the host
            correspondences + poses + window tables go host->device and the poses come back, exactly the arguments
            OptimizerGpu::optimizeFrames takes from the host; depth/normal maps are device-resident Frame members in the
            reference API (Frame::_depth_gpu/_normal_gpu) and are passed as device pointers.
  keyframe_cache.rebuild_every_call   the same batch with the reference's pattern (all N maps of every window rebuilt in every call).
  roofline  dominant kernel = k_solve; achieved = algorithmic bytes (SURVEY.md 8d: iters*(N*npix*32 + C*32) + 2*N*64 per window) /
            CUDA-event duration of that kernel; peak = MEASURED_PEAKS.json hbm_gbs (fallback 6650); plus the FP32 and the
            issue-slot view, because the kernel's working set stays in L2 (SURVEY.md 8d asks for the FP32 bound in that case).
  cpu_baseline  oracle/ (CPU restatement, "port": the reference has no CPU optimizer) on the host cores, bounded sample; and the
            reference's own kernels on ONE window in this same process (single_window_vs_reference).
  --impl reference   the reference's OWN CUDA kernels + host-glue allocation pattern (oracle/_ref, built verbatim from
            /root/reference) called once per window like Bundler::optimizeGPU does, on EVERY rank's GPU; plus the CPU port beside it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--windows", type=int, default=32, help="windows per GPU per step (BASELINE configs[3]: 256 over 8 GPUs)")
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--corr", type=int, default=2000)
    ap.add_argument("--scenes", type=int, default=4, help="distinct rendered scenes per GPU; windows cycle through them with their own pose noise and their own copy of the frame maps")
    ap.add_argument("--cpu-windows", type=int, default=0, help="cpu_baseline sample size (0 = 2 per core)")
    ap.add_argument("--ref-windows", type=int, default=8, help="windows per step for --impl reference")
    ap.add_argument("--min-seconds", type=float, default=0.0, help="repeat each timed region's K-step block until it has run this long (default: K steps once)")
    ap.add_argument("--skip-cfg3", action="store_true", help="leave out the BASELINE configs[2] block (30-keyframe pool)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the poses of the timed paths' last step to DIR/*.npy (--impl ours)")
    return ap.parse_args()


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self.proc = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self._stop.is_set():
                    break
        except Exception:
            pass

    def stop(self):
        self._stop.set()
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def make_batch(args, rank, dev):
    """`windows` windows per GPU: `scenes` rendered scenes, every window gets its OWN device copy of the frame maps (so
    the batch footprint, windows*frames*6.1 MB, is far larger than the 126 MB L2) and its own initial-pose noise."""
    import torch
    from bundletrack_b200 import synth
    from bundletrack_b200.optimizer import SolveWindow
    scenes = [synth.make_window(1000 * rank + s, n_frames=args.frames, n_corr=args.corr) for s in range(min(args.scenes, args.windows))]
    wins, host = [], []
    # every window's correspondences live in ONE page-locked host block (the contract's "inputs from pinned host memory"): the
    # library then lets the copy engine read them in place instead of staging them through its own pinned buffer
    n_ent = sum(len(scenes[k % len(scenes)].corr) for k in range(args.windows))
    pinned = torch.empty(max(n_ent, 1) * 32, dtype=torch.uint8).pin_memory()
    corr_all = pinned.numpy().view(synth.ENTRYJ_DTYPE)
    make_batch.keep = pinned
    c0 = 0
    for k in range(args.windows):
        sc = scenes[k % len(scenes)]
        corr_k = corr_all[c0:c0 + len(sc.corr)]
        corr_k[:] = sc.corr
        c0 += len(sc.corr)
        rng = np.random.default_rng(77 + 1000 * rank + k)
        poses = sc.poses_gt.copy()
        for f in range(1, sc.n_frames):
            poses[f] = sc.poses_gt[f] @ synth.se3(synth.so3_exp(rng.normal(0, np.deg2rad(1.0), 3)), rng.normal(0, 0.003, 3))
        depth = [torch.from_numpy(sc.depth[f]).to(dev) for f in range(sc.n_frames)]
        normal = [torch.from_numpy(sc.normal[f]).to(dev) for f in range(sc.n_frames)]
        # the per-pair counts travel with the correspondences like Bundler::optimizeGPU's n_match_per_pair (Bundler.cpp:298-351)
        wins.append(SolveWindow(corr_k, sc.H, sc.W, depth, normal, poses.astype(np.float32), sc.K, corr_block_n=SolveWindow.block_counts(sc.corr)))
        host.append((sc, poses.astype(np.float32)))
    return wins, host


def tensor_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["bf16_tflops"]), "measured"
    except Exception:
        return 1590.0, "fallback"


def tensor_peak_sustained():
    """cuBLAS 16-bit throughput run back to back for seconds (MEASURED_PEAKS.json bf16_tflops_sustained): the chip's power-limited rate.  The
    matcher's tensor pass is one 84 us kernel between non-tensor kernels, so the BURST figure is the denominator of tc_frac_of_tensor_peak;
    the sustained one is reported next to it."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["bf16_tflops_sustained"])
    except Exception:
        return None


def matcher_microbench(dev, stream):
    """Secondary evidence for the matcher half of the path (BASELINE configs[4]/[1]/[2]): kernel times from CUDA events inside the library.
    Tensor fraction = ALGORITHMIC flops (SURVEY.md 8d: F_match = 2 nA nB 256 per pair - one contraction serves both directions, and
    that is also what the kernel executes) / measured cuBLAS 16-bit tensor peak (MEASURED_PEAKS.json bf16_tflops; fp16 runs at the same rate)."""
    import torch
    from bundletrack_b200 import synth
    from bundletrack_b200.matcher import KnnMatcher
    tf_peak, src = tensor_peak()
    m = KnnMatcher(max_pairs=48, max_feats=5120, stream=stream)
    m.enable_timing(True)
    tf_sus = tensor_peak_sustained()
    out = {"peak_tensor_tflops": tf_peak, "peak_source": src, "peak_kind": "burst (kernel timed alone); sustained figure alongside", "peak_tensor_tflops_sustained": tf_sus,
           "operand_dtype": "f16", "accumulate_dtype": "f32"}
    a, b, _, _ = synth.make_descriptors(5, 5000, 5000)
    frames = [torch.from_numpy(synth.make_descriptors(100 + f, 2000, 8)[0]).to(dev) for f in range(10)]
    m.pool_reserve(12)                                      # descriptors converted once per frame (Lfnet::detectFeature uploads them once)
    for f in range(10):
        m.pool_store(f, frames[f])
    m.pool_store(10, torch.from_numpy(a).to(dev)); m.pool_store(11, torch.from_numpy(b).to(dev))
    idx = [(j, i) for i in range(10) for j in range(i + 1, 10)]
    for name, sl, sz in (("cfg5_5000x5000", [(10, 11)], [(5000, 5000)]), ("cfg2_45pairs_x2000", idx, [(2000, 2000)] * 45)):
        flop = sum(2.0 * na * nb * 256 for na, nb in sz)
        for _ in range(3):
            m.knn_match_slots(sl, sz, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            m.knn_match_slots(sl, sz, device=dev)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / 20
        tm = m.timing()
        out[name] = {"pairs": len(sl), "call_ms": wall * 1e3, "pairs_per_s": len(sl) / wall, "tc_kernel_ms": tm["tc_ms"], "select_rerank_ms": tm["rerank_ms"],
                     "fallback_ms": tm["fallback_ms"], "fallback_rows": tm["fallback_rows"], "tc_tflops_algorithmic": flop / (tm["tc_ms"] * 1e-3) / 1e12,
                     "tc_frac_of_tensor_peak": flop / (tm["tc_ms"] * 1e-3) / 1e12 / tf_peak,
                     "tc_frac_of_sustained_tensor_peak": (flop / (tm["tc_ms"] * 1e-3) / 1e12 / tf_sus) if tf_sus else None, "call_tflops_algorithmic": flop / wall / 1e12}
    m.close()
    try:      # the whole device-resident chain of the matcher side: kNN -> prune -> mutual -> RANSAC (2000 trials) -> EntryJ, 45 pairs of a 10-frame window
        from bundletrack_b200.matcher import MatchPipeline
        w = synth.make_window(77, n_frames=10, n_corr=10)
        fr = synth.make_feature_frames(w, 2000, seed=77, n_surface=12000)
        devf = [{"kpts": torch.from_numpy(fr[k]["kpts"]).to(dev), "desc": torch.from_numpy(fr[k]["desc"]).to(dev), "depth": torch.from_numpy(w.depth[k]).to(dev),
                 "normal": torch.from_numpy(w.normal[k]).to(dev), "pose": w.poses_init[k], "id": k, "window_index": k} for k in range(10)]
        mp = MatchPipeline(None, max_pairs=48, max_feats=2048, stream=stream)
        mp.pool_reserve(10)
        for k in range(10):
            mp.pool_store(k, devf[k]["desc"])
        prs = [(devf[j], devf[i]) for i in range(10) for j in range(i + 1, 10)]
        slots = [(j, i) for i in range(10) for j in range(i + 1, 10)]
        for _ in range(3):
            ent, n_ent, off = mp.match_pairs(prs, w.H, w.W, w.K, slots=slots)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            ent, n_ent, off = mp.match_pairs(prs, w.H, w.W, w.K, slots=slots)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / 10
        out["pipeline_45pairs"] = {"call_ms": wall * 1e3, "pairs_per_s": 45 / wall, "feats_per_frame": int(np.mean([len(f["kpts"]) for f in fr])),
                                   "entries_out": int(np.sum(n_ent)), "note": "bt_match_pairs_pool (descriptors in the pool) incl. the D2H of the EntryJ list"}
        mp.close()
    except Exception as e:
        out["pipeline_error"] = repr(e)
    return out


def cfg3_microbench(dev, stream, steps=20):
    """BASELINE configs[2]: 30-keyframe pool, 3000 features per frame, YCBInEOAT-shaped occlusion.  Solver: windows of 15 frames (the
    unchanged max_BA_frames) and of 30 frames (the whole pool), 3000 correspondences; matcher: all 435 pairs of the pool at 3000 x 3000."""
    import torch
    from bundletrack_b200 import synth
    from bundletrack_b200.optimizer import OptimizerGpu, SolveWindow
    from bundletrack_b200.matcher import KnnMatcher
    out = {}
    peak, _ = hbm_peak()
    npix = (640 // 4) * (480 // 4)
    for N, nwin in ((15, 8), (30, 4)):
        try:
            scenes = [synth.make_window(3000 + 10 * N + s, n_frames=N, n_corr=3000, occlusion=True) for s in range(2)]
            opt = OptimizerGpu(None, max_windows=nwin, max_frames=N, max_corr=3000, stream=stream)
            opt.enable_timing(True)
            wins = []
            for k in range(nwin):
                sc = scenes[k % 2]
                depth = [torch.from_numpy(sc.depth[f]).to(dev) for f in range(N)]
                normal = [torch.from_numpy(sc.normal[f]).to(dev) for f in range(N)]
                wins.append(SolveWindow(sc.corr, sc.H, sc.W, depth, normal, sc.poses_init, sc.K))
            opt.stage(wins)
            for _ in range(3):
                opt.run()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                opt.run()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            tm = opt.timing_ms()
            alg = nwin * (7 * (N * npix * 32 + 3000 * 32) + 2 * N * 64)
            ach = alg / (tm["solve"] * 1e-3) / 1e9
            one = [wins[0]]
            for _ in range(3):
                opt.optimizeWindows(one)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(20):
                opt.optimizeWindows(one)
            torch.cuda.synchronize()
            out[f"solver_N{N}"] = {"windows": nwin, "value": nwin / (ms * 1e-3), "unit": "windows/s", "ms_per_step": ms, "kernel_ms": tm,
                                   "single_window_e2e_ms": (time.perf_counter() - t0) / 20 * 1e3,
                                   "roofline": {"bound": "hbm", "kernel": "k_solve", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                                "algorithmic_bytes_per_launch": alg}}
            opt.close()
        except Exception as e:
            out[f"solver_N{N}_error"] = repr(e)
    try:
        tf_peak, _ = tensor_peak()
        m = KnnMatcher(max_pairs=435, max_feats=3072, stream=stream)
        m.enable_timing(True)
        m.pool_reserve(30)
        for f in range(30):
            m.pool_store(f, torch.from_numpy(synth.make_descriptors(500 + f, 3000, 8)[0]).to(dev))
        idx = [(j, i) for i in range(30) for j in range(i + 1, 30)]
        sz = [(3000, 3000)] * len(idx)
        for _ in range(2):
            m.knn_match_slots(idx, sz, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            m.knn_match_slots(idx, sz, device=dev)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / 5
        tm = m.timing()
        flop = len(idx) * 2.0 * 3000 * 3000 * 256
        out["matcher_435pairs_x3000"] = {"pairs": len(idx), "call_ms": wall * 1e3, "tc_kernel_ms": tm["tc_ms"], "select_rerank_ms": tm["rerank_ms"], "fallback_rows": tm["fallback_rows"],
                                         "tc_tflops_algorithmic": flop / (tm["tc_ms"] * 1e-3) / 1e12, "tc_frac_of_tensor_peak": flop / (tm["tc_ms"] * 1e-3) / 1e12 / tf_peak}
        m.close()
    except Exception as e:
        out["matcher_error"] = repr(e)
    return out


def frontend_microbench(opt, dev, stream):
    """SURVEY.md 8f rank 1: the fused depth front end (erode + 2x filter + points + normals) on 640x480 frames against its 40 B/pixel roofline."""
    import torch
    from bundletrack_b200 import synth
    from bundletrack_b200.frontend import FrameFrontEnd
    out = {}
    try:
        peak, _ = hbm_peak()
        fe = FrameFrontEnd(ctx=opt.ctx, stream=stream)
        nfr, H, W = 64, 480, 640
        raws = [torch.from_numpy(synth.make_raw_depth(s, H, W)[0]).to(dev) for s in range(4)]
        tin = [raws[i % 4].clone() for i in range(nfr)]
        dout = [torch.empty((H, W), device=dev) for _ in range(nfr)]
        nout = [torch.empty((H, W, 4), device=dev) for _ in range(nfr)]
        xout = [torch.empty((H, W, 4), device=dev) for _ in range(nfr)]
        for _ in range(3):
            fe.process(tin, H, W, synth.NOCS_K, dout, nout, xout)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            fe.process(tin, H, W, synth.NOCS_K, dout, nout, xout)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / 10 * 1e-3
        gbs = nfr * H * W * 40 / t / 1e9
        out["frontend"] = {"frames_per_s": nfr / t, "us_per_frame": t / nfr * 1e6, "achieved_GBps": gbs, "peak_GBps": peak, "frac": gbs / peak,
                           "algorithmic_bytes_per_pixel": 40, "sample": f"{nfr} frames 640x480 per call, 4+16+16 B written and 4 B read per pixel"}
    except Exception as e:      # secondary evidence must never take the headline down
        out["frontend_error"] = repr(e)
    return out


def ncu_profile(kernel):
    """Per-launch counters of the committed `ncu --set full` capture of the same bench command (profiles/traffic_r*.json, written by
    scripts/ncu_summary.py): dram bytes, warp instructions, fp32 thread instructions; {} when no capture is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "traffic_r*.json")))
    if not files:
        return {}
    try:
        with open(files[-1]) as f:
            return json.load(f).get(kernel, {})
    except Exception:
        return {}


def bind_to_gpu_numa_node(local):
    """Keep this rank's host threads (staging, marshalling, the copies' source pages) on the NUMA node its GPU hangs off: with 8 ranks on
    one host the e2e path is host-bound, and cross-socket staging costs it."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node = int(open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node").read())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, set(cpus))
        return node
    except Exception:
        return None


def cpu_baseline(host, n_windows, check_against=None, single_window=None):
    """Oracle A (float build) on the host cores: threads over windows (the C call releases the GIL).  `check_against`: the GPU
    poses of window 0 - the oracle's own result for that window doubles as the parity check of this very run.  `single_window`:
    (SolveWindow, ours_e2e_ms) - the reference's own kernels (oracle/_ref) on that ONE window in this same process, for the
    per-window ratio north_star asks for."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n = n_windows or 2 * cores
    oracle.build()
    jobs = [host[k % len(host)] for k in range(n)]
    def run(j):
        sc, poses = j
        return oracle.solve_window(sc.depth, sc.normal, sc.K, sc.corr, poses)
    run(jobs[0])
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:
        res = list(ex.map(run, jobs))
    dt = time.perf_counter() - t0
    out = {"value": n / dt, "unit": "windows/s", "cores": cores, "kind": "port",
           "sample": f"{n} windows of the bench workload, oracle/solver_oracle.c (fp32), {cores} threads, {dt:.1f} s"}
    if check_against is not None:
        from bundletrack_b200 import synth
        r, t = synth.pose_errors(check_against, res[0])
        out["gpu_vs_port_window0"] = {"rot_rad": r, "trans_m": t}
    if single_window is not None:
        try:
            w, ours_ms = single_window
            oracle.ref_lib()
            outer, solve = [], []
            for k in range(13):
                _, _, t_outer, t_solve = oracle.ref_optimize_frames(w.depths, w.normals, w.H, w.W, w.K, w.corr, w.poses)
                if k >= 3:
                    outer.append(t_outer); solve.append(t_solve)
            out["single_window_vs_reference"] = {"reference_outer_ms": float(np.median(outer)), "reference_solve_ms": float(np.median(solve)), "ours_e2e_ms": ours_ms,
                                                 "ratio": float(np.median(outer)) / ours_ms, "kind": "reference",
                                                 "sample": "median of 10 optimizeFrames-equivalent calls of the reference's own kernels + allocation pattern (oracle/_ref) on one "
                                                           "10-keyframe x 2000-correspondence window, same process, same GPU, after 3 warm-ups"}
        except Exception as e:
            out["single_window_vs_reference"] = {"unavailable": repr(e)}
    return out


def timed_blocks(step, steps, min_seconds, sync, est_ms):
    """K steps per block, as many back-to-back blocks as it takes to fill `min_seconds` (a 12 ms timed region tells little about clocks);
    CUDA events bracket every block on the launching stream.  Returns per-block ms and wall ms lists."""
    import torch
    n_blocks = int(max(1, min(400, np.ceil(min_seconds * 1e3 / max(steps * est_ms, 1e-3)))))
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_blocks)]
    walls = []
    sync()
    for b in range(n_blocks):
        t0 = time.perf_counter()
        evs[b][0].record()
        for _ in range(steps):
            step()
        evs[b][1].record()
        walls.append((time.perf_counter() - t0) * 1e3)
    sync()
    return [a.elapsed_time(b) for a, b in evs], walls


def main():
    args = parse()
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    numa = bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    windows_cfg = args.windows
    if args.impl == "reference":      # the reference arm only touches its sample: do not keep 1.9 GB of unused maps resident next to its cudaMalloc/cudaFree pattern
        args.windows = min(args.windows, args.ref_windows)
    wins, host = make_batch(args, rank, dev)
    args.windows = windows_cfg
    N, C = args.frames, args.corr
    npix = (640 // 4) * (480 // 4)
    workload = f"{args.windows} windows/GPU x ({N} keyframes, {C} corr, 640x480 -> 160x120 cache, 7 GN x 5 PCG), BASELINE configs[1] batched as configs[3]"
    base = {"metric": "pose-graph windows/sec (10 KF x 2k corr)", "unit": "windows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "windows_per_gpu": args.windows, "frames": N, "corr": C, "gn_iters": 7, "pcg_iters": 5,
                       "l2": f"inputs larger than L2: {args.windows * N * 6.1:.0f} MB of frame maps per GPU, each window its own copy", "parallelism": f"windows sharded, {world} rank(s), no data-path collective"}}

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    if args.impl == "reference":
        import oracle
        try:
            oracle.ref_lib()
        except Exception as e:      # oracle/_ref did not travel: the CPU port of the same algorithm stands in (kind "port")
            if rank == 0:
                cb = cpu_baseline(host, args.cpu_windows)
                out = dict(base, impl="reference", value=cb["value"], ms_per_step=None, gpu_launches=0,
                           e2e={"value": cb["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, cpu_baseline=cb,
                           note=f"oracle/_ref unavailable ({e}); timed the CPU port instead")
                print(json.dumps(out))
            if world > 1:
                dist.barrier(); dist.destroy_process_group()
            return
        # EVERY rank drives its own GPU through the reference's kernels (the reference has no CPU optimizer: its implementation of this
        # path is CUDA), so the whole-job number scales with the GPU count exactly like the repo's arm
        n = min(args.ref_windows, len(wins))
        outer, solve = [], []
        def step(record=False):
            for k in range(n):
                w = wins[k]
                _, _, t_o, t_s = oracle.ref_optimize_frames(w.depths, w.normals, w.H, w.W, w.K, w.corr, w.poses)
                if record:
                    outer.append(t_o); solve.append(t_s)
        for _ in range(args.warmup):
            step()
        sync_all()
        sampler = ClockSampler(local); sampler.start()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step(True)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        clocks = sampler.stop()
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        val = world * n * args.steps / dt
        if rank == 0:
            cb = cpu_baseline(host, args.cpu_windows)
            out = dict(base, impl="reference", value=val, ms_per_step=dt / args.steps * 1e3, gpu_launches=0,
                       e2e={"value": val, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                       cpu_baseline={"value": val, "unit": "windows/s", "cores": world, "kind": "reference",
                                     "sample": f"{n} windows per step per rank, one optimizeFrames-equivalent call each through the reference's OWN kernels + allocation pattern "
                                               f"(oracle/_ref), {world} rank(s) each driving its own GPU with one host thread: the reference has no CPU optimizer (SURVEY.md D5), its implementation of this path IS CUDA"},
                       reference_call_ms={"outer_median": float(np.median(outer)), "solve_median": float(np.median(solve)), "outer_min": float(np.min(outer)), "outer_max": float(np.max(outer)),
                                          "note": "per optimizeFrames-equivalent call on rank 0: whole call (cache build + allocations + solve + frees, LossGPU.cu:74-132) and the m_solver->solve region (SBA.cpp:132-135)"},
                       reference_ranks=world, cpu_port=cb, clocks=clocks, numa_node=numa)
            print(json.dumps(out))
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    from bundletrack_b200.optimizer import OptimizerGpu, SolveWindow
    stream = torch.cuda.current_stream().cuda_stream
    opt = OptimizerGpu(None, device=local, max_windows=args.windows, max_frames=max(N, 2), max_corr=max(C, 1), stream=stream)
    opt.enable_timing(True)

    # ---- the keyframe pool: every frame's quarter-resolution maps are built ONCE, when the frame enters the pool (the reference
    #      rebuilds all N of them inside every optimizeFrames call, CUDACache.cpp:76-88).  Honest accounting for a tracker: each step,
    #      every window gets ONE new frame (the tracked frame of Bundler::processNewFrame) whose maps are built inside the timed region;
    #      its N-1 keyframes are reused.
    nF = len(wins) * N
    opt.reserve_frame_cache(nF, wins[0].H, wins[0].W)
    slots = list(range(nF))
    opt.store_frames(slots, [d for w in wins for d in w.depths], [n_ for w in wins for n_ in w.normals], wins[0].H, wins[0].W, wins[0].K)
    cwins = [SolveWindow(w.corr, w.H, w.W, None, None, w.poses, w.K, cache_slots=slots[i * N:(i + 1) * N], corr_block_n=w.corr_block_n) for i, w in enumerate(wins)]
    new_slots = [i * N + (N - 1) for i in range(len(wins))]
    new_d = [w.depths[N - 1] for w in wins]; new_n = [w.normals[N - 1] for w in wins]
    store_args = opt.prepare_store(new_slots, new_d, new_n, wins[0].H, wins[0].W, wins[0].K)      # the call's argument arrays, marshalled once (as a C++ caller holds them)
    def store_new():
        opt.store_prepared(store_args)

    sampler = ClockSampler(local); sampler.start()
    # ---- value: resident inputs, kernels only (new-frame store + pose prep + persistent solve)
    opt.stage(cwins)
    def step_value():
        store_new(); opt.run()
    for _ in range(args.warmup):
        step_value()
    blk_ms, _ = timed_blocks(step_value, args.steps, args.min_seconds, sync_all, 0.5)
    tm = opt.timing_ms()                      # per-kernel device time of the last step
    stats = opt.stats()
    poses = opt.fetch()
    ms_step = float(np.median(blk_ms)) / args.steps
    t_val = torch.tensor([ms_step], device=dev)
    # ---- e2e: per step the new frames are stored and host correspondences/poses/tables go in, host poses come out.  Streaming form
    #      (bt_solve_windows_begin / _end, two batches in flight): step k's host work overlaps step k-1's GPU work; every step still
    #      uploads its own inputs and downloads a batch of poses.
    batch = opt.prepare_batch(cwins)      # bt_window array + pose block, marshalled once; every step still passes them through the C-ABI, which stages / uploads all of it
    pose_buf = np.empty((batch.poses.shape[0], 4, 4), np.float32)
    def step_e2e():
        store_new()
        opt.begin_prepared(batch)
        if step_e2e.inflight:
            opt.end_prepared(batch, pose_buf)
        step_e2e.inflight = True
    step_e2e.inflight = False
    for _ in range(max(args.warmup, 2)):
        step_e2e()
    _, wall_ms = timed_blocks(step_e2e, args.steps, args.min_seconds, sync_all, 0.6)
    opt.end_prepared(batch, pose_buf); step_e2e.inflight = False
    out_poses = [pose_buf[batch.off[i]:batch.off[i + 1]].copy() for i in range(len(cwins))]
    t_e2e = torch.tensor([float(np.median(wall_ms)) / args.steps], device=dev)
    # the blocking form of the same call, one batch at a time (what a caller without the streaming loop gets)
    def step_sync():
        store_new()
        opt.solve_prepared(batch, pose_buf)
    for _ in range(args.warmup):
        step_sync()
    _, sync_wall = timed_blocks(step_sync, args.steps, min(args.min_seconds, 0.3), sync_all, 0.7)
    host_us = opt.host_timing_us()
    t_sync = torch.tensor([float(np.median(sync_wall)) / args.steps], device=dev)
    # ---- the reference's own calling pattern, for comparison: every map rebuilt inside every call
    opt.stage(wins)
    for _ in range(args.warmup):
        opt.run()
    rb_ms, _ = timed_blocks(opt.run, args.steps, min(args.min_seconds, 0.3), sync_all, 0.7)
    tm_rb = opt.timing_ms()
    for _ in range(args.warmup):
        opt.optimizeWindows(wins)
    _, rb_wall = timed_blocks(lambda: opt.optimizeWindows(wins), args.steps, min(args.min_seconds, 0.3), sync_all, 0.8)
    t_rb = torch.tensor([float(np.median(rb_ms)) / args.steps, float(np.median(rb_wall)) / args.steps], device=dev)
    clocks = sampler.stop()      # sampled across all timed regions
    if world > 1:
        for t in (t_val, t_e2e, t_rb, t_sync):
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        from bundletrack_b200.sharding import gather_poses   # NCCL only gathers the results (windows are sharded per rank)
        poses = gather_poses(poses, args.windows * world, [N] * (args.windows * world), rank, world, device=dev)
        if args.dump_outputs:
            out_poses = gather_poses(out_poses, args.windows * world, [N] * (args.windows * world), rank, world, device=dev)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "poses.npy"), np.stack(poses).astype(np.float32))
        np.save(os.path.join(args.dump_outputs, "e2e_poses.npy"), np.stack(out_poses).astype(np.float32))
    ms_step = float(t_val.item())
    value = world * args.windows / (ms_step * 1e-3)
    e2e_val = world * args.windows / (float(t_e2e.item()) * 1e-3)
    new_frame_bytes = 0      # the new frames' depth/normal maps are device-resident Frame members in the reference API (Frame::_depth_gpu/_normal_gpu)
    h2d = sum(len(w.corr) * 32 + w.n_frames * 64 + w.n_frames * 20 + 120 + 45 * 8 + 46 * 12 for w in wins) + new_frame_bytes
    d2h = sum(w.n_frames * 64 for w in wins)

    if rank == 0:
        peak, peak_src = hbm_peak()
        alg_bytes = args.windows * (7 * (N * npix * 32 + C * 32) + 2 * N * 64)
        ach = alg_bytes / (tm["solve"] * 1e-3) / 1e9
        prof = ncu_profile("k_solve")
        sm_clock = (clocks.get("sm_mhz") or 1965.0) * 1e6
        # SURVEY.md 8d: when dram__bytes falls below B_alg (the batch's maps stay in L2) report the FP32 bound as well.  F_alg counts every
        # quarter-resolution pixel of every pair (400 flop each); the kernel only walks the compacted valid source lists (n_src_pixels).
        f_alg = args.windows * 7.0 * (N * (N - 1) / 2) * npix * 400
        f_valid = 7.0 * stats["n_src_pixels"] * 400
        fp32_peak = 148 * 128 * 2 * sm_clock / 1e12
        roof = {"bound": "hbm", "kernel": "k_solve", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": prof.get("dram_bytes_per_launch"),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": tm,
                "note": "effective-bandwidth figure: the batch's working set stays in L2 (traffic << algorithmic bytes); the kernel is latency/issue-bound, see fp32 / issue",
                "fp32": {"peak_tflops": fp32_peak, "peak_source": "148 SMs x 128 FMA lanes x 2 x sampled SM clock",
                         "alg_tflops_all_pixels": f_alg / (tm["solve"] * 1e-3) / 1e12, "alg_tflops_valid_pixels": f_valid / (tm["solve"] * 1e-3) / 1e12,
                         "frac_valid_pixels": f_valid / (tm["solve"] * 1e-3) / 1e12 / fp32_peak,
                         "executed_fp32_thread_inst_per_launch": prof.get("fp32_thread_inst_per_launch")},
                "issue": {"warp_inst_per_launch": prof.get("warp_inst_per_launch"),
                          "frac_of_issue_peak": (prof["warp_inst_per_launch"] / (tm["solve"] * 1e-3 * sm_clock * 148 * 4)) if prof.get("warp_inst_per_launch") else None,
                          "note": "warp instructions of the committed ncu capture / (live kernel time x 4 schedulers x 148 SMs x SM clock)"}}
        one = [wins[0]]
        for _ in range(5):
            opt.optimizeWindows(one)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(50):
            opt.optimizeWindows(one)
        torch.cuda.synchronize()
        single_ms = (time.perf_counter() - t0) / 50 * 1e3
        tm1 = opt.timing_ms()
        single = {"e2e_ms": single_ms, "kernel_ms": {"prep": tm1["prep"], "solve": tm1["solve"]},
                  "note": "bt_solve_windows on ONE 10-keyframe x 2000-correspondence window, host buffers in/out, all maps rebuilt in the call (the reference's call)"}
        # the same window the way a tracker presents it: the new frame's maps stored once (bt_frame_cache_store), its 9 keyframes already in the cache
        try:
            one_c = [cwins[0]]
            st1 = opt.prepare_store(new_slots[:1], new_d[:1], new_n[:1], wins[0].H, wins[0].W, wins[0].K)
            for _ in range(5):
                opt.store_prepared(st1); opt.optimizeWindows(one_c)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(50):
                opt.store_prepared(st1); opt.optimizeWindows(one_c)
            torch.cuda.synchronize()
            tmc = opt.timing_ms()
            single["keyframes_cached"] = {"e2e_ms": (time.perf_counter() - t0) / 50 * 1e3, "kernel_ms": {"prep": tmc["prep"], "solve": tmc["solve"]},
                                          "note": "bt_frame_cache_store of the ONE new frame + bt_solve_windows with cache slots (9 keyframes reused), host buffers in/out"}
        except Exception as e:
            single["keyframes_cached"] = {"error": repr(e)}
        # (before the matcher / cfg3 blocks allocate gigabytes: the reference's per-call cudaMalloc/cudaFree pattern slows down with the memory the process holds)
        cb = cpu_baseline(host, args.cpu_windows, check_against=out_poses[0], single_window=(wins[0], single_ms))
        matcher = matcher_microbench(dev, stream)
        extras = frontend_microbench(opt, dev, stream)
        cfg3 = cfg3_microbench(dev, stream) if not args.skip_cfg3 else None
        # per step: the new frames' store (k_cache_count + k_cache_build below 2 x SM-count frames, else one k_frame_cache_store) + pose prep + k_solve
        store_launches = 2 if len(new_slots) < 2 * torch.cuda.get_device_properties(dev).multi_processor_count else 1
        launches_per_step = store_launches + int(stats["n_kernel_launches"])
        out = dict(base, value=value, ms_per_step=ms_step, gpu_launches=launches_per_step * args.steps * len(blk_ms),
                   e2e={"value": e2e_val, "unit": "windows/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": float(t_e2e.item()),
                        "api": "bt_frame_cache_store + bt_solve_windows_begin / bt_solve_windows_end (two batches in flight)",
                        "blocking_call": {"value": world * args.windows / (float(t_sync.item()) * 1e-3), "ms_per_step": float(t_sync.item()), "api": "bt_frame_cache_store + bt_solve_windows",
                                          "host_us_last_call": host_us}},
                   roofline=roof, cpu_baseline=cb, clocks=clocks,
                   timing={"blocks": len(blk_ms), "steps_per_block": args.steps, "block_ms_min_med_max": [float(np.min(blk_ms)), float(np.median(blk_ms)), float(np.max(blk_ms))],
                           "launches_per_step": launches_per_step, "numa_node": numa},
                   keyframe_cache={"per_step": "one new frame per window built inside the timed region (k_frame_cache_store), N-1 keyframes reused",
                                   "rebuild_every_call": {"value": world * args.windows / (float(t_rb[0].item()) * 1e-3), "e2e": world * args.windows / (float(t_rb[1].item()) * 1e-3),
                                                          "unit": "windows/s", "kernel_ms": tm_rb, "note": "the reference's pattern: all N maps of every window rebuilt inside every call"}},
                   single_window=single, matcher=matcher, cfg3=cfg3, **extras, solver_stats=stats)
        print(json.dumps(out))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()
    opt.close()


if __name__ == "__main__":
    main()
