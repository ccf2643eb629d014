#!/usr/bin/env python
"""bench.py -- frame-pairs/sec of the rgbdslam_v2 frame-pair hot path (ORB Hamming brute-force match +
RANSAC SE(3)) on B200, BASELINE.json config C2: a batch of 256 synthetic frame pairs, 1000 ORB keypoints
per frame, per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W

One "step" = Node::matchNodePair (node.cpp:1305) for every pair of the batch through the C ABI.
  value : pairs/s with the nodes' features already resident in HBM (rgbdslam_b200_match_pairs on node
          handles) over exactly K timed steps in steady state (the pipeline is full when the timed region
          starts and when it ends), max over ranks.
  e2e   : same metric through rgbdslam_b200_match_pairs_host with pinned HOST buffers in and HOST
          MatchingResults out (H2D + D2H inside the timed region).
  roofline     : the Hamming kernel against the HBM roofline (SURVEY.md 8d: 72 000 B / pair @1000 kp).
  cpu_baseline : the CPU oracle (plain-C port of the reference path) on this box's host cores.
--impl reference times that CPU oracle as the reference arm (the reference itself cannot be built: ROS /
Qt / PCL / g2o / OpenCV-C++ are absent -- see DESIGN.md).
--dump-outputs DIR writes what the last timed step of both paths returned to its caller (rank 0), one
DIR/<path>_<array>_<field>.npy per field, integers as float64: the inputs are fixed by seeds, so two builds
of the library can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

PAIRS_PER_GPU = 256
N_KP = 1000
SEED = 2026
METRIC = "frame_pairs_per_sec_640x480_1k_orb"
UNIT = "pairs/s"
ALGO_BYTES_PER_PAIR = (N_KP + N_KP) * 32 + N_KP * 8  # SURVEY.md section 8(d): 72 000 B
# one string for both arms (the driver compares config.workload of `ours` and `reference`)
WORKLOAD = (f"C2: {PAIRS_PER_GPU} frame pairs x {N_KP} ORB kp per GPU, Hamming BF match + 4-pt RANSAC "
            "(200 hypotheses, max_matches 300), synthetic feature-level pairs (rgbdslam_v2_b200/synth.py make_batch)")
MIN_TIMED_MS = 50.0  # the rendered-frame C2 sub-measurement times at least this much


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed regions.  NVML in a thread (a handful of cheap driver
    queries every 20 ms) -- the recipe's `nvidia-smi -lms` loop is the fallback when pynvml is missing."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.nvml = None
        self.lines = []
        self.sm, self.mx, self.reasons = [], [], set()
        self.stop_flag = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.idx
            if vis:
                ent = vis.split(",")[self.idx].strip()
                phys = int(ent) if ent.isdigit() else None
            self.h = (pynvml.nvmlDeviceGetHandleByIndex(phys) if phys is not None
                      else pynvml.nvmlDeviceGetHandleByUUID(vis.split(",")[self.idx].strip()))
            self.nvml = pynvml
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        bits = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))
        try:
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
        except Exception:
            pass
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, bit in bits:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.th.join(timeout=2)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# dram__bytes_read.sum + dram__bytes_write.sum of ONE tc_hamming_expand_kernel launch on this workload, from the committed
# `ncu --set full` capture: 16.48 MB read + 0 written (the 2 MB of results stay in L2 for the selection kernel) against 18.4 MB
# algorithmic -- the kernel expands the 32-byte descriptors to MMA operands in shared memory itself.  (Round 1 read a resident
# +-1 int8 expansion instead: 139.3 MB per launch, 7.6 x the algorithmic bytes.)
NCU_DRAM_BYTES_PER_LAUNCH = 16479744
NCU_TRAFFIC_SOURCE = "profiles/r2_final_c2_kernels_ncu_full.txt (ncu --set full, 1 launch, C2 batch)"
# tcgen05.mma.kind::i8 M128 N128 K32 issued back to back on all 148 SMs, no epilogue (tools/microbench/tc_peaks.cu on this pool's
# B200s, profiles/r2_v7_tc_peaks.json): 64.0 cycles per MMA = 4514.7 TOP/s at the 1.86 GHz the SMs hold under that load
INT8_MMA_MEASURED_TOPS = 4514.7


def tensor_roofline(kernel_ms: float) -> dict:
    """The match kernel against the tensor roofline: exact +-1 int8 GEMM, 2 * Nq * Nt * 256 integer ops per pair.  Peak:
    dense int8 = 2 x the dense bf16 rate on B200 (4.5 vs 2.25 POP/s nominal), scaled from the MEASURED bf16 number."""
    ops = 2.0 * N_KP * N_KP * 256 * PAIRS_PER_GPU
    achieved = ops / (kernel_ms * 1e-3) / 1e12
    peak = 2.0 * 1701.0
    src = "2 x nominal-ratio of fallback bf16 1701 TF/s"
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")) as f:
            peak = 2.0 * float(json.load(f)["bf16_tflops"])
            src = "2 x MEASURED_PEAKS.json bf16_tflops (int8 dense = 2 x bf16 dense on sm_100)"
    except Exception:
        pass
    return {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TOP/s (int8)", "frac": achieved / peak, "peak_source": src,
            "ops_counted": "algorithmic 2 * Nq * Nt * 256 per pair (the ninth, column-index k-step and the padding to 128-row tiles are overhead)",
            "int8_mma_issue_peak": INT8_MMA_MEASURED_TOPS, "frac_of_int8_mma_issue_peak": achieved / INT8_MMA_MEASURED_TOPS,
            "int8_mma_issue_peak_source": "tools/microbench/tc_peaks.cu (profiles/r2_v7_tc_peaks.json): tcgen05.mma.kind::i8 alone, 64.0 cycles per M128 N128 K32"}


def make_workload(rank: int):
    from rgbdslam_v2_b200 import synth
    return synth.make_batch(PAIRS_PER_GPU, N_KP, seed0=SEED + rank * PAIRS_PER_GPU)


def usable_cpus() -> int:
    """Host threads this process can really run on: affinity mask and cgroup CPU quota, not just os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:  # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, -(-int(q) // int(per))))
    except (OSError, ValueError):
        pass
    try:  # cgroup v1
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and per > 0:
            n = min(n, max(1, -(-q // per)))
    except (OSError, ValueError):
        pass
    return n


def pick_threads(b) -> tuple[int, dict]:
    """The thread count the CPU port runs FASTEST with on this host (256 pairs of ~1.5 ms each do not keep 128 OpenMP threads
    busy: measured 2.5 k pairs/s with 128 threads on the GPU box vs 690 single-threaded).  One warm + one timed pass each."""
    top = usable_cpus()
    cands = sorted({c for c in (top, top // 2, top // 4, 32, 16, 8, 4) if 1 <= c <= top}, reverse=True)
    timings = {}
    for c in cands:
        oracle_run(b, 0, c)
        timings[c] = min(oracle_run(b, 0, c)[0] for _ in range(2))
    best = min(timings, key=timings.get)
    return best, {str(k): round(PAIRS_PER_GPU / v, 1) for k, v in timings.items()}


def oracle_run(b, first_pair, threads, npairs=None):
    from oracle import oracle
    prm = oracle.make_params(depth_cov_z0=2.0)
    n = npairs or len(b["n_newer"])
    t0 = time.perf_counter()
    res, _, _ = oracle.match_pairs(prm, b["desc_newer"][: n * N_KP], b["xyz_newer"][: n * N_KP], b["n_newer"][:n],
                                   b["desc_older"][: n * N_KP], b["xyz_older"][: n * N_KP], b["n_older"][:n],
                                   b["id_newer"][:n], b["id_older"][:n], seed=SEED, first_pair_index=first_pair, threads=threads)
    return time.perf_counter() - t0, res


def run_reference(args, rank, world):
    """Reference arm: the CPU port of the reference path (oracle/), all host threads, rank 0 only."""
    if rank != 0:
        return
    from oracle import oracle
    oracle.build()
    b = make_workload(0)
    oracle_run(b, 0, usable_cpus())  # the first passes are 5-6 x slower (OpenMP team start-up, allocator arenas)
    cores, thread_scan = pick_threads(b)
    for _ in range(max(args.warmup, 3)):
        oracle_run(b, 0, cores)
    times = []
    for _ in range(args.steps):
        dt, _ = oracle_run(b, 0, cores)
        times.append(dt)
    tot = sum(times)
    value = PAIRS_PER_GPU * args.steps / tot
    sample = f"{PAIRS_PER_GPU} pairs x {N_KP} kp per step (the full C2 batch of one GPU), OpenMP over pairs"
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 popcount + f32 fit + f64 Mahalanobis", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "note": "CPU port of the reference path (oracle/frontend_oracle.c); the reference itself is unbuildable here"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "cores_available": usable_cpus(), "pairs_per_s_by_thread_count": thread_scan},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


def fe_device(fe):
    import torch
    return torch.cuda.current_device()


def bench_posegraph(fe):
    """Secondary: BASELINE config C5 (5000 vertices / 30000 edges) pose-graph LM: the GPU solve and the CPU oracle (plain-C port of
    g2o's LM + block-Jacobi PCG, single thread like g2o's solver) on the SAME graph."""
    from oracle import oracle
    from rgbdslam_v2_b200 import synth
    g = synth.make_pose_graph(5000, 30000, seed=0)
    fe.optimize_graph(g["init"], g["fixed"], g["ij"], g["meas"], g["info"], stop=0.01)  # warm-up
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        x, chi2, it, cg = fe.optimize_graph(g["init"], g["fixed"], g["ij"], g["meas"], g["info"], stop=0.01)
        ts.append(time.perf_counter() - t0)
    dt = min(ts)
    t0 = time.perf_counter()
    ox, ochi2, oit, ocg = oracle.posegraph_optimize(g["init"], g["fixed"], g["ij"], g["meas"], g["info"], stop=0.01)
    dto = time.perf_counter() - t0
    # algorithmic HBM bytes (SURVEY 8d): 18.9 MB per PCG iteration, 45 MB per linearisation
    return {"workload": "C5: 5000 V / 30000 E, optimizer_iterations 0.01, pcg", "seconds": dt, "lm_iterations": it, "pcg_iterations": cg,
            "chi2": chi2, "ate_m": synth.ate_rmse(x[:, :3], g["gt"][:, :3]), "pcg_iter_per_s": cg / dt, "us_per_pcg_iteration": 1e6 * dt / max(cg, 1),
            "algorithmic_GBps": (cg * 18.9e6 + it * 45e6) / dt / 1e9,
            "cpu_baseline": {"seconds": dto, "kind": "port", "cores": 1, "lm_iterations": oit, "pcg_iterations": ocg, "chi2": ochi2,
                             "sample": "the same C5 graph, full solve", "speedup": dto / dt,
                             "chi2_rel_diff": abs(chi2 - ochi2) / max(ochi2, 1e-30),
                             "ate_gpu_vs_cpu_m": synth.ate_rmse(x[:, :3], ox[:, :3])}}


def bench_c2_rendered(fe, local_rank, cpu=True):
    """The C2 step on a harder, more realistic workload (SURVEY 8d specified C2 on the rendered-frame generator): nodes built by
    rgbdslam_b200_nodes_create from rendered 640x480 frames (real, correlated ORB descriptors), 256 pairs per batch of which
    HALF pair a frame with a frame of a DIFFERENT scene (no true correspondences: the reference's loop-closure candidate lists
    are dominated by such pairs -- they run all 200 RANSAC iterations and fail), the other half with a frame 1-8 steps back."""
    import ctypes as C
    import torch
    from rgbdslam_v2_b200 import synth
    from rgbdslam_v2_b200._capi import PAIR_RESULT_DTYPE, default_params
    dev = torch.device("cuda", local_rank)
    K4 = (synth.FX, synth.FY, synth.CX, synth.CY)
    prm = default_params(); prm.depth_cov_z0 = 2.0; prm.max_keypoints = N_KP
    old = fe.params
    fe.params = prm
    fe._check(fe.lib.rgbdslam_b200_init(local_rank, C.byref(prm)))
    out = {}
    try:
        nA, nB, NB = 300, 160, 5
        poses = synth.trajectory(2000)
        hs = []
        for tex, n, off in ((7, nA, 0), (8, nB, 700)):
            g_d, d_d = synth.render_frames_torch(poses[off:off + n], dev, first_index=off, tex_seed=tex)
            det = fe.detector_create()
            h, nf = fe.nodes_create(det, g_d.cpu().numpy(), d_d.cpu().numpy(), None, K4, mask_from_depth=True)
            fe.detector_destroy(det)
            hs.append((h, nf))
        (hA, nfA), (hB, nfB) = hs
        rng = np.random.default_rng(5)
        batches = []
        for b in range(NB):
            newer, older = [], []
            for i in range(PAIRS_PER_GPU):
                k = int(rng.integers(10, nA))
                newer.append(hA[k])
                older.append(hB[int(rng.integers(0, nB))] if i % 2 else hA[k - int(rng.choice([1, 2, 3, 5, 8]))])
            res = torch.zeros(PAIRS_PER_GPU * PAIR_RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
            batches.append((np.array(newer, np.uint64), np.array(older, np.uint64), res.numpy().view(PAIR_RESULT_DTYPE), res))

        def run(K):
            for k in range(K):
                if k >= NB:
                    fe.wait_slot(1 + (k - NB) % NB)
                nw, ol, r, _ = batches[k % NB]
                fe.submit_node_pairs(1 + k % NB, nw, ol, (r, None, None), seed=SEED, first_pair_index=(k % NB) * PAIRS_PER_GPU)
            for k in range(max(0, K - NB), K):
                fe.wait_slot(1 + k % NB)
        run(2 * NB)
        torch.cuda.synchronize()
        t0 = time.perf_counter(); run(20); torch.cuda.synchronize(); probe = (time.perf_counter() - t0) / 20
        K = max(20, int(np.ceil(MIN_TIMED_MS * 1e-3 / probe)))
        t0 = time.perf_counter(); run(K); torch.cuda.synchronize(); dt = time.perf_counter() - t0
        sync_dev = []
        for _ in range(5):
            nw, ol, r, _ = batches[0]
            fe.match_node_pairs(nw, ol, seed=SEED, first_pair_index=0, out=(r, None, None))
            sync_dev.append(fe.last_timing(0))
        r0 = batches[0][2]
        out = {"workload": f"C2 on rendered frames: {PAIRS_PER_GPU} pairs x <= {N_KP} ORB kp per batch, nodes from rgbdslam_b200_nodes_create "
                           f"(mean {float(np.mean(nfA)):.0f} features), 50 % of the pairs across two different scenes (no overlap), "
                           f"{NB} batches in flight",
               "value": PAIRS_PER_GPU * K / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / K, "timed_steps": K,
               "synchronous_device_ms_per_step": statistics.median(t for _, t in sync_dev),
               "hamming_kernel_ms": statistics.median(h for h, _ in sync_dev),
               "valid_fraction": float((r0["id1"] >= 0).mean()),
               "valid_fraction_same_scene_pairs": float((r0["id1"][0::2] >= 0).mean()),
               "valid_fraction_cross_scene_pairs": float((r0["id1"][1::2] >= 0).mean())}
        if cpu:
            from oracle import oracle  # CPU arm on the same features (the GPU-built nodes are bit-identical to the cv2 pipeline's)
            feats = {}
            nw, ol, _, _ = batches[0]
            for h in set(nw.tolist()) | set(ol.tolist()):
                feats[h] = fe.node_download(int(h))
            cat = lambda hh, j: np.ascontiguousarray(np.concatenate([feats[int(x)][j] for x in hh]))
            n_n = np.array([len(feats[int(x)][0]) for x in nw], np.int32); n_o = np.array([len(feats[int(x)][0]) for x in ol], np.int32)
            dn, xn, do, xo = cat(nw, 0), cat(nw, 1), cat(ol, 0), cat(ol, 1)
            oprm = oracle.make_params(depth_cov_z0=2.0)
            cores = usable_cpus()
            best = None
            for _ in range(3):
                t0 = time.perf_counter()
                ores, _, _ = oracle.match_pairs(oprm, dn, xn, n_n, do, xo, n_o, np.arange(PAIRS_PER_GPU, dtype=np.int32) + 1,
                                                np.arange(PAIRS_PER_GPU, dtype=np.int32), seed=SEED, first_pair_index=0, threads=cores,
                                                want_matches=False)
                t = time.perf_counter() - t0
                best = t if best is None else min(best, t)
            out["cpu_baseline"] = {"value": PAIRS_PER_GPU / best, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": "one 256-pair batch of the same workload, best of 3, OpenMP over pairs",
                                   "valid_flag_agreement": float(((ores["id1"] >= 0) == (r0["id1"] >= 0)).mean())}
        for h in hA + hB:
            fe.node_destroy(h)
    finally:
        fe.params = old
        fe._check(fe.lib.rgbdslam_b200_init(local_rank, C.byref(old)))
    return out


C3_KP = 2000
C3_PAIRS = 64


def bench_c3(fe, local_rank, cpu=True):
    """BASELINE config C3: SIFT 128-d float descriptors, 2000 keypoints per frame, the distance matrix as a bf16 tensor-core
    GEMM (ratio / uniqueness matcher = the FLANN branch node.cpp:610-667 with an exact search) and the SiftGPU matcher (u8
    dot products); pairs/s with resident nodes, the tensor roofline of the match kernel, end to end from host descriptors,
    the fraction of exact nearest neighbours, and cv2's brute-force / FLANN matchers on the host cores."""
    import torch
    from rgbdslam_v2_b200 import synth
    rng = np.random.default_rng(33)
    out = {"workload": f"C3: {C3_PAIRS} frame pairs x {C3_KP} SIFT-128 descriptors per frame (synthetic SIFT-like rows, 50 % of the "
                       "newer frame's features are noisy copies of the older frame's), exact 2-NN via bf16 tcgen05 GEMM + fp32 re-rank, "
                       "ratio 0.95 / uniqueness, 4-pt RANSAC"}
    peak_bf16 = 1701.0
    try:
        peak_bf16 = float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["bf16_tflops"])
        out["peak_source"] = "MEASURED_PEAKS.json bf16_tflops (burst)"
    except Exception:
        out["peak_source"] = "fallback 1701 TF/s"
    for kind, matcher in (("sift", 0), ("siftgpu", 1)):
        fe.set_sift_matcher(matcher)
        pairs = [synth.make_pair_sift(9000 + k, C3_KP, overlap=0.5, kind=kind) for k in range(C3_PAIRS)]
        newer = [fe.node_from_sift(2 * k + 1, q["desc_newer"], q["xyz_newer"]) for k, q in enumerate(pairs)]
        older = [fe.node_from_sift(2 * k, q["desc_older"], q["xyz_older"]) for k, q in enumerate(pairs)]
        for _ in range(3):
            res, _, _ = fe.match_node_pairs(newer, older, seed=5, want_matches=False)
        ts, kern = [], []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res, _, _ = fe.match_node_pairs(newer, older, seed=5, want_matches=False)
            ts.append(time.perf_counter() - t0)
            st = fe.stage_times(0)
            kern.append((st["hamming"], st["total"]))
        k_ms = statistics.median(k for k, _ in kern)
        dev_ms = statistics.median(t for _, t in kern)
        items = 2 if matcher == 1 else 1  # the SiftGPU matcher runs the row and the column pass (two GEMMs) in one launch
        flops = 2.0 * C3_KP * C3_KP * 128 * C3_PAIRS * items
        entry = {"pairs_per_s_resident": C3_PAIRS / (dev_ms * 1e-3), "device_ms_per_batch": dev_ms, "wall_ms_per_batch": 1e3 * statistics.median(ts),
                 "match_kernel_ms": k_ms, "valid_pairs": int((res["id1"] >= 0).sum()),
                 "roofline": {"bound": "tensor", "kernel": "tc_match256_kernel<%d>" % (1 if matcher == 0 else 2),
                              "achieved": flops / (k_ms * 1e-3) / 1e12, "peak": peak_bf16 * (2.0 if matcher == 1 else 1.0),
                              "unit": "TFLOP/s (bf16)" if matcher == 0 else "TOP/s (u8; peak = 2 x measured bf16)",
                              "algorithmic_flops_per_launch": flops}}
        entry["roofline"]["frac"] = entry["roofline"]["achieved"] / entry["roofline"]["peak"]
        # end to end: host descriptors in (upload + RootSIFT / tile preparation inside), host results out
        def e2e_pass():
            t0 = time.perf_counter()
            hn = [fe.node_from_sift(5000 + 2 * k + 1, q["desc_newer"], q["xyz_newer"]) for k, q in enumerate(pairs)]
            ho = [fe.node_from_sift(5000 + 2 * k, q["desc_older"], q["xyz_older"]) for k, q in enumerate(pairs)]
            fe.match_node_pairs(hn, ho, seed=5, want_matches=False)
            dt = time.perf_counter() - t0
            for h in hn + ho:
                fe.node_destroy(h)
            return dt
        e2e_pass()
        e2e = min(e2e_pass() for _ in range(2))
        entry["e2e"] = {"pairs_per_s": C3_PAIRS / e2e, "h2d_bytes": int(2 * C3_PAIRS * C3_KP * (512 + 16)),
                        "note": "node_from_sift per frame (synchronous uploads, RootSIFT + tile preparation) + one batched match"}
        if matcher == 0:
            from oracle import sift_oracle  # checker: exact float64 2-NN
            same = []
            for k in range(4):
                q, t = pairs[k]["desc_newer"], pairs[k]["desc_older"]
                idx, _ = fe.knn2_l2(q, t)
                oidx, _ = sift_oracle.knn2_exact(sift_oracle.root_sift(q), sift_oracle.root_sift(t))
                same.append(float((idx[:, 0] == oidx[:, 0]).mean()))
            entry["exact_nearest_neighbour_fraction"] = float(np.mean(same))
            if cpu:
                import cv2
                cv2.setNumThreads(usable_cpus())
                rs = [(sift_oracle.root_sift(q["desc_newer"]), sift_oracle.root_sift(q["desc_older"])) for q in pairs[:4]]
                bf = cv2.BFMatcher(cv2.NORM_L2)
                bf.knnMatch(rs[0][0], rs[0][1], k=2)
                t0 = time.perf_counter()
                for q, t in rs:
                    bf.knnMatch(q, t, k=2)
                t_bf = (time.perf_counter() - t0) / 4
                fl = cv2.FlannBasedMatcher(dict(algorithm=1, trees=4), dict(checks=16))  # node.cpp:503-510, 1573-1581
                t0 = time.perf_counter()
                for q, t in rs:
                    fl.knnMatch(q, t, k=2)
                t_fl = (time.perf_counter() - t0) / 4
                entry["cpu_baseline"] = {"cv2_bfmatcher_knn2_pairs_per_s": 1.0 / t_bf, "cv2_flann_kdtree4_checks16_pairs_per_s": 1.0 / t_fl,
                                         "cores": usable_cpus(), "kind": "reference dependency (cv2 4.13) -- matching stage only, no RANSAC",
                                         "sample": "4 pairs of the same workload"}
        out["ratio_matcher" if matcher == 0 else "siftgpu_matcher"] = entry
        for h in newer + older:
            fe.node_destroy(h)
    fe.set_sift_matcher(0)
    return out


C4_FRAMES = 2000
C4_SEED = 11


def bench_sequence(fe, local_rank, rank, world, comm, n_frames=C4_FRAMES, with_oracle=False, oracle_frames=120):
    """BASELINE config C4: a 2000-frame synthetic sequence end to end through the C ABI -- pinned HOST images in,
    optimised trajectory out: Node::Node for every frame (rgbdslam_b200_nodes_create_ex), the 3 sequential + 4 window +
    4 random candidate pairs per frame (~22 k pairs) through Node::matchNodePair in batches of 256 on the pipeline slots,
    (N > 1: frames and pairs sharded over the ranks, ONE all-gather of the edge records), addEdgeToG2O glue, optimizeGraph
    on every rank, ATE against the rendering ground truth.  Strong scaling: the work is fixed as N grows."""
    import torch
    from rgbdslam_v2_b200 import pipeline, synth
    from rgbdslam_v2_b200._capi import PAIR_RESULT_DTYPE, default_params, graph_from_pairs
    import ctypes as C
    dev = torch.device("cuda", local_rank)
    poses = synth.trajectory(n_frames)
    K4 = (synth.FX, synth.FY, synth.CX, synth.CY)
    prm = default_params(); prm.depth_cov_z0 = 2.0; prm.max_keypoints = N_KP
    old = fe.params
    fe.params = prm
    fe._check(fe.lib.rgbdslam_b200_init(local_rank, C.byref(prm)))
    out = {"workload": f"C4: {n_frames}-frame synthetic sequence 640x480 (torch-rendered box room, trajectory with revisits), "
                       f"max_keypoints {N_KP}, candidates 3 sequential + 4 window + 4 random per frame, pose_relative_to first, "
                       f"optimizer_iterations 0.01", "n_gpus": world}
    try:
        # ---- data (not timed): this rank's frames rendered on its GPU, copied to pinned host memory
        per = -(-n_frames // world)
        f0, f1 = (0, n_frames) if world == 1 else (min(rank * per, n_frames), min((rank + 1) * per, n_frames))
        g_d, d_d = synth.render_frames_torch(poses[f0:f1], dev, first_index=f0)
        gray = torch.empty(g_d.shape, dtype=torch.uint8).pin_memory(); gray.copy_(g_d)
        depth = torch.empty(d_d.shape, dtype=torch.float32).pin_memory(); depth.copy_(d_d)
        del g_d, d_d
        torch.cuda.synchronize()
        pairs = np.array(pipeline.candidate_pairs(n_frames, seed=C4_SEED), np.int64)
        gt = np.stack([pipeline.mat_to_pose7(np.linalg.inv(poses[0]) @ P) for P in poses])

        def run(nf):
            """frames [0, nf) (own shard of them) -> trajectory; returns (traj, stage seconds, info)"""
            t = {}
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            det = fe.detector_create()
            if world == 1:
                handles, nfeat = fe.nodes_create(det, gray[:nf], depth[:nf], None, K4, ids=np.arange(nf, dtype=np.int32),
                                                 mask_from_depth=True)
            else:
                # this rank's block of the first nf frames (for nf < n_frames -- the warm-up -- the block is cut from the rank's
                # own shard: wrong frames, right sizes)
                from rgbdslam_v2_b200.sharding import frame_shard
                own = len(frame_shard(nf, rank, world))
                handles, nfeat = fe.nodes_create_sharded(det, comm, nf, gray[:own], depth[:own], None, K4, mask_from_depth=True)
            t["nodes"] = time.perf_counter() - t0
            pp = pairs[pairs[:, 0] < nf]
            per_p = -(-len(pp) // world)
            p0, p1 = min(rank * per_p, len(pp)), min((rank + 1) * per_p, len(pp))
            t1 = time.perf_counter()
            local = np.zeros(per_p, PAIR_RESULT_DTYPE); local["id1"] = -1; local["id2"] = -1
            pipeline.match_pairs_pipelined(fe, handles, pp[p0:p1], seed=C4_SEED, first_pair_index=p0, out=local[: p1 - p0])
            t["match"] = time.perf_counter() - t1
            t2 = time.perf_counter()
            if world > 1:
                res = fe.allgather_edges(comm, local, world)[: len(pp)]  # the ONE exchange of the pair stage (SURVEY 8e)
            else:
                res = local[: len(pp)]
            t["gather"] = time.perf_counter() - t2
            t3 = time.perf_counter()
            graph = graph_from_pairs(pp, res, nf)  # host glue of the C ABI (addEdgeToG2O bookkeeping)
            t["graph_host"] = time.perf_counter() - t3
            t4 = time.perf_counter()
            traj, chi2, lm, cg = fe.optimize_graph(graph["init"], graph["fixed"], graph["ij"], graph["meas"], graph["info"], stop=0.01)
            t["solve"] = time.perf_counter() - t4
            t["total"] = time.perf_counter() - t0
            info = dict(pairs=int(len(pp)), valid_edges=int(graph["n_valid_edges"]), const_edges=int(graph["n_const_edges"]),
                        mean_features=float(np.mean(nfeat)), lm_iterations=lm, pcg_iterations=cg, chi2=chi2)
            fe.detector_destroy(det)
            for h in handles:
                fe.node_destroy(h)
            return traj, t, info, res

        fe.posegraph_reserve(n_frames, 12 * n_frames)  # solver buffers sized for the session, like the pinned image buffers
        run(min(n_frames, 96 * world))  # warm-up (allocations, first launches)
        traj, t, info, _ = run(n_frames)
        tt = torch.tensor([t[k] for k in ("nodes", "match", "gather", "graph_host", "solve", "total")], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        tt = tt.tolist()
        out.update(info)
        out["seconds"] = dict(zip(("nodes", "match", "gather", "graph_host", "solve", "total"), tt))
        out["frames_per_s"] = n_frames / tt[5]
        out["pairs_per_s"] = info["pairs"] / tt[5]
        out["node_constructor_frames_per_s"] = n_frames / tt[0]
        out["match_stage_pairs_per_s"] = info["pairs"] / tt[1]
        out["ate_vs_gt_m"] = synth.ate_rmse(traj[:, :3], gt[:, :3])
        out["h2d_bytes"] = int(n_frames * synth.W * synth.H * 5)
        out["scaling"] = "strong (fixed 2000 frames / pair list)"
        if with_oracle and world == 1 and rank == 0:
            # the same pipeline on the CPU oracle (cv2 ORB + C port) on a prefix of the sequence: ATE of both against the
            # ground truth and against each other (north star: within 1 mm), and the CPU frames/s of the whole chain
            from oracle import oracle
            from oracle.backend import OracleBackend
            from oracle import orb_oracle
            nf = oracle_frames
            g_traj, _, g_info, g_res = run(nf)
            gn, dn = gray[:nf].numpy(), depth[:nf].numpy()
            mn = np.stack([orb_oracle.depth_to_mask(d) for d in dn])
            ob = OracleBackend(oracle, N_KP)
            c0 = time.perf_counter()
            nodes = ob.construct_nodes(gn, dn, mn, K4)
            c1 = time.perf_counter()
            pp = pairs[pairs[:, 0] < nf]
            ores = ob.match(nodes, [tuple(x) for x in pp], C4_SEED)
            c2 = time.perf_counter()
            ograph = pipeline.build_graph_fast(pp, ores, nf)
            o_traj, o_chi2 = ob.optimize(ograph, 0.01)
            c3 = time.perf_counter()
            out["oracle_prefix"] = {
                "frames": nf, "pairs": int(len(pp)),
                "ate_gpu_vs_gt_m": synth.ate_rmse(g_traj[:, :3], gt[:nf, :3]), "ate_oracle_vs_gt_m": synth.ate_rmse(o_traj[:, :3], gt[:nf, :3]),
                "ate_gpu_vs_oracle_m": synth.ate_rmse(g_traj[:, :3], o_traj[:, :3]),
                "valid_flag_agreement": float(((g_res["id1"] >= 0) == (ores["id1"] >= 0)).mean()),
                "cpu_seconds": {"nodes_cv2": c1 - c0, "match_port": c2 - c1, "graph_and_solve": c3 - c2},
                "cpu_frames_per_s": nf / (c3 - c0), "cpu_threads": usable_cpus(),
                "note": "oracle = cv2 ORB + reference glue + C port of matching / RANSAC / LM on the first frames of the same sequence"}
    finally:
        fe.params = old
        fe._check(fe.lib.rgbdslam_b200_init(local_rank, C.byref(old)))
    return out


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    from rgbdslam_v2_b200 import Frontend
    from rgbdslam_v2_b200._capi import default_params, PAIR_RESULT_DTYPE, DMATCH_DTYPE

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- rgbdslam_v2_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    prm = default_params()
    prm.depth_cov_z0 = 2.0  # fixed emulation of the depth_covariance static (same on all ranks and in the oracle)
    fe = Frontend(local_rank, prm)
    # A real (non-default) stream shared by torch and the library's slot 0: torch's legacy default stream has handle 0, which
    # rgbdslam_b200_set_stream reads as "use the library's own stream" -- the L2 flush and the timing events of the synchronous
    # reference point would then run concurrently with the kernels they are meant to bracket.
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    fe.set_stream(stream.cuda_stream)

    # Two independent batches (A/B) alternate between two pipeline slots: their resident inputs (2 x 156 MB of node
    # data incl. the int8 operands) exceed the 126 MB L2, so no explicit flush is needed between steps, and the
    # host->device copies / latency-bound RANSAC phases of step k+1 overlap the kernels of step k.
    # batches in flight (measured, 200 steps: depth 3 / 4 / 5 / 7 -> 1.62 / 1.71 / 1.75 / 1.73 M pairs/s on one GPU; with the
    # per-step all-gather every batch also waits for the slowest rank: 2 GPUs, depth 4 / 6 -> 3.20 / 3.37 M pairs/s)
    DEPTH = int(os.environ.get("RB200_BENCH_DEPTH", "5" if world == 1 else "6"))
    sets = []
    for j in range(DEPTH):
        b = make_workload(rank + j * world)
        first_pair = (rank + j * world) * PAIRS_PER_GPU
        newer = np.array([fe.node_from_features(int(b["id_newer"][i]), p["desc_newer"], p["xyz_newer"]) for i, p in enumerate(b["pairs"])], np.uint64)
        older = np.array([fe.node_from_features(int(b["id_older"][i]), p["desc_older"], p["xyz_older"]) for i, p in enumerate(b["pairs"])], np.uint64)
        pin = {k: torch.from_numpy(b[k]).pin_memory() for k in ("desc_newer", "xyz_newer", "desc_older", "xyz_older")}
        mm = prm.max_matches
        out_res = torch.zeros(PAIRS_PER_GPU * PAIR_RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        out_all = torch.zeros(PAIRS_PER_GPU * mm * DMATCH_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        out_inl = torch.zeros(PAIRS_PER_GPU * mm * DMATCH_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        sets.append(dict(b=b, first=first_pair, newer=newer, older=older, pin=pin, keep=(out_res, out_all, out_inl),
                         res=out_res.numpy().view(PAIR_RESULT_DTYPE),
                         allm=out_all.numpy().view(DMATCH_DTYPE).reshape(PAIRS_PER_GPU, mm),
                         inl=out_inl.numpy().view(DMATCH_DTYPE).reshape(PAIRS_PER_GPU, mm)))
    b, res_np = sets[0]["b"], sets[0]["res"]
    pin = sets[0]["pin"]
    out_res, out_all, out_inl = sets[0]["keep"]

    # the one exchange step of the multi-GPU path: all-gather of the edge records over NCCL (SURVEY 8e)
    comm = None
    all_edges = None
    if world > 1:
        uid = torch.from_numpy(fe.comm_unique_id() if rank == 0 else np.zeros(128, np.uint8)).cuda()
        dist.broadcast(uid, 0)
        comm = fe.comm_init(rank, world, uid.cpu().numpy())
    # edge records of every step of a timed region, all-gathered ONCE at its end (north star: "a single NCCL all-gather of the
    # resulting SE(3) edges before the global solve"; round 1 gathered every step: 8 ranks then rendezvous every 0.15 ms)
    local_edges = {"buf": None, "n": 0, "pin_buf": None, "pin_all": None}

    def pinned_records(n):
        t = torch.empty(n * PAIR_RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        return t, t.numpy().view(PAIR_RESULT_DTYPE)

    def reserve_exchange(K):
        """pinned host buffers for the region's edge records and their gathered union, and the communicator's device buffers at
        their final size -- allocated once, outside the timed regions (a fresh 30 MB pageable array per region cost the 8-GPU
        run a quarter of its timed region in page faults and a pageable device-to-host copy)"""
        if comm is None:
            return
        local_edges["pin_buf"] = pinned_records(K * PAIRS_PER_GPU)
        local_edges["pin_all"] = pinned_records(world * K * PAIRS_PER_GPU)
        local_edges["pin_buf"][1][:] = np.zeros(1, PAIR_RESULT_DTYPE)
        fe.allgather_edges(comm, local_edges["pin_buf"][1], world, out=local_edges["pin_all"][1])

    def submit_resident(k):
        st = sets[k % DEPTH]
        fe.submit_node_pairs(1 + k % DEPTH, st["newer"], st["older"], (st["res"], None, None), seed=SEED, first_pair_index=st["first"])

    def submit_e2e(k):
        st = sets[k % DEPTH]
        bb, pp = st["b"], st["pin"]
        fe.submit_pairs_host(1 + k % DEPTH, pp["desc_newer"], pp["xyz_newer"], bb["n_newer"], pp["desc_older"], pp["xyz_older"],
                             bb["n_older"], bb["id_newer"], bb["id_older"], (st["res"], st["allm"], st["inl"]), seed=SEED,
                             first_pair_index=st["first"])

    def finish(k, timed):
        """results of step k are on the host; N > 1: a timed step's are kept for the exchange at the end of the region"""
        fe.wait_slot(1 + k % DEPTH)
        if comm is not None and timed:
            n = local_edges["n"]
            local_edges["buf"][n:n + PAIRS_PER_GPU] = sets[k % DEPTH]["res"]
            local_edges["n"] = n + PAIRS_PER_GPU

    region = {}

    def run_steps(submit, K, lead=0, tail=0):
        """`lead` untimed steps, K timed steps and `tail` untimed steps back to back.  Returns the host seconds from the
        completion of the last lead step (from the call when lead == 0) to the completion of the last timed step, plus the
        exchange of the timed steps' records.  With lead >= DEPTH and tail == DEPTH - 1 the pipeline is full from the start to
        the end of that window, so it measures K steps of steady state."""
        if comm is not None:
            pin = local_edges["pin_buf"]
            local_edges["buf"] = pin[1][:K * PAIRS_PER_GPU] if pin is not None and len(pin[1]) >= K * PAIRS_PER_GPU else \
                np.zeros(K * PAIRS_PER_GPU, PAIR_RESULT_DTYPE)
            local_edges["n"] = 0
        n = lead + K + tail
        t = {"start": time.perf_counter()}

        def done(j):
            finish(j, lead <= j < lead + K)
            if j == lead - 1:
                t["start"] = time.perf_counter()
            elif j == lead + K - 1:
                t["end"] = time.perf_counter()
                last = sets[j % DEPTH]  # what the last timed step handed to its caller
                region["last"] = {k: last[k].copy() for k in ("res", "allm", "inl")}

        for k in range(n):
            if k >= DEPTH:
                done(k - DEPTH)
            if k == lead:
                launches0 = fe.launch_count
            elif k == lead + K:
                region["launches"] = fe.launch_count - launches0
            submit(k)
        if tail == 0:
            region["launches"] = fe.launch_count - launches0
        for j in range(max(0, n - DEPTH), n):
            done(j)
        dt = t["end"] - t["start"]
        if comm is not None:  # the one exchange: every rank ends up with every rank's edges of the whole region
            t0 = time.perf_counter()
            pin = local_edges["pin_all"]
            out = pin[1][:world * K * PAIRS_PER_GPU] if pin is not None and len(pin[1]) >= world * K * PAIRS_PER_GPU else None
            local_edges["all"] = fe.allgather_edges(comm, local_edges["buf"], world, out=out)
            dt += time.perf_counter() - t0
        return dt

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run_steps(submit_resident, max(args.warmup, DEPTH))
    run_steps(submit_e2e, max(args.warmup, DEPTH))

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- timed: device-resident inputs, pipelined over DEPTH slots ------------------------------------
    # exactly --steps K steps between DEPTH untimed steps that fill the pipeline and DEPTH - 1 that keep it full, so that a short
    # region measures neither the ramp nor the drain (20 steps of 0.15 ms are four pipeline turn-overs).  The host clock reads
    # after the stream synchronise of a step.
    timed_steps = args.steps
    reserve_exchange(timed_steps)
    barrier()
    resident_s = run_steps(submit_resident, timed_steps, lead=DEPTH, tail=DEPTH - 1)
    barrier()
    launches = region["launches"]
    resident_out = region["last"]["res"]
    ham_ms, dev_ms = [], []
    for j in range(DEPTH):
        h, t = fe.last_timing(1 + j)
        ham_ms.append(h); dev_ms.append(t)
    total_ms = torch.tensor([1e3 * resident_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    n_valid = int((res_np["id1"] >= 0).sum())

    # ---- timed: end to end through the host-buffer C ABI (pinned host buffers in, host results out) -----
    barrier()
    e2e_wall = run_steps(submit_e2e, timed_steps, lead=DEPTH, tail=DEPTH - 1)
    barrier()
    e2e_out = region["last"]
    if rank == 0 and args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, {
            "resident_results": resident_out, "e2e_results": e2e_out["res"],
            "e2e_all_matches": first_n(e2e_out["allm"], e2e_out["res"]["n_all_matches"]),
            "e2e_inlier_matches": first_n(e2e_out["inl"], e2e_out["res"]["n_inliers"])})
    e2e_total = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_total = float(e2e_total.item())

    # ---- reference point: the same step, one at a time (synchronous API, L2 flushed before every step) ----
    # READ a 256 MiB buffer (> 126 MB L2): the lines it leaves behind are clean.  (A memset flush leaves 126 MB of dirty lines
    # whose write-back lands inside the timed kernels: the cold Hamming launch then measures 86 us instead of the 53 us the
    # ncu launch list -- which invalidates the caches between kernels -- shows for the same cold launch.)
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.int32, device="cuda")
    sync_ms, sync_ham, sync_dev = [], [], []
    for k in range(3 + min(args.steps, 10)):
        flush_sink = flush.sum()
        a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fe.match_node_pairs(sets[0]["newer"], sets[0]["older"], seed=SEED, first_pair_index=sets[0]["first"], out=(res_np, None, None))
        c.record(stream)
        torch.cuda.synchronize()
        if k >= 3:
            sync_ms.append(a.elapsed_time(c))
            h, t = fe.last_timing(0)
            sync_ham.append(h); sync_dev.append(t)
    clocks = sampler.stop() if rank == 0 else None
    del flush

    c4 = None
    if not args.no_c4:
        try:
            c4 = bench_sequence(fe, local_rank, rank, world, comm, n_frames=args.c4_frames,
                                with_oracle=(world == 1 and not args.no_cpu_baseline))
        except Exception as ex:  # secondary measurements must never hide the headline line
            import traceback
            c4 = {"error": repr(ex), "trace": traceback.format_exc()[-800:]}

    if rank == 0:
        value = world * PAIRS_PER_GPU * timed_steps / (total_ms * 1e-3)
        e2e_value = world * PAIRS_PER_GPU * timed_steps / e2e_total
        peak, peak_src = measured_peaks()
        ham = statistics.mean(sync_ham)  # the kernel alone (one step at a time); pipelined launches share SMs with RANSAC
        achieved = ALGO_BYTES_PER_PAIR * PAIRS_PER_GPU / (ham * 1e-3) / 1e9
        h2d = sum(int(pin[k].numel() * pin[k].element_size()) for k in pin)
        mm = prm.max_matches
        d2h = int(out_res.numel() + out_all.numel() + out_inl.numel())
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / timed_steps, "timed_steps": timed_steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 descriptors (exact integer Hamming) + f32 fit + f64 Mahalanobis", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "l2": f"inputs larger than L2: {DEPTH} alternating batches = {DEPTH} x 156 MB resident node data (126 MB L2); "
                             "the synchronous reference point flushes L2 (a 256 MiB read) before every step",
                       "pipeline": f"{DEPTH} batches in flight on {DEPTH} library streams (rgbdslam_b200_match_pairs_submit / _wait)",
                       "pairs_per_gpu": PAIRS_PER_GPU,
                       "exchange": "none (1 GPU)" if world == 1 else f"ONE ncclAllGather of the {world} x {timed_steps} x {PAIRS_PER_GPU} edge records (120 B) of the region at its end (rgbdslam_b200_allgather_edges), inside the timed region",
                       "edges_gathered": None if comm is None else int((local_edges["all"]["id1"] >= 0).sum()),
                       "valid_edges_rank0": n_valid,
                       "timing": f"--steps {args.steps} timed back to back between {DEPTH} untimed steps that fill the pipeline "
                                 f"and {DEPTH - 1} that keep it full; host clock from the completion of the step before the first "
                                 "timed step to that of the last timed step"},
            "roofline": {"bound": "hbm", "kernel": "hamming_match", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": NCU_DRAM_BYTES_PER_LAUNCH, "traffic_source": NCU_TRAFFIC_SOURCE, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_PAIR * PAIRS_PER_GPU, "kernel_ms": ham,
                         "kernel_share_of_step": ham / statistics.mean(sync_dev),
                         "kernel_ms_when_pipelined": statistics.mean(ham_ms),
                         "tensor": tensor_roofline(ham),
                         "note": "binding resource is the integer/tensor pipe, not HBM (1e6 256-bit distance evals per 72 kB)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_total / timed_steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "device_ms_per_step": statistics.mean(dev_ms),
            "synchronous": {"value": PAIRS_PER_GPU / (statistics.mean(sync_ms) * 1e-3), "ms_per_step": statistics.mean(sync_ms),
                            "device_ms_per_step": statistics.mean(sync_dev), "note": "one batch at a time, L2 flushed, rank 0"},
        }
        out["c4"] = c4
        if c4 and "ate_vs_gt_m" in c4:  # the second half of BASELINE's metric: "...; ATE RMSE vs reference"
            op = c4.get("oracle_prefix") or {}
            out["ate"] = {"sequence": f"C4 ({c4.get('pairs')} pairs, {args.c4_frames} frames)", "ate_rmse_vs_ground_truth_m": c4["ate_vs_gt_m"],
                          "ate_rmse_gpu_vs_cpu_reference_path_m": op.get("ate_gpu_vs_oracle_m"),
                          "cpu_reference_path_ate_vs_ground_truth_m": op.get("ate_oracle_vs_gt_m"),
                          "cpu_reference_path_frames": op.get("frames"), "target": "within 1 mm of the reference path"}
        if world == 1 and not args.no_c3:
            try:
                out["c2_rendered"] = bench_c2_rendered(fe, local_rank, cpu=not args.no_cpu_baseline)
            except Exception as ex:
                import traceback
                out["c2_rendered"] = {"error": repr(ex), "trace": traceback.format_exc()[-800:]}
            try:
                out["c3"] = bench_c3(fe, local_rank, cpu=not args.no_cpu_baseline)
            except Exception as ex:
                import traceback
                out["c3"] = {"error": repr(ex), "trace": traceback.format_exc()[-800:]}
        if world == 1 and not args.no_cpu_baseline:
            try:
                if c4 and "node_constructor_frames_per_s" in c4:  # the Node constructor is measured inside the C4 sequence
                    op = c4.get("oracle_prefix") or {}
                    cs = (op.get("cpu_seconds") or {}).get("nodes_cv2")
                    out["node_create"] = {"metric": "node_constructor_frames_per_sec_640x480_1k_orb", "value": c4["node_constructor_frames_per_s"],
                                          "unit": "frames/s", "frames": args.c4_frames, "includes": "H2D of gray + depth from pinned host memory "
                                          "(mask derived from depth on the device), detect, describe, project",
                                          "h2d_GBps": c4["h2d_bytes"] / c4["seconds"]["nodes"] / 1e9,
                                          "cpu_cv2_value": (op.get("frames") / cs) if cs else None, "cpu_threads": usable_cpus()}
                out["posegraph"] = bench_posegraph(fe)
            except Exception as ex:  # secondary measurements must never hide the headline line
                out["secondary_error"] = repr(ex)
            from oracle import oracle
            oracle.build()
            dt1, _ = oracle_run(b, 0, 1, npairs=32)
            oracle_run(b, 0, usable_cpus())  # the first passes pay for the OpenMP team and the allocator arenas
            cores, thread_scan = pick_threads(b)
            dtn, ores = min((oracle_run(b, 0, cores) for _ in range(3)), key=lambda t: t[0])
            out["cpu_baseline"] = {"value": PAIRS_PER_GPU / dtn, "unit": UNIT, "cores": cores, "kind": "port",
                                   "cores_available": usable_cpus(), "pairs_per_s_by_thread_count": thread_scan,
                                   "sample": f"the same {PAIRS_PER_GPU} pairs x {N_KP} kp, best of 3 warm passes, OpenMP over pairs",
                                   "single_thread_value": 32 / dt1}
            agree = int(((ores["id1"] >= 0) == (res_np["id1"] >= 0)).sum())
            out["config"]["oracle_agreement_valid_flags"] = f"{agree}/{PAIRS_PER_GPU}"
        emit(out)
    if comm is not None:
        fe.comm_destroy(comm)
    fe.close()
    if world > 1:
        dist.destroy_process_group()


def first_n(matches: np.ndarray, n: np.ndarray) -> np.ndarray:
    """Row i keeps its first n[i] entries, the rest are zeroed: only those were written by the step."""
    out = matches.copy()
    out[np.arange(matches.shape[1])[None, :] >= n[:, None]] = np.zeros(1, matches.dtype)
    return out


def dump_outputs(d: Path, arrays: dict):
    """One DIR/<name>_<field>.npy per field of each structured array: float32 fields as they are, every other field as
    float64 (exact for these 32-bit integers).  Padding fields (trailing underscore) are left out."""
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        for f in a.dtype.names:
            if not f.endswith("_"):
                np.save(d / f"{name}_{f}.npy", a[f].astype(np.float32 if a[f].dtype == np.float32 else np.float64))


_JSON_OUT = None


def emit(out: dict):
    f = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    f.write(json.dumps(out) + "\n")
    f.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)  # 200 x 0.16 ms: long enough that one scheduling hiccup does not halve the number
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the 2000-frame sequence (config C4) sub-measurement")
    ap.add_argument("--c4-frames", type=int, default=C4_FRAMES)
    ap.add_argument("--no-c3", action="store_true", help="skip the SIFT-128 (config C3) sub-measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the results of the last timed step as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries the ONE JSON line and nothing else: libraries that write to file descriptor 1 on their own (NCCL prints its
    # version banner there at the first communicator) are sent to stderr; the line is written to the saved descriptor
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        import __graft_entry__ as g
        if local_rank == 0:
            g.build()
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
