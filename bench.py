#!/usr/bin/env python
"""bench.py -- stereo front-end throughput on B200 (BASELINE.json metric: stereo pairs/s @1241x376, ~2000 feat).

  python bench.py --gpus N --steps K --warmup W          our CUDA path (libjsfe.so through the C ABI)
  python bench.py --impl reference ...                    the CPU restatement of the reference's path on the host cores
  python bench.py ... --dump-outputs DIR                  also write the last timed step's results to DIR/*.npy

One "step" = one pass of the whole hot path (pyramid -> FAST/NMS -> compaction -> angle+blur+rBRIEF for both eyes,
then the left<->right Hamming + SAD stereo match) over a batch of `--pairs` synthetic stereo pairs per GPU.
`value`  : pairs/s with the level-0 images already resident in HBM (the handle's image slots).
`e2e`    : the same metric through the public API with HOST buffers: pinned H2D of every image and the D2H of
           every result slab inside the timed region.
Inputs: 2*pairs images of 1241x376 u8 per GPU per step = 150 MB at the default 160 pairs -> larger than the 126 MB L2,
so no L2 flush is needed between iterations (config.l2: "inputs>L2").
Timing: CUDA events on the launching stream, bracketed by barrier + synchronize, max over ranks.
Multi-GPU: pairs are independent -> one process per GPU, no data-path collective (weak scaling): `value` at N GPUs is that.  For
N > 1 the same line also carries `gather`: the step with the C ABI's jsfe_gather_* behind it (every rank's results, trimmed to the
keypoint counts, stored into rank 0's memory over NVLink on a side stream while the next batch is extracted), and `c5_batch_gather`:
BASELINE configs[4] (1920x1080, one pair per GPU, gathered).
Parity is asserted in the same run: the results of the timed configuration are compared with the committed reference goldens and with
the CPU oracle; any mismatch makes the run fail.
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

METRIC = "stereo front-end pairs/sec @1241x376, ~2000 feat (keypoints bit-exact vs ref)"
UNIT = "pairs/s"


def bytes_per_pair(levels_hw, cap):
    """SURVEY.md 8(d): compulsory traffic of a perfectly fused implementation, per stereo pair.
    bytes_pair = 2*[P0 + 2*sum(P_i>=1) + N*(24+32)] + N*(64 + 2*11*21 + 8)"""
    p0 = levels_hw[0][0] * levels_hw[0][1]
    prest = sum(h * w for h, w in levels_hw[1:])
    return 2 * (p0 + 2 * prest + cap * 56) + cap * (64 + 462 + 8)


def kernel_algorithmic_bytes(levels_hw, cap, n_mean):
    """Per-IMAGE (per-pair for the stereo kernels) algorithmic bytes of each kernel (DESIGN.md section 5)."""
    p0 = levels_hw[0][0] * levels_hw[0][1]
    prest = sum(h * w for h, w in levels_hw[1:])
    return {
        "k_pyramid": p0 + prest,                       # read L0 once, write every resampled level once
        "k_fast_cells": p0 + prest + 12 * cap,         # read every level once, write (x,y,score) per cell
        "k_blur": 2 * (p0 + prest),                     # read every level once, write its blurred copy (an implementation artefact)
        "k_compact": 12 * cap + 16 * n_mean,           # read cells, write compacted (x,y,score,level)
        "k_orient_desc": n_mean * (31 * 31 + 37 * 37 + 16 + 56 + 4),  # read disc + blurred window + kp, write SoA 24B + desc 32B + angle
        "k_stereo_match": n_mean * (64 + 462 + 8),     # per PAIR: 2 descriptors, two 11x21 strips, uRight+depth
        "k_stereo_outlier": n_mean * 4,                # per PAIR
        "k_nms_ms": 12 * cap,
    }


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (pynvml, fallback nvidia-smi)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel, units):
    """DRAM bytes per launch of `kernel`: dram__bytes_read+write per image (per pair for the stereo kernels) from the
    committed `ncu --set full` capture (profiles/traffic.json), scaled to the units one bench launch processes."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            per_unit = json.load(open(p)).get(kernel, {}).get("dram_bytes_per_unit")
            return None if per_unit is None else per_unit * units
        except Exception:
            return None
    return None


def workload_config(cfg, pairs_per_gpu):
    """The workload definition both arms print as `config` (identical keys and values; what a run measured goes elsewhere)."""
    return {"workload": cfg.name, "height": cfg.height, "width": cfg.width, "n_levels": cfg.n_levels, "tile": cfg.tile_h,
            "fast_threshold": cfg.th_fast_max, "fast_arc": [cfg.fast_n_min, cfg.fast_n_max], "pairs_per_step_per_gpu": pairs_per_gpu,
            "l2": "inputs>L2 (%.0f MB of level-0 images per step per GPU)" % (2 * pairs_per_gpu * cfg.height * cfg.width / 1e6)}


_FULL_AFFINITY = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None   # before any NUMA pinning


class full_affinity:
    """The CPU legs run on every host core the process started with, not on the NUMA node the GPU arm pinned itself to, so both
    arms search and use the same thread counts."""

    def __enter__(self):
        self.saved = os.sched_getaffinity(0) if _FULL_AFFINITY is not None else None
        if _FULL_AFFINITY is not None:
            os.sched_setaffinity(0, _FULL_AFFINITY)

    def __exit__(self, *exc):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)


def pin_to_gpu_numa(index):
    """Bind this process to the CPUs of the NUMA node its GPU hangs off, BEFORE pinned buffers are allocated (first touch): on the
    8-GPU box ranks 0-3 sit on node 0 and 4-7 on node 1, and unpinned uploads from the wrong socket cost ~5 % at N = 8."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:      # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": None}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:   # affinity is an optimisation, never a failure
        return {"numa_node": None, "note": repr(e)[:80]}


def best_cpu_threads(cfg, imgs, fixed=0):
    """All the host threads the port can USE: with SMT and shared caches the fastest count is often below os.cpu_count(), so try
    cores, cores/2 and cores/4 on a small sample and keep the best (both arms use this)."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if fixed:
        return max(1, min(cores, fixed)), {}
    tried = {}
    for t in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
        cpu_pairs_per_s(cfg, imgs, t, max(1, t // 4))                  # spin the threads up
        tried[t] = cpu_pairs_per_s(cfg, imgs, t, 2 * t)[0]
    return max(tried, key=tried.get), tried


def check_parity(cfg, pairs_seeds, get_pair, golden_dir, n_oracle=2):
    """Compare the results of the timed configuration with (1) the committed goldens of the reference's own kernels and (2) the CPU
    oracle.  get_pair(i) -> dict(kps_l, desc_l, kps_r, desc_r, u_right, depth) for the i-th distinct pair.  -> (checked, mismatches, notes)"""
    from jetson_slam_b200 import synth
    from oracle import oracle as orc
    checked, bad, notes = 0, 0, []

    def cmp(tag, got, want):
        nonlocal bad
        for k, w in want.items():
            g = got[k]
            same = g.shape == w.shape and (np.array_equal(g.view(np.int32), w.view(np.int32)) if g.dtype == np.float32 else np.array_equal(g, w))
            if not same:
                bad += 1
                notes.append(f"{tag}:{k}")

    for i, seed in enumerate(pairs_seeds):
        gp = os.path.join(golden_dir, f"ref_C2_seed{seed}.npz")
        if cfg.name.startswith("C2") and os.path.exists(gp):
            g = np.load(gp)
            cmp(f"golden seed{seed}", get_pair(i), {k: g[k] for k in ("kps_l", "desc_l", "kps_r", "desc_r", "u_right", "depth")})
            checked += 1
    for i, seed in list(enumerate(pairs_seeds))[:n_oracle]:
        L, R = synth.stereo_pair(cfg.height, cfg.width, seed)
        ol, orr = orc.Oracle(**cfg.extractor_kwargs()), orc.Oracle(**cfg.extractor_kwargs())
        kl, dl = ol.extract(L)
        kr, dr = orr.extract(R)
        ur, dp, _, _ = orc.stereo_match(ol, orr, kl, dl, kr, dr, cfg.mb, cfg.mbf)
        cmp(f"oracle seed{seed}", get_pair(i), dict(kps_l=kl, desc_l=dl, kps_r=kr, desc_r=dr, u_right=ur, depth=dp))
        checked += 1
    return checked, bad, notes


DUMP_BYTES = 64 << 20


def step_outputs(fe, n_pairs, stream):
    """What the device-resident step hands its caller (jsfe_get_keypoints / jsfe_get_stereo), as float arrays for --dump-outputs:
    the keypoint count of every slot and, for the pairs in `pairs` (all of them when they fit in DUMP_BYTES at full keypoint
    capacity, else a sample fixed by seed 0 and the batch size), their results concatenated in pair order.  kps_* rows are
    x, y, score, angle (degrees), octave, size."""
    per_pair = fe.max_kp * (2 * (6 + 32) + 4) * 4         # two eyes' keypoints and descriptors, four stereo rows of the left eye
    k = max(1, min(n_pairs, (DUMP_BYTES - 24 * n_pairs) // per_pair))
    pairs = np.arange(n_pairs) if k == n_pairs else np.sort(np.random.default_rng(0).choice(n_pairs, k, replace=False))
    chosen = set(pairs.tolist())
    n = np.zeros(2 * n_pairs)
    cols = {key: [] for key in ("kps_l", "desc_l", "kps_r", "desc_r", "u_right", "depth", "best_idx_r", "best_dist")}
    for p in range(n_pairs):
        kl, dl = fe.get_keypoints(2 * p, stream)
        kr, dr = fe.get_keypoints(2 * p + 1, stream)
        n[2 * p], n[2 * p + 1] = kl.shape[1], kr.shape[1]
        if p not in chosen:
            continue
        for key, kps in (("kps_l", kl), ("kps_r", kr)):
            f = kps.astype(np.float32)
            f[3] = kps[3].view(np.float32)                    # the angle row holds float32 bits
            cols[key].append(f)
        cols["desc_l"].append(dl.astype(np.float32))
        cols["desc_r"].append(dr.astype(np.float32))
        for key, a in zip(("u_right", "depth", "best_idx_r", "best_dist"), fe.get_stereo(p, stream)):
            cols[key].append(a.astype(np.float32))
    out = {"n_keypoints": n, "pairs": pairs.astype(np.float64)}
    for key, parts in cols.items():
        out[key] = np.concatenate(parts, axis=1 if key.startswith("kps") else 0)
    return out


# ------------------------------------------------------------------------------------------------ CPU legs
_CPU_CTX_POOL = {}


def cpu_pairs_per_s(cfg, pairs_imgs, threads, pairs_total):
    """Time the oracle (CPU restatement of the reference's path) on `threads` host threads, one stereo pair per task."""
    from oracle import oracle as orc
    import ctypes as C
    kw = cfg.extractor_kwargs()
    # per-thread contexts and output buffers are kept across calls: a fresh context is ~20 MB of untouched pages, and first-touch
    # page faults of 128 threads inside a short timed pass (they serialise on the process's address-space lock) used to make the
    # port look slower on 64 and 128 threads than on 32
    pool = _CPU_CTX_POOL.setdefault(cfg.name, [])
    while len(pool) < threads:
        ctx = (orc.Oracle(**kw), orc.Oracle(**kw))
        cap = ctx[0].max_kp
        pool.append((ctx, dict(kl=np.zeros(6 * cap, np.int32), dl=np.zeros(32 * cap, np.uint8), kr=np.zeros(6 * cap, np.int32),
                               dr=np.zeros(32 * cap, np.uint8), ur=np.zeros(cap, np.float32), dp=np.zeros(cap, np.float32),
                               nr=C.c_int32())))
    ctxs = [p[0] for p in pool[:threads]]
    bufs = [p[1] for p in pool[:threads]]
    L = orc.lib()
    counter = {"next": 0}
    lock = threading.Lock()

    def worker(t):
        ol, orr = ctxs[t]
        b = bufs[t]
        while True:
            with lock:
                i = counter["next"]
                counter["next"] += 1
            if i >= pairs_total:
                return
            il, ir = pairs_imgs[i % len(pairs_imgs)]
            L.orc_stereo_pair(ol._h, orr._h, il.ctypes.data, ir.ctypes.data, cfg.mb, cfg.mbf, b["kl"].ctypes.data,
                              b["dl"].ctypes.data, C.byref(b["nr"]), b["kr"].ctypes.data, b["dr"].ctypes.data,
                              b["ur"].ctypes.data, b["dp"].ctypes.data, 1)

    ths = [threading.Thread(target=worker, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return pairs_total / dt, dt


def _ref_cuda_inproc(cfg, pair, iters=40):
    from oracle import ref
    if not ref.available():
        return None
    kw = cfg.extractor_kwargs()
    rl, rr = ref.RefEye(**kw), ref.RefEye(**kw)
    ref.time_pairs(rl, rr, pair[0], pair[1], cfg.mb, cfg.mbf, 10, True)
    out = {}
    for two in (True, False):
        dt = ref.time_pairs(rl, rr, pair[0], pair[1], cfg.mb, cfg.mbf, iters, two)
        out["two_threads" if two else "one_thread"] = iters / dt
    rl.close()
    rr.close()
    return {"value": max(out.values()), "unit": UNIT, "detail": out, "iters": iters,
            "how": "ORB_GPU::extract x2 (host images, its own H2D/D2H) + ORB_compute_stereo_match, wall clock, in a fresh process"}


def ref_cuda_pairs_per_s(cfg, seed=0, iters=40):
    """The reference's own src/cuda (compiled unmodified for sm_100a, oracle/_ref) driven like Frame::Frame does.  Run in a
    fresh interpreter without torch: the reference allocates, frees and creates a cuBLAS handle per frame, and those driver
    calls were measured 4-10x slower inside a process that already holds a torch CUDA context and this library's arenas."""
    import subprocess
    key = [k for k, v in __import__("jetson_slam_b200.configs", fromlist=["CONFIGS"]).CONFIGS.items() if v is cfg][0]
    code = ("import json,sys; sys.path.insert(0, %r); import bench; from jetson_slam_b200 import synth; from jetson_slam_b200.configs import CONFIGS; "
            "cfg = CONFIGS[%r]; print(json.dumps(bench._ref_cuda_inproc(cfg, synth.stereo_pair(cfg.height, cfg.width, %d), %d)))"
            % (ROOT, key, seed, iters))
    try:
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
        last = [l for l in r.stdout.strip().splitlines() if l.startswith("{") or l == "null"]
        if r.returncode != 0 or not last:
            return {"unavailable": (r.stderr or r.stdout)[-200:]}
        return json.loads(last[-1])
    except Exception as e:  # the reference library is optional colour, never the measured product
        return {"unavailable": repr(e)[:200]}


def compat_api_fps(cfg, pair, frames=300):
    """The reference-API path a Jetson-SLAM user calls, through compat/: tests/cpp/frame_hotpath replays Frame::Frame's hot path (two
    extractor threads on two ORBExtractor shims, 4 D2H, SoA unpack, ORB_compute_stereo_match; src/Frame.cpp:103-122,124-196,780-803)
    `frames` times.  Compare with ref_cuda.detail.two_threads: the reference's own kernels under the same call pattern."""
    import subprocess
    import tempfile
    exe = os.path.join(ROOT, "tests", "cpp", "frame_hotpath")
    if not os.path.exists(exe):
        return {"unavailable": "tests/cpp/frame_hotpath not built"}
    try:
        with tempfile.TemporaryDirectory() as d:
            lp, rp, op = (os.path.join(d, n) for n in ("l.raw", "r.raw", "o.bin"))
            pair[0].tofile(lp)
            pair[1].tofile(rp)
            cmd = [exe, str(cfg.height), str(cfg.width), str(cfg.n_levels), str(cfg.scale_factor), str(cfg.fast_n_min), str(cfg.fast_n_max),
                   str(cfg.th_fast_min), str(cfg.th_fast_max), str(cfg.tile_h), str(cfg.tile_w), lp, rp, repr(cfg.mb), repr(cfg.mbf), op,
                   "--time", str(frames)]
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        fps = [float(l.split()[1]) for l in r.stdout.splitlines() if l.startswith("fps ")]
        if r.returncode != 0 or not fps:
            return {"unavailable": (r.stderr or r.stdout)[-200:]}
        return {"value": fps[0], "unit": UNIT, "frames": frames,
                "how": "compat/ shims driven like Frame::Frame (2 extractor threads, 4 D2H, unpack, stereo match), one pair at a time, wall clock"}
    except Exception as e:
        return {"unavailable": repr(e)[:200]}


def sbp_microbench(iters=200):
    """SURVEY.md 8(f1): ORBmatcher::SearchByProjection fused on the device, on the C4-sized synthetic problem (3412 keypoints),
    timed with CUDA events (grid build + search per call) beside the CPU restatement (one thread) of the reference's host loops."""
    import torch
    from jetson_slam_b200 import frontend, synth
    from oracle import oracle as orc
    last, cur, R, t = synth.projection_scene(n_cur=3412, n_last=3412, seed=7)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dl, dc, dR, dt = {k: d(v) for k, v in last.items()}, {k: d(v) for k, v in cur.items()}, d(R), d(t)
    sf = np.cumprod(np.array([1.0] + [1.2] * 7, np.float32)).astype(np.float32)
    kw = dict(**synth.SBP_K, **synth.SBP_BOUNDS, mbf=synth.SBP_MBF, th=7.0, scale_factors=sf, level_mode=0)
    for _ in range(10):
        out = frontend.search_by_projection(dl, dc, dR, dt, **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        out = frontend.search_by_projection(dl, dc, dR, dt, **kw)
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / iters
    t0 = time.perf_counter()
    for _ in range(5):
        want = orc.search_by_projection(last, cur, R, t, **kw)
    cpu_ms = (time.perf_counter() - t0) / 5 * 1e3
    same = int(out["n_matches"].cpu()[0]) == want["nmatches"] and np.array_equal(out["cur_match"].cpu().numpy(), want["cur_match"])
    return {"n_last": 3412, "n_cur": 3412, "matches": want["nmatches"], "device_ms_per_call": dev_ms, "cpu_port_ms_per_call": cpu_ms,
            "identical_to_cpu_port": bool(same), "how": "jsfe_build_frame_grid + jsfe_search_by_projection (3 kernels + 3 memsets) per call, "
            "device-resident inputs, CUDA events over %d calls; CPU = oracle restatement of the host loops, 1 thread" % iters}


def remap_microbench(n_images=64, iters=50):
    """SURVEY.md 8(f3): device rectification (cv::remap INTER_LINEAR semantics) of a batch of EuRoC-size frames sharing one
    map pair.  Algorithmic bytes per launch: n * (src h*w read + dst h*w write) + 8 B/px of maps once."""
    import torch
    from jetson_slam_b200 import frontend
    h, w = 480, 752
    rng = np.random.default_rng(5)
    xs, ys = np.meshgrid(np.arange(w, dtype=np.float32), np.arange(h, dtype=np.float32))
    r2 = ((xs - w / 2) ** 2 + (ys - h / 2) ** 2) / np.float32(w * w)
    mx = torch.from_numpy((xs + (xs - w / 2) * 0.1 * r2 + 0.37).astype(np.float32)).cuda()
    my = torch.from_numpy((ys + (ys - h / 2) * 0.1 * r2 - 0.21).astype(np.float32)).cuda()
    src = torch.from_numpy(rng.integers(0, 256, size=(n_images, h, w), dtype=np.uint8)).cuda()
    out = torch.empty_like(src)
    for _ in range(5):
        frontend.remap_bilinear(src, mx, my, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        frontend.remap_bilinear(src, mx, my, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    alg = n_images * 2 * h * w + 8 * h * w
    peak, _ = measured_hbm_peak()
    return {"images": n_images, "height": h, "width": w, "ms_per_launch": ms, "us_per_image": ms * 1e3 / n_images,
            "alg_bytes_per_launch": alg, "gbs": alg / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": alg / (ms * 1e-3) / 1e9 / peak}


def opencv_orb_pairs_per_s(cfg, pair, iters=5):
    """Colour only, NOT parity-comparable (a different algorithm: the reference contains no OpenCV extractor): OpenCV's CPU ORB
    (cv2.ORB_create(2000, 1.2, 8)) on both eyes + brute-force Hamming matching, one thread."""
    try:
        import cv2
        cv2.setNumThreads(1)
        orb = cv2.ORB_create(nfeatures=2000, scaleFactor=1.2, nlevels=cfg.n_levels)
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        L, R = pair
        orb.detectAndCompute(L, None)
        t0 = time.perf_counter()
        for _ in range(iters):
            kl, dl = orb.detectAndCompute(L, None)
            kr, dr = orb.detectAndCompute(R, None)
            if dl is not None and dr is not None:
                bf.match(dl, dr)
        dt = (time.perf_counter() - t0) / iters
        return {"value": 1.0 / dt, "unit": UNIT, "cores": 1, "keypoints": len(kl), "note": "OpenCV %s CPU ORB + BFMatcher; different algorithm, not parity-comparable" % cv2.__version__}
    except Exception as e:
        return {"unavailable": repr(e)[:120]}


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from jetson_slam_b200 import synth
    imgs = [synth.stereo_pair(cfg.height, cfg.width, s) for s in range(4)]
    threads, tried = best_cpu_threads(cfg, imgs, args.cpu_threads)
    # bounded sample: a step is at most four pairs per host thread, and the K steps together about 30 s of wall clock
    rate = max(tried.values()) if tried else cpu_pairs_per_s(cfg, imgs, threads, 2 * threads)[0]
    per_step = max(1, min(4 * threads, int(rate * 30.0 / max(1, args.steps))))
    for _ in range(max(0, min(args.warmup, 3) - 1)):
        cpu_pairs_per_s(cfg, imgs, threads, max(1, per_step // 4))
    steps = args.steps
    t_total, n_total = 0.0, 0
    for _ in range(steps):
        v, dt = cpu_pairs_per_s(cfg, imgs, threads, per_step)
        t_total += dt
        n_total += per_step
    value = n_total / t_total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": dict(workload_config(cfg, args.pairs), parallelism=f"{threads} host threads on rank 0, one pair per thread; no GPU"),
        "note": "the reference has no CPU extractor/matcher (SURVEY F2/F3); this arm is the CPU restatement (oracle port) of its CUDA "
                "path, one pair per host thread, on a bounded sample of the workload",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n_total} {cfg.name.split()[0]} stereo pairs over {steps} timed passes, {threads} threads",
                         "threads_tried": {str(k): v for k, v in tried.items()}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:
        import torch
        if torch.cuda.is_available():
            line["ref_cuda"] = ref_cuda_pairs_per_s(cfg)
    except Exception:
        pass
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    from jetson_slam_b200 import frontend, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU port)")
    numa = pin_to_gpu_numa(local)           # before any pinned allocation
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the communicator is created; the contract is ONE JSON line on
        # stdout, so file descriptor 1 points at stderr while the communicator comes up
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

    B = args.pairs
    # distinct synthetic pairs cycled over the slots.  Rank 0 starts with seeds 0 and 1: the committed goldens of the reference's
    # own kernels exist for them (tests/golden/ref_C2_seed{0,1}.npz), so the timed batch itself is checked against the reference.
    n_distinct = min(B, args.distinct)
    seeds = [s if (rank == 0 and s < 2) else 1000 * rank + s for s in range(n_distinct)]
    pairs = [synth.stereo_pair(cfg.height, cfg.width, sd) for sd in seeds]
    # colour only: the reference's own src/cuda on this GPU, timed before this process owns any device memory of ours
    # (it allocates and frees per frame, which gets slower the more the process has mapped)
    ref_cuda = ref_cuda_pairs_per_s(cfg, seeds[0]) if (rank == 0 and world == 1 and not args.no_ref_cuda) else None
    fe = frontend.Frontend(**cfg.extractor_kwargs(), device=local, max_images=2 * B)
    # input images: pinned host memory from jsfe_host_alloc, write-combined unless --host-cached (the producer only writes it;
    # uploads that are not snooped through the CPU caches are worth ~5 % of e2e once several GPUs of a socket upload at once)
    host_buf = frontend.HostBuffer((2 * B, cfg.height, cfg.width), np.uint8, write_combined=not args.host_cached)
    hv = host_buf.array
    for p in range(B):
        hv[2 * p], hv[2 * p + 1] = pairs[p % n_distinct]
    stream = torch.cuda.Stream()
    fe.set_images(hv, 0, stream)
    stream.synchronize()
    # the second handle: two batches in flight in the e2e loop, and the other half of the double buffer when results are gathered
    fe_b = frontend.Frontend(**cfg.extractor_kwargs(), device=local, max_images=2 * B)
    fe_b.set_images(hv, 0, stream)
    stream.synchronize()
    fes = (fe, fe_b)

    def step_device():
        fe.extract(0, 2 * B, stream)
        fe.stereo_match(cfg.mb, cfg.mbf, 0, B, stream=stream)

    def step_e2e():
        # the public blocking end-to-end call: host images in, host result slabs out (chunked 3-stream pipeline inside)
        return fe.process_host_pairs(hv, cfg.mb, cfg.mbf, chunk_pairs=args.chunk)

    # half-batch chunks: measured 41.5 k pairs/s vs 41.2 k (chunks of 32) and 30.9 k (one 160-pair chunk: a single long upload
    # does not overlap the other handle's kernels)
    ovl_chunk = int(os.environ.get("BENCH_OVL_CHUNK", max(1, B // 2)))

    def steps_e2e_overlapped(k_steps, stamps=None):
        fes[0].process_host_pairs_begin(hv, cfg.mb, cfg.mbf, chunk_pairs=ovl_chunk)
        for k in range(1, k_steps):
            fes[k % 2].process_host_pairs_begin(hv, cfg.mb, cfg.mbf, chunk_pairs=ovl_chunk)
            fes[(k - 1) % 2].process_host_pairs_end()
            if stamps is not None:
                stamps.append(time.perf_counter())
        r = fes[(k_steps - 1) % 2].process_host_pairs_end()
        if stamps is not None:
            stamps.append(time.perf_counter())
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize; CUDA events on the launching stream around the region and after every step."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        ev[0].record(stream)
        for k in range(steps):
            fn(k)
            ev[k + 1].record(stream)
        stream.synchronize()
        barrier()
        per = np.array([ev[k].elapsed_time(ev[k + 1]) for k in range(steps)])
        return max_over_ranks(ev[0].elapsed_time(ev[steps])), per

    warm = max(3, args.warmup)
    for _ in range(warm):
        step_device()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = fe.launch_count()
    ms, per_step = timed(lambda k: step_device(), args.steps)
    launches = fe.launch_count() - l0
    clocks = sampler.stop()
    value = world * B * args.steps / (ms / 1e3)
    # read before the e2e legs below reuse the handle's slots
    outputs = step_outputs(fe, B, stream) if (rank == 0 and args.dump_outputs) else None

    # ---- parity of the timed configuration (device-resident results of the distinct pairs), asserted in this run
    parity = None
    if rank == 0 and not args.no_parity:
        stream.synchronize()

        def dev_pair(i):
            kl, dl = fe.get_keypoints(2 * i)
            kr, dr = fe.get_keypoints(2 * i + 1)
            ur, dp, _, _ = fe.get_stereo(i)
            return dict(kps_l=kl, desc_l=dl, kps_r=kr, desc_r=dr, u_right=ur, depth=dp)
        n_chk = min(n_distinct, 4)
        checked, bad, notes = check_parity(cfg, seeds[:n_chk], dev_pair, os.path.join(ROOT, "tests", "golden"))
        parity = {"checked_pairs": checked, "mismatches": bad, "against": "tests/golden/ref_C2_seed*.npz (the reference's own kernels) + CPU oracle",
                  "path": "device-resident", "notes": notes[:8]}

    # ---- e2e: host buffers in, host results out, every step
    for _ in range(2):
        step_e2e()
    # the e2e call is synchronous (it returns with the results on the host), so its time is wall-clock, max over ranks
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    ms_e2e_serial = max_over_ranks((time.perf_counter() - t0) * 1e3)
    barrier()
    e2e_serial = world * B * args.steps / (ms_e2e_serial / 1e3)
    # two batches in flight (begin/end over two handles): every step still uploads its 2*B images and downloads its result slabs
    steps_e2e_overlapped(3)
    barrier()
    stamps = [time.perf_counter()]
    steps_e2e_overlapped(args.steps, stamps)
    torch.cuda.synchronize()
    wall_e2e = time.perf_counter() - stamps[0]
    ms_e2e = max_over_ranks(wall_e2e * 1e3)
    e2e_per_step = np.diff(np.array(stamps)) * 1e3
    barrier()
    res = step_e2e()
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    n_mean = float(res["n"].mean())
    d2h = int(res["bytes"])
    matched = int((res["u_right"][0::2] >= 0).sum())
    if parity is not None:     # the same pairs through the host-to-host call
        cap = res["kps"].shape[2]

        def e2e_pair(i):
            nl, nr = int(res["n"][2 * i]), int(res["n"][2 * i + 1])
            return dict(kps_l=np.array(res["kps"][2 * i, :, :nl]), desc_l=np.array(res["desc"][2 * i, :nl]), kps_r=np.array(res["kps"][2 * i + 1, :, :nr]),
                        desc_r=np.array(res["desc"][2 * i + 1, :nr]), u_right=np.array(res["u_right"][2 * i, :nl]), depth=np.array(res["depth"][2 * i, :nl]))
        c2, b2, n2 = check_parity(cfg, seeds[:min(n_distinct, 4)], e2e_pair, os.path.join(ROOT, "tests", "golden"), n_oracle=1)
        parity["e2e_checked_pairs"], parity["e2e_mismatches"] = c2, b2
        parity["notes"] = (parity["notes"] + n2)[:8]
    # what the PCIe link alone gives for this step's input (pinned host -> device, nothing else running): the floor under e2e
    dev_in = torch.empty((2 * B, cfg.height, cfg.width), dtype=torch.uint8, device="cuda")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        import ctypes as C
        rt = C.CDLL("libcudart.so.12")     # the runtime torch has already loaded
        rt.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    except OSError:
        rt = None

    def upload():
        rt.cudaMemcpyAsync(dev_in.data_ptr(), hv.ctypes.data, hv.nbytes, 1, torch.cuda.current_stream().cuda_stream)

    h2d_ms = None
    if rt is not None:
        upload()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(3):
            upload()
        ev1.record()
        torch.cuda.synchronize()
        h2d_ms = ev0.elapsed_time(ev1) / 3
    del dev_in

    # ---- N > 1: the same step with the results gathered on rank 0 (jsfe_gather_*), double-buffered over the two handles so that the
    #      transfer of batch k overlaps the extraction of batch k+1
    gather_info = None
    if world > 1 and not args.no_gather:
        from jetson_slam_b200 import distributed as jd
        gs = [jd.Gatherer(f, B, root=0, transport=args.gather_transport) for f in fes]

        def step_gather(k):
            f, g = fes[k % 2], gs[k % 2]
            if k >= 2:
                g.end()                                  # batch k-2 of this handle has landed (and the root has released its buffer)
            f.extract(0, 2 * B, stream)
            f.stereo_match(cfg.mb, cfg.mbf, 0, B, stream=stream)
            g.begin(0, B, stream)

        def drain(k_steps):
            for k in range(max(0, k_steps - 2), k_steps):
                gs[k % 2].end()
        for k in range(4):
            step_gather(k)
        drain(4)
        barrier()
        t0 = time.perf_counter()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for k in range(args.steps):
            step_gather(k)
        ev1.record(stream)
        drain(args.steps)
        stream.synchronize()
        wall = max_over_ranks((time.perf_counter() - t0) * 1e3)       # includes the last transfers (nothing left in flight)
        barrier()
        gval = world * B * args.steps / (wall / 1e3)
        # where a gather's time goes on its own stream (all of it overlaps the next extraction): stage times of 8 more steps per rank
        for g in gs:
            g.profile(True)
        acc = np.zeros(4)
        nprof = 8
        for k in range(nprof + 2):
            step_gather(k)
            if k >= 2:
                acc += np.array(list(gs[k % 2].stage_times().values()))   # of the gather end() just returned (batch k-2)
        drain(nprof + 2)
        for g in gs:
            g.profile(False)
        st_t = torch.tensor(acc / nprof, device="cuda", dtype=torch.float64)
        st_all = [torch.zeros_like(st_t) for _ in range(world)]
        dist.all_gather(st_all, st_t)
        st_all = np.stack([t.cpu().numpy() for t in st_all])
        last = gs[(args.steps - 1) % 2].last
        payload = None
        if rank == 0:
            regs = gs[(args.steps - 1) % 2].regions_to_host(last)
            payload = [int(len(r)) for r in regs]
            u = jd.unpack_region(regs[-1])               # the farthest rank's region decodes and carries that rank's batch
            assert u["rank"] == world - 1 and u["n_pairs"] == B
        gather_info = {"value": gval, "unit": UNIT, "efficiency_vs_no_gather": gval / value, "ms_per_step": wall / args.steps,
                       "transport": gs[0].transport, "bytes_per_rank_per_step": payload,
                       "stages_us": {"stages": list(jd.Gatherer.STAGES), "root": [round(float(x), 1) for x in st_all[0]],
                                     "max_over_ranks": [round(float(x), 1) for x in st_all.max(axis=0)],
                                     "how": "CUDA events on each rank's gather stream (jsfe_gather_profile), mean of %d gathers; the credit "
                                            "all-reduce ends when the slowest rank has joined" % nprof},
                       "how": "extract + match + jsfe_gather_begin per step, alternating two handles (batch k is packed and stored into rank 0's "
                              "memory on the gather stream while batch k+1 is extracted); wall clock incl. the final transfers, max over ranks"}
        for g in gs:
            g.close()

    # ---- BASELINE configs[4]: C5 1920x1080, one pair per GPU, gathered (latency of a batch request over all GPUs)
    c5 = None
    if world > 1 and not args.no_gather:
        from jetson_slam_b200 import distributed as jd
        from jetson_slam_b200.configs import CONFIGS
        c5cfg = CONFIGS["C5"]
        f5 = frontend.Frontend(**c5cfg.extractor_kwargs(), device=local, max_images=2)
        p5 = synth.stereo_pair(c5cfg.height, c5cfg.width, 7000 + rank)
        f5.set_images(np.stack(p5), 0, stream)
        g5 = jd.Gatherer(f5, 1, root=0, transport=args.gather_transport)

        def c5_batch():
            f5.extract(0, 2, stream)
            f5.stereo_match(c5cfg.mb, c5cfg.mbf, 0, 1, stream=stream)
            g5.begin(0, 1, stream)
            g5.end()
        for _ in range(5):
            c5_batch()
        barrier()
        t0 = time.perf_counter()
        n5 = 50
        for _ in range(n5):
            c5_batch()
        wall5 = max_over_ranks((time.perf_counter() - t0) * 1e3)
        barrier()
        c5 = {"workload": c5cfg.name, "pairs_per_batch": world, "ms_per_batch": wall5 / n5, "value": world * n5 / (wall5 / 1e3), "unit": UNIT,
              "transport": g5.transport, "how": "one pair per GPU (device-resident images), extract + match + gather to rank 0, each batch waited for"}
        g5.close()
        f5.close()

    # single-pair latency (the reference's real-time use: one frame at a time), host images in -> host results out
    lat = None
    if rank == 0:
        fe1 = frontend.Frontend(**cfg.extractor_kwargs(), device=local, max_images=2)
        one = torch.empty((2, cfg.height, cfg.width), dtype=torch.uint8).pin_memory()
        one.numpy()[0], one.numpy()[1] = pairs[0]
        for _ in range(20):
            fe1.process_host_pairs(one.numpy(), cfg.mb, cfg.mbf, chunk_pairs=1)
        ts = []
        for _ in range(200):
            t0 = time.perf_counter()
            fe1.process_host_pairs(one.numpy(), cfg.mb, cfg.mbf, chunk_pairs=1)
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e3
        lat = {"pairs_in_flight": 1, "median_ms": float(np.median(ts)), "p95_ms": float(np.percentile(ts, 95)),
               "how": "jsfe_process_host_pairs(1 pair): pinned H2D + one CUDA-graph launch (re-pitch, kernels, result copies) + sync, wall clock, 200 iterations"}

    # per-kernel durations (CUDA events on the launching stream around every launch)
    fe.profile(True)
    prof_steps = min(args.steps, 20)
    for _ in range(prof_steps):
        step_device()
    stream.synchronize()
    prof = fe.profile_read()
    fe.profile(False)
    levels = [(li.height, li.width) for li in fe.levels]
    alg = kernel_algorithmic_bytes(levels, fe.max_kp, n_mean)
    per_kernel = {}
    for k, (tot_ms, cnt) in prof.items():
        if cnt:
            units = B if k.startswith("k_stereo") else 2 * B
            per_kernel[k] = {"ms_per_launch": tot_ms / cnt, "alg_bytes_per_launch": alg[k] * units}
    total_k = sum(v["ms_per_launch"] for v in per_kernel.values()) or 1.0
    for v in per_kernel.values():
        v["share"] = v["ms_per_launch"] / total_k
        v["gbs"] = v["alg_bytes_per_launch"] / (v["ms_per_launch"] * 1e-3) / 1e9
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_per_launch"])
    peak, peak_src = measured_hbm_peak()
    bpp = bytes_per_pair(levels, fe.max_kp)

    def device_ladder():
        # device-resident ladder (SURVEY 8d): 1 / 8 / 64 pairs in flight, stream launches vs one CUDA-graph replay
        sweep = {}
        for nb in (1, 8, 64):
            if nb > B:
                continue

            def small():
                fe.extract(0, 2 * nb, stream)
                fe.stereo_match(cfg.mb, cfg.mbf, 0, nb, stream=stream)

            for _ in range(5):
                small()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            stream.synchronize()
            e0.record(stream)
            for _ in range(50):
                small()
            e1.record(stream)
            stream.synchronize()
            ent = {"stream_ms": e0.elapsed_time(e1) / 50}
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream):
                    small()
                for _ in range(5):
                    g.replay()
                torch.cuda.synchronize()
                e0.record()
                for _ in range(50):
                    g.replay()
                e1.record()
                torch.cuda.synchronize()
                ent["graph_ms"] = e0.elapsed_time(e1) / 50
                del g
            except Exception as e:  # capture is optional colour
                ent["graph_error"] = repr(e)[:160]
                torch.cuda.synchronize()
            ent["pairs_per_s"] = nb / (min(ent.get("graph_ms", 1e9), ent["stream_ms"]) / 1e3)
            sweep[str(nb)] = ent
        return sweep

    if rank == 0:
        if lat is not None and world == 1:
            lat["device_resident_ladder"] = device_ladder()
        with full_affinity():
            cpu_threads, cpu_tried = best_cpu_threads(cfg, pairs[: min(4, len(pairs))], args.cpu_threads)
            sample_pairs = 20 * cpu_threads   # a bounded sample of the same workload: ~20 s of CPU work
            cpu_v, cpu_dt = cpu_pairs_per_s(cfg, pairs[: min(4, len(pairs))], cpu_threads, sample_pairs)
        config = workload_config(cfg, B)
        config["parallelism"] = f"pairs sharded one-batch-per-GPU x{world}, no data-path collective in `value`" + ("; `gather` adds the exchange step" if gather_info else "")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": config,
            "workload_stats": {"max_keypoints_per_eye": fe.max_kp, "mean_keypoints_per_eye": n_mean, "stereo_matches_per_step": matched,
                               "distinct_pairs": n_distinct, "numa": numa},
            "step_ms": {"median": float(np.median(per_step)), "p95": float(np.percentile(per_step, 95)), "min": float(per_step.min()),
                        "max": float(per_step.max()), "n": int(len(per_step)), "how": "CUDA events after every step on the launching stream (this rank)"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(2 * B * cfg.height * cfg.width),
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps, "wall_s": wall_e2e,
                    "step_ms": {"median": float(np.median(e2e_per_step)), "p95": float(np.percentile(e2e_per_step, 95)), "n": int(len(e2e_per_step))},
                    "how": "jsfe_process_host_pairs_begin/_end, two handles alternating (a batch uploads while the previous one computes); "
                           "pinned host images in, pinned host result slabs out, wall clock over all steps",
                    "blocking_call": {"value": e2e_serial, "unit": UNIT, "ms_per_step": ms_e2e_serial / args.steps,
                                      "how": "one jsfe_process_host_pairs call per step (chunked 3-stream pipeline inside), nothing else in flight"},
                    "h2d_only_ms_per_step": h2d_ms, "h2d_only_gbs": 2 * B * cfg.height * cfg.width / h2d_ms / 1e6 if h2d_ms else None,
                    "host_input": "jsfe_host_alloc, " + ("cached pinned" if args.host_cached else "write-combined pinned")},
            "gpu_launches": int(launches),
            "parity": parity,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": per_kernel[dom]["gbs"], "peak": peak, "unit": "GB/s",
                         "frac": per_kernel[dom]["gbs"] / peak, "traffic": ncu_traffic(dom, B if dom.startswith("k_stereo") else 2 * B), "peak_source": peak_src,
                         "ms_per_launch": per_kernel[dom]["ms_per_launch"], "share_of_step": per_kernel[dom]["share"]},
            "pipeline_roofline": {"bytes_per_pair": bpp, "achieved": bpp * value / world / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": bpp * value / world / 1e9 / peak},
            "kernels": per_kernel,
            "latency": lat,
            "cpu_baseline": {"value": cpu_v, "unit": UNIT, "cores": cpu_threads, "kind": "port",
                             "sample": f"{sample_pairs} {cfg.name.split()[0]} stereo pairs on {cpu_threads} threads ({cpu_dt:.1f} s wall)",
                             "threads_tried": {str(k): v for k, v in cpu_tried.items()}},
        }
        if gather_info is not None:
            line["gather"] = gather_info
        if c5 is not None:
            line["c5_batch_gather"] = c5
        if ref_cuda is not None:
            line["ref_cuda"] = ref_cuda
        if world == 1:
            ours_api = compat_api_fps(cfg, pairs[0])
            line["compat_api"] = {"ours": ours_api, "ref_cuda": (ref_cuda or {}).get("detail", {}).get("two_threads"),
                                  "note": "pairs/s of the reference's own per-frame interface (Jetson_SLAM::ORBExtractor x2 + ORB_GPU::ORB_compute_stereo_match)"}
            line["opencv_cpu_orb"] = opencv_orb_pairs_per_s(cfg, pairs[0])
            try:
                line["adjacent"] = {"search_by_projection": sbp_microbench(), "remap_bilinear": remap_microbench()}
            except Exception as e:   # adjacent-row colour must never break the headline line
                line["adjacent"] = {"search_by_projection": {"error": repr(e)[:200]}}
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity is not None and (parity["mismatches"] or parity.get("e2e_mismatches")):
        raise SystemExit(f"bench.py: PARITY FAILED {parity}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--pairs", type=int, default=160, help="stereo pairs per step per GPU")
    ap.add_argument("--distinct", type=int, default=16, help="distinct synthetic pairs cycled over the batch")
    ap.add_argument("--chunk", type=int, default=32, help="pairs per pipeline chunk of the end-to-end call")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="N>1: skip the gather measurements")
    ap.add_argument("--gather-transport", default="p2p", choices=["p2p", "nccl"], help="peer-memory stores over NVLink (CUDA IPC) or NCCL send/recv")
    ap.add_argument("--host-cached", action="store_true", help="input images in ordinary (cached) pinned memory instead of write-combined")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity check against goldens and oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed step computed in its last run (rank 0's pairs) to "
                    "DIR/<name>.npy as float32 / float64, at most 64 MB; the inputs are seeded, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's results; the reference arm keeps none")
    from jetson_slam_b200.configs import CONFIGS
    cfg = CONFIGS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
