#!/usr/bin/env python
"""bench.py — headline benchmark of the pairwise SIFT-128 matching hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 2|3|4|5]     # this repo's CUDA path, one JSON line
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU (NCCL)
  python bench.py --gpus N --engine single ...                                   # ONE process, C++ multi-GPU engine
  python bench.py --impl reference [--steps K] [--warmup W]                      # the reference's CPU engine
  python bench.py ... --dump-outputs DIR                                         # + the last timed step's match lists as DIR/*.npy

Metric (BASELINE.json): image-pairs/sec on SIFT-128 descriptor sets; a *step* is one pass of the hot path — 2-NN + ratio
(0.85 "all" / 0.6 "good", fine_matching_graph.cc:42-43) + mutual cross-check — over the whole candidate pair list.
Workloads (BASELINE.json configs; synthetic descriptors generated on the GPU, metricsfm_b200/synth_gpu.py):
  2 (default)  100 web images x 8192 per GPU, exhaustive pairs (4,950 per GPU).  With N GPUs ONE collection of 100*N images
               is matched: the images are staged in contiguous blocks (one per GPU) but paired exhaustively within the N
               interleaved classes id mod N, so every shard reads rows that arrived over NCCL.  Weak scaling.
  3            aerial block, 1,000 x 20,000, GPS-neighbour guided pair list (~30k pairs).      Strong scaling.
  4            web collection, 5,000 x 16,384, ~200k retrieval-candidate pairs.                Strong scaling.
  5            aerial survey, 10,000 x 32,768, ~500k guided pairs (41.9 GB table per replica). Strong scaling.
Numbers in the line:
  value   pairs/s with the packed table resident in HBM (CUDA events on the library's stream, L2 flushed between steps,
          max over ranks)
  e2e     pairs/s through the public API from page-locked HOST rows: per step every image is packed + uploaded (H2D, in
          groups on the upload stream), replicated over NCCL when N > 1, matched as soon as its group has landed, and the
          match lists are copied back (D2H).  The host rows are float32 (the reference's CV_32FC1 container) for
          workload 2, uint8 otherwise (--e2e-dtype).
  parity  after the timed regions rank 0 re-generates the images of sampled pairs (also pairs matched on other ranks, also
          images this rank received over NCCL), runs the CPU oracle on them and compares the match lists bit for bit
  roofline / cpu_baseline: see DESIGN.md §6
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RATIO_ALL, RATIO_GOOD = 0.85, 0.6
INT8_SPEC_PEAK_TOPS = 4500.0

WORKLOADS = {
    2: dict(label="exhaustive matching of {ipg} web images x {rows} SIFT-128 descriptors ({ppg} pairs) per GPU (BASELINE config #2)",
            images_per_gpu=100, rows=8192, scaling="weak", e2e_dtype="f32", groups=4, parity_pairs=32),
    3: dict(label="aerial block of {images} images x {rows} descriptors, GPS-neighbour guided pair list (BASELINE config #3)",
            images=1000, rows=20000, pairs="gps", k=56, scaling="strong", e2e_dtype="u8", groups=4, parity_pairs=12),
    4: dict(label="web collection of {images} images x {rows} descriptors, retrieval-candidate pair list (BASELINE config #4)",
            images=5000, rows=16384, pairs="retrieval", k=40, scaling="strong", e2e_dtype="u8", groups=4, parity_pairs=12),
    5: dict(label="aerial survey of {images} images x {rows} descriptors, GPS-neighbour guided pair list (BASELINE config #5)",
            images=10000, rows=32768, pairs="gps", k=93, scaling="strong", e2e_dtype="u8", groups=8, parity_pairs=6),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--engine", default="auto", choices=["auto", "ranks", "single"],
                    help="ranks: one process per GPU (torchrun, NCCL via torch.distributed); single: one process, the C++ multi-GPU engine")
    ap.add_argument("--images", type=int, default=0, help="override: images per GPU (workload 2) / images in the collection (3-5)")
    ap.add_argument("--rows", type=int, default=0, help="override: descriptors per image")
    ap.add_argument("--pairs-k", type=int, default=0, help="override: neighbours / partners per image of the guided pair lists")
    ap.add_argument("--cpu-sample-pairs", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-dtype", default="", choices=["", "f32", "u8"])
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--groups", type=int, default=0, help="override: staging groups per step (uploads / all-gathers / sub-lists)")
    ap.add_argument("--no-e2e-prefetch", action="store_true", help="do not stage step k+1's host rows under step k's matching (no second context)")
    ap.add_argument("--parity-pairs", type=int, default=-1, help="pairs checked against the CPU oracle after the timed regions")
    ap.add_argument("--mutual", type=int, default=1, help="1 = ratio + mutual cross-check (headline), 0 = ratio only")
    ap.add_argument("--no-int8-peak", action="store_true", help="skip the cuBLAS int8 GEMM peak measurement (rank 0, N = 1)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the match lists of the last timed step as DIR/<name>.npy (rank 0's pairs; "
                         "see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the lists of the native path; the reference arm keeps none")
    return args


DUMP_BYTES = 64 << 20   # all files written by --dump-outputs together


def dump_outputs(out_dir: str, pairs: np.ndarray, res) -> None:
    """--dump-outputs: the match lists a caller of the timed call receives, as DIR/<name>.npy, so that two builds can be
    compared output for output.  Indices and flags are float32 (exact: all below 2^24), offsets float64:
      pairs [k, 2]     (ref, query) image ids of the written pairs, ascending (independent of the staging order and engine)
      ok [k]           1 = matched, 0 = gated (fewer than 20 keypoints)
      offsets [k + 1]  pair p's matches are matches[offsets[p]:offsets[p + 1]]
      matches [n, 2]   (ref row, query row) of every match
      good [n]         1 = the match also passes the 'good' ratio
    Every pair when the files fit in DUMP_BYTES; otherwise a fixed sample of whole pairs: the longest prefix that fits of a
    permutation of the ascending list drawn with seed 0, written in ascending order."""
    pairs = np.asarray(pairs)
    n = len(pairs)
    offs = np.asarray(res.offsets[:n + 1], np.int64)
    counts = np.diff(offs)
    per_pair = 8 + 4 + 8 + counts * (8 + (4 if res.good is not None else 0))
    budget = DUMP_BYTES - 5 * 128                       # one .npy header per file
    keep = np.lexsort((pairs[:, 1], pairs[:, 0]))
    if per_pair.sum() > budget:
        perm = np.random.default_rng(0).permutation(n)
        keep = keep[np.sort(perm[:int(np.searchsorted(np.cumsum(per_pair[keep[perm]]), budget, side="right"))])]
    new_offs = np.concatenate([[0], np.cumsum(counts[keep])]).astype(np.int64)
    rows = np.repeat(offs[keep] - new_offs[:-1], counts[keep]) + np.arange(new_offs[-1])
    arrays = {"pairs": pairs[keep].astype(np.float32), "ok": np.asarray(res.ok[:n])[keep].astype(np.float32),
              "offsets": new_offs.astype(np.float64), "matches": np.asarray(res.matches)[rows].astype(np.float32)}
    if res.good is not None:
        arrays["good"] = np.asarray(res.good)[rows].astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print(f"[bench] --dump-outputs: match lists of {len(keep)} of {n} pairs ({int(new_offs[-1])} matches) written to {out_dir}",
          file=sys.stderr, flush=True)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def ncu_traffic(workload: int, rows: int, images_per_gpu: int, world: int):
    """DRAM bytes per launch of the matching kernel from the committed `ncu --set full` capture of THIS configuration
    (profiles/r2_match_kernel_traffic.json), or None: the figure is never extrapolated to another table size."""
    path = os.path.join(ROOT, "profiles", "r2_match_kernel_traffic.json")
    if not os.path.exists(path):
        return None, "no capture committed"
    with open(path) as f:
        t = json.load(f)
    for c in t.get("captures", []):
        if c.get("workload") == workload and c.get("rows") == rows and c.get("images_per_gpu") == images_per_gpu and c.get("n_gpus", 1) == world:
            return c["dram_bytes_per_launch"], c.get("source", "profiles/r2_match_kernel_traffic.json")
    return None, "no ncu capture of this configuration"


def measure_int8_peak(dev):
    """Dense int8 tensor-core rate of this GPU as cuBLAS delivers it (torch._int_mm, 8192^3, int32 accumulate), with the
    protocol of MEASURED_PEAKS.json: best of 10 (burst) and back to back for ~2 s (sustained).  TOP/s or None."""
    import torch
    try:
        n = 8192
        a = torch.randint(-8, 8, (n, n), dtype=torch.int8, device=dev)
        b = torch.randint(-8, 8, (n, n), dtype=torch.int8, device=dev)
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = max(10, int(2000.0 / best))
        e0.record()
        for _ in range(iters):
            torch._int_mm(a, b)
        e1.record(); e1.synchronize()
        ops = 2.0 * n ** 3
        return {"burst_tops": ops / (best * 1e-3) / 1e12, "sustained_tops": ops * iters / (e0.elapsed_time(e1) * 1e-3) / 1e12,
                "how": "torch._int_mm 8192^3 (cuBLASLt int8, s32 accumulate): best of 10 and back to back for ~2 s"}
    except Exception as exc:  # noqa: BLE001
        return {"error": str(exc)[:200]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, enabled: bool = True):
        self.index, self.lines, self.proc, self.enabled = index, [], None, enabled
        self.t0 = self.t1 = None   # timed window (perf_counter)

    def _start_nvml(self) -> bool:
        """Preferred sampler: NVML polled every 5 ms from a thread (a 0.2 s timed region then holds ~40 samples instead of the
        1-2 that nvidia-smi's 100 ms loop gives).  Same quantities as the nvidia-smi query below."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            get_reasons(h)
        except Exception:
            return False
        bits = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
        self.nvml_stop = threading.Event()

        def poll():
            while not self.nvml_stop.is_set():
                try:
                    sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                    pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                    r = int(get_reasons(h))
                    flags = ",".join("Active" if r & b else "Not Active" for _, b in bits)
                    self.lines.append((time.perf_counter(), f"{self.index},{sm},{mx},{pw},{r},{flags}"))
                except Exception:
                    pass
                time.sleep(0.005)

        self.thread = threading.Thread(target=poll, daemon=True)
        self.thread.start()
        self.proc = "nvml"
        return True

    def start(self):
        if not self.enabled:
            return
        if self._start_nvml():
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self) -> dict:
        if not self.enabled:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["sampled on rank 0 only"]}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.proc == "nvml":
            self.nvml_stop.set()
            self.thread.join(timeout=2)
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        # samples inside the timed window; nvidia-smi needs ~1 s to come up, so it is started before the warm-up steps and
        # a window shorter than its period falls back to the warm-up + timed span (same kernels, same load)
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else float("inf")
        inside = [ln for t, ln in self.lines if t0 <= t <= t1 + 0.1]
        window = "timed region"
        if not inside:
            inside, window = [ln for t, ln in self.lines if t <= t1 + 0.1], "warm-up + timed region (timed region shorter than the sampling period)"
        sm, mx, pw, reasons = [], [], [], set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)), "samples": len(sm),
                "window": window, "reasons": sorted(reasons), "sampler": "NVML, 5 ms" if self.proc == "nvml" else "nvidia-smi -lms 100"}


# ====================================================================================================== reference arm
def cpu_reference_sample(images, pairs, n_pairs: int):
    """Time the reference's vendored exact engine (nanoflann; oracle/_ref) — or the oracle port when it is absent —
    on the first n_pairs pairs of the workload, all host threads.  Returns (pairs_per_s, kind, cores, seconds)."""
    from oracle import oracle
    oracle.use_all_host_threads()   # torchrun exports OMP_NUM_THREADS=1; the reference uses every core (OpenMP default)
    use_ref = oracle.ref_available()
    cores = oracle.ref_lib().ref_nanoflann_max_threads() if use_ref else oracle.max_threads()
    f32 = {}
    t0 = time.perf_counter()
    for r, q in pairs[:n_pairs]:
        if use_ref:
            for i in (r, q):
                if i not in f32:
                    f32[i] = images[i].astype(np.float32)   # the reference's container: CV_32FC1 rows
            # tree on idx1, query idx2 rows, ratio test (feature_matching.cpp:319-342; fine_matching_graph.cc:72-133)
            oracle.ref_match(f32[r], f32[q], RATIO_ALL, 20)
        else:
            oracle.match_pair_u8(images[r], images[q], RATIO_ALL, mutual=True, ratio_good=RATIO_GOOD)
    dt = time.perf_counter() - t0
    return n_pairs / dt, ("reference" if use_ref else "port"), cores, dt


def flann_forest_sample(images, pairs, n_pairs: int):
    """Behavioural twin of the reference's PRODUCTION kNN (fine_matching_graph.cc:72-99: FLANN randomized KD forest, 8 trees,
    64 checks, k = 2) through the cv2.flann_Index build of this image: seconds per pair for index build (once per idx1 in
    the reference) and for the batch query of one partner.  The reference runs one such query per OpenMP thread
    (fine_matching_graph.cc:87).  None when cv2 is unavailable."""
    try:
        import cv2
    except Exception:  # noqa: BLE001
        return None
    build_s = query_s = 0.0
    for r, q in pairs[:n_pairs]:
        ref = np.ascontiguousarray(images[r], dtype=np.float32)
        qry = np.ascontiguousarray(images[q], dtype=np.float32)
        t0 = time.perf_counter()
        index = cv2.flann_Index(ref, dict(algorithm=1, trees=8))
        t1 = time.perf_counter()
        index.knnSearch(qry, 2, params=dict(checks=64))
        t2 = time.perf_counter()
        build_s += t1 - t0
        query_s += t2 - t1
    n = max(1, min(n_pairs, len(pairs)))
    return {"kd_forest_build_s_per_image": build_s / n, "kd_forest_query_s_per_pair": query_s / n,
            "what": "one cv2.flann_Index(KDTREE, trees=8) build + one knnSearch(k=2, checks=64) call per pair (approximate search; the "
                    "production path of fine_matching_graph.cc:72-99 runs one such query per OpenMP thread)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from metricsfm_b200 import synth
    rows = args.rows or WORKLOADS[args.workload]["rows"]
    col = synth.Collection(rows, seed=0)
    per_step = 2
    n_img = min(100, 2 * per_step * (args.steps + args.warmup))
    images = {i: col.image_u8(i) for i in range(n_img)}
    pairs = synth.exhaustive_pairs(n_img)
    vals = []
    kind, cores = "port", 1
    k = 0
    for s in range(args.warmup + args.steps):
        sel = [tuple(pairs[(k + j) % len(pairs)]) for j in range(per_step)]
        k += per_step
        v, kind, cores, dt = cpu_reference_sample(images, sel, per_step)
        if s >= args.warmup:
            vals.append((per_step, dt))
    total_pairs = sum(p for p, _ in vals)
    total_s = sum(d for _, d in vals)
    value = total_pairs / total_s
    line = {
        "impl": "reference", "metric": f"image-pairs/sec ({rows} x {rows} SIFT-128)", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_s / max(args.steps, 1), "higher_is_better": True,
        "scaling": WORKLOADS[args.workload]["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE config #{args.workload} ({rows}-row SIFT-128 images), bounded sample of {per_step} pairs per step"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind,
                         "sample": f"{per_step} pairs of {rows}x{rows} per step x {args.steps} steps: nanoflann exact KD-tree "
                                   f"on idx1 + 2-NN of idx2 rows + ratio {RATIO_ALL} (feature_matching.cpp:319-342), OpenMP over queries"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)


# ====================================================================================================== workloads
def e2e_prefetch_enabled(args) -> bool:
    """Two alternating contexts in the end-to-end measurement (step k+1's host rows staged under step k's matching).  On for
    the headline workload; configs #3-#5 stage once per 0.16-7 s step, where it changes nothing and doubles the table."""
    return (not args.no_e2e) and (not args.no_e2e_prefetch) and args.workload == 2


def build_workload(args, world: int):
    """Global description of the workload: image count, rows, candidate pair list (identical on every rank)."""
    from metricsfm_b200 import synth
    w = dict(WORKLOADS[args.workload])
    rows = args.rows or w["rows"]
    # With the next step's host rows prefetched under the current step (two contexts) the staging groups no longer hide
    # anything after the first step; one group means one upload batch, one all-gather and ONE matching call per step.
    # Short e2e runs (configs #3-#5: 2-3 steps) keep the groups, which shorten the un-prefetched first step.
    prefetch_amortised = e2e_prefetch_enabled(args) and args.e2e_steps >= 8
    if args.workload == 2:
        ipg = args.images or w["images_per_gpu"]
        n_images = ipg * world
        base = synth.exhaustive_pairs(ipg).astype(np.int64)
        # one collection; class c = {ids = c mod world}: its members sit in every owner block (blocks are contiguous id ranges)
        pairs = np.concatenate([base * world + c for c in range(world)], axis=0).astype(np.int32)
        order = np.lexsort((pairs[:, 1], pairs[:, 0]))   # grouped by reference image, like the reference's idx1 loop
        pairs = pairs[order]
        label = w["label"].format(ipg=ipg, rows=rows, ppg=len(base))
    else:
        n_images = args.images or w["images"]
        k = args.pairs_k or w["k"]
        pairs = synth.gps_neighbour_pairs(n_images, k=k) if w["pairs"] == "gps" else synth.retrieval_pairs(n_images, partners=k)
        label = w["label"].format(images=n_images, rows=rows) + f", {len(pairs)} pairs"
    return dict(n_images=n_images, rows=rows, pairs=np.ascontiguousarray(pairs, np.int32), label=label, scaling=w["scaling"],
                e2e_dtype=args.e2e_dtype or w["e2e_dtype"], groups=args.groups or (1 if prefetch_amortised else w["groups"]),
                parity_pairs=w["parity_pairs"] if args.parity_pairs < 0 else args.parity_pairs)


def group_layout(n_images: int, world: int, n_groups: int):
    """Staging layout.  Owner blocks are contiguous id ranges (msfm_sched_image_owner); every block is cut into n_groups
    slices and the table is laid out group-major — [group 0: slice of rank 0, slice of rank 1, ...][group 1: ...] — so
    that one group is one contiguous arena range made of `world` equal parts: one in-place all-gather replicates it, and
    the pairs of groups <= g can be matched while group g + 1 is still being copied.
    Returns (owner[n_images], group[n_images], slices[g][r] = list of ids)."""
    from metricsfm_b200 import scheduler
    owner = scheduler.image_owner(n_images, world)
    group = np.zeros((n_images,), np.int32)
    slices = [[[] for _ in range(world)] for _ in range(n_groups)]
    for r in range(world):
        ids = np.nonzero(owner == r)[0]
        per = (len(ids) + n_groups - 1) // n_groups
        for k, i in enumerate(ids):
            g = min(k // max(per, 1), n_groups - 1)
            group[i] = g
            slices[g][r].append(int(i))
    return owner, group, slices


def parity_check(sampled, regenerate, mutual: bool):
    """sampled: list of (ref id, query id, matches [n,2], good [n]) — the lists the GPU path produced.  Re-generates the
    images and compares with the CPU oracle bit for bit.  Returns (checked, ok, first failure or None)."""
    from oracle import oracle
    oracle.use_all_host_threads()
    cache, bad = {}, None
    for r, q, m, g in sampled:
        for i in (r, q):
            if i not in cache:
                cache[i] = regenerate(i)
        exp = oracle.match_pair_u8(cache[r], cache[q], RATIO_ALL, mutual=mutual, ratio_good=RATIO_GOOD)
        if not (np.array_equal(np.asarray(m).reshape(-1, 2), exp["pairs"]) and np.array_equal(np.asarray(g), exp["good"])):
            bad = bad or (int(r), int(q))
    return len(sampled), bad is None, bad


# ====================================================================================================== native arm: ranks
def run_native_ranks(args):
    import torch
    import torch.distributed as dist
    from metricsfm_b200 import distributed as D, scheduler
    from metricsfm_b200.matcher import Matcher, MatchResult
    from metricsfm_b200.synth_gpu import GpuCollection

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = {"pinned": False, "why": "single process: the CPU baseline keeps every host core"}
    if world > 1:
        numa = D.pin_to_gpu_numa_node(local_rank)   # before the page-locked staging buffers are allocated
        dist.init_process_group("nccl", device_id=dev)

    wl = build_workload(args, world)
    n_images, rows, pairs = wl["n_images"], wl["rows"], wl["pairs"]
    rows_padded = (rows + 255) // 256 * 256
    arena_rows = n_images * rows_padded
    owner, group, slices = group_layout(n_images, world, wl["groups"])
    n_groups = wl["groups"]
    my_ids = [i for g in range(n_groups) for i in slices[g][rank]]
    slot_of = {gid: k for k, gid in enumerate(my_ids)}

    # ---- synthetic descriptors: generated on the GPU, kept in page-locked host memory (the e2e step starts from there)
    col = GpuCollection(rows, dev, seed=0)
    host_u8 = torch.empty((len(my_ids), rows, 128), dtype=torch.uint8).pin_memory()
    for k, gid in enumerate(my_ids):
        host_u8[k].copy_(col.image_u8(gid))
    e2e_f32 = wl["e2e_dtype"] == "f32" and not args.no_e2e
    host_f32 = None
    if e2e_f32:
        host_f32 = torch.empty((len(my_ids), rows, 128), dtype=torch.float32).pin_memory()   # CV_32FC1 rows (integer-valued: VLSIFT + rounding)
        host_f32.copy_(host_u8)

    # ---- pair list: ONE list for the whole job, sharded by cost (C++ scheduler, msfm_sched_shard).  The pairs are taken in
    #      the order their images land (staging group of the newer image) and every group's sub-list is sharded on its
    #      own, so that all ranks finish a sub-list together: the all-gather of the next group is a rendezvous of the ranks.
    rows_per_image = np.full((n_images,), rows, np.int32)
    pg_all = np.maximum(group[pairs[:, 0]], group[pairs[:, 1]])
    my_parts, pg_parts = [], []
    for g in range(n_groups):
        idx_g = np.nonzero(pg_all == g)[0]
        if len(idx_g) == 0:
            continue
        mine = idx_g[scheduler.shard_pairs(pairs[idx_g], rows_per_image, world)[rank]]
        my_parts.append(mine)
        pg_parts.append(np.full((len(mine),), g, np.int64))
    my_idx = np.concatenate(my_parts) if my_parts else np.zeros((0,), np.int64)
    pg = np.concatenate(pg_parts) if pg_parts else np.zeros((0,), np.int64)
    my_pairs = np.ascontiguousarray(pairs[my_idx])
    sub_bounds = [int(np.searchsorted(pg, g, side="left")) for g in range(n_groups)] + [len(my_idx)]
    foreign_reads = int(np.sum(owner[my_pairs[:, 0]] != rank) + np.sum(owner[my_pairs[:, 1]] != rank))

    # ---- packed table in torch-owned memory so NCCL can fill it during replication
    desc_arena = torch.empty((arena_rows, 128), dtype=torch.uint8, device=dev)
    norm_arena = torch.empty((arena_rows,), dtype=torch.int32, device=dev)
    m = Matcher(device=local_rank, max_images=n_images, arena_rows=arena_rows, external_desc_arena=desc_arena.data_ptr(),
                external_norm_arena=norm_arena.data_ptr())
    lib_stream = torch.cuda.ExternalStream(m.cuda_stream(), device=dev)
    up_stream = torch.cuda.ExternalStream(m.upload_stream(), device=dev)
    # what staging / replication need to know about a context: (matcher, its main stream, its upload stream, its arenas)
    cx_main = (m, lib_stream, up_stream, desc_arena, norm_arena)

    def stage_table(use_f32: bool, cx=cx_main):
        """Queue the staging of the whole table, group by group: H2D + pack of this rank's slice on the library's upload
        streams, the other ranks' slices reserved.  Nothing waits on the host.  Returns, per group, what replicate_group()
        needs (the event after the group's uploads and its arena range), and the H2D bytes."""
        m, _, up_stream = cx[:3]
        m.release_all()
        groups_meta, h2d = [], 0
        base_row = 0
        for g in range(n_groups):
            for r in range(world):        # identical allocation order on every rank => identical arena offsets
                ids = slices[g][r]
                if not ids:
                    continue
                if r == rank:
                    if use_f32:
                        m.upload_f32_batch_async(ids, [host_f32[slot_of[i]] for i in ids], scale=1.0)
                        h2d += len(ids) * rows * 512
                    else:
                        m.upload_batch(ids, [host_u8[slot_of[i]] for i in ids], wait=False)
                        h2d += len(ids) * rows * 128
                else:
                    m.reserve_batch(ids, [rows] * len(ids), wait=False)
            n_rows_g = sum(len(slices[g][r]) for r in range(world)) * rows_padded
            ev_up = None
            if world > 1:
                ev_up = torch.cuda.Event()
                ev_up.record(up_stream)
            groups_meta.append((ev_up, base_row, n_rows_g))
            base_row += n_rows_g
        return groups_meta, h2d

    def replicate_group(g: int, meta, cx=cx_main):
        """One in-place all-gather of group g (descriptor rows + side words) over NCCL, queued on the library's MAIN stream:
        it runs between two matching launches, never next to one — the matching kernel is persistent (one CTA per SM,
        statically partitioned work), and a collective kernel that sits on a few SMs waiting for a peer that is still
        matching would stall the CTAs that cannot be placed.  The next matching launch is ordered behind it by the stream."""
        if world == 1:
            return
        _, lib_stream, _, desc_arena, norm_arena = cx
        ev_up, base_row, n_rows_g = meta
        part = max(len(slices[g][r]) for r in range(world)) * rows_padded
        equal = all(len(slices[g][r]) * rows_padded == part for r in range(world))
        with torch.cuda.stream(lib_stream):
            lib_stream.wait_event(ev_up)
            lo = base_row + sum(len(slices[g][r]) for r in range(rank)) * rows_padded
            hi = lo + len(slices[g][rank]) * rows_padded
            if equal:
                dist.all_gather_into_tensor(desc_arena[base_row:base_row + n_rows_g], desc_arena[lo:hi])
                dist.all_gather_into_tensor(norm_arena[base_row:base_row + n_rows_g], norm_arena[lo:hi])
            else:                  # ragged slices: one broadcast per owner
                off = base_row
                for r in range(world):
                    nr = len(slices[g][r]) * rows_padded
                    if nr:
                        dist.broadcast(desc_arena[off:off + nr], src=r)
                        dist.broadcast(norm_arena[off:off + nr], src=r)
                    off += nr

    kw = dict(ratio_good=RATIO_GOOD, mutual=bool(args.mutual), min_keypoints=20, orientation=0)
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value"): table staged once, untimed
    metas, _ = stage_table(False)
    for g, meta in enumerate(metas):
        replicate_group(g, meta)
    m.sync()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank, enabled=(rank == 0))
    sampler.start()
    for _ in range(args.warmup):
        m.match_pairs_resident(my_pairs, RATIO_ALL, **kw)
    barrier()
    sampler.mark_begin()
    step_ms, kern_ms, launches, match_launches, ops, twin_pairs = [], [], 0, 0, 0, 0
    n_matches = 0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        with torch.cuda.stream(lib_stream):
            flush.zero_()                       # L2 flush between timed iterations (not timed)
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(lib_stream)
        n_matches = m.match_pairs_resident(my_pairs, RATIO_ALL, **kw)
        e1.record(lib_stream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        t = m.timing()
        kern_ms.append(t["match_kernel_ms"])
        launches += t["total_launches"]
        match_launches += t["match_launches"]
        ops = t["int8_ops"]
        twin_pairs = t["twin_pairs"]
    barrier()
    sampler.mark_end()
    wall_s = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    total_ms = float(sum(step_ms))
    if world > 1:
        tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt.item())
    pairs_done = float(len(pairs) * args.steps)   # all ranks together match the whole list once per step
    value = pairs_done / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # the resident call leaves its lists in HBM and returns only their count: the same call on the same table through
        # msfm_match_pairs copies them to the host, and must find exactly as many
        res = m.match_pairs(my_pairs, RATIO_ALL, capacity=n_matches, **kw)
        if len(res.matches) != n_matches:
            raise RuntimeError(f"msfm_match_pairs found {len(res.matches)} matches, the timed resident call {n_matches}")
        dump_outputs(args.dump_outputs, my_pairs, res)

    # ---- end to end through the public API from host buffers, staging pipelined against matching
    e2e, sampled_local = None, []
    cap = int(min(len(my_pairs) * min(rows, 4096), 1 << 29)) + 1024
    out = MatchResult(offsets=np.zeros((len(my_pairs) + n_groups + 1,), np.int64), ok=np.zeros((len(my_pairs) + 1,), np.int32),
                      matches=torch.empty((cap, 2), dtype=torch.int32).pin_memory().numpy(),
                      good=torch.empty((cap,), dtype=torch.uint8).pin_memory().numpy())
    list_off = np.zeros((len(my_pairs) + 1,), np.int64)   # absolute offsets of this rank's lists in `out`

    trace = os.environ.get("BENCH_TRACE") is not None

    # Two contexts (two copies of the table in HBM) alternate, so that the NEXT step's rows are copied from the host and
    # packed (upload stream / copy engine of the other context) while the current step is matched.  Every step's
    # host->device copy and its device->host read of the match lists still happen inside the timed region; only their
    # overlap changes.  With N > 1 the all-gathers of a step stay where they were — on the main stream of the step's own
    # context, between its matching launches — but they no longer wait for the host copies of any rank.
    cx_alt = None
    if e2e_prefetch_enabled(args):
        d2, n2 = torch.empty((arena_rows, 128), dtype=torch.uint8, device=dev), torch.empty((arena_rows,), dtype=torch.int32, device=dev)
        m2 = Matcher(device=local_rank, max_images=n_images, arena_rows=arena_rows, external_desc_arena=d2.data_ptr(), external_norm_arena=n2.data_ptr())
        cx_alt = (m2, torch.cuda.ExternalStream(m2.cuda_stream(), device=dev), torch.cuda.ExternalStream(m2.upload_stream(), device=dev), d2, n2)
    m_alt = cx_alt[0] if cx_alt else None
    staged = {}   # matcher -> (metas, h2d) of a table already queued for it by the previous step

    def e2e_step(use_f32: bool, step: int = 0, last: bool = True):
        t_begin = time.perf_counter()
        cx = cx_main if (cx_alt is None or step % 2 == 0) else cx_alt
        cur = cx[0]
        metas, h2d = staged.pop(cur, None) or stage_table(use_f32, cx)
        stager = None
        if cx_alt is not None and not last:
            # the next step's staging is queued by a helper thread while this thread sits in the (GIL-free) matching call:
            # the ~1 ms of host work it takes would otherwise leave the GPU idle between two steps
            nxt = cx_alt if cx is cx_main else cx_main
            box = {}

            def stage_next():
                try:
                    torch.cuda.set_device(dev)
                    box["staged"] = stage_table(use_f32, nxt)
                except BaseException as exc:                 # noqa: BLE001  (re-raised by the joining thread)
                    box["error"] = exc

            stager = threading.Thread(target=stage_next)
            stager.start()

        def join_stager():
            if stager is not None:
                stager.join()
                if "error" in box:
                    raise box["error"]
                staged[nxt[0]] = box["staged"]

        stamps = [time.perf_counter() - t_begin]
        done, d2h = 0, 0
        if world == 1:
            # ONE call over the whole list (ordered by staging group): the library cuts its batches where the next pair's
            # images have not landed yet, so matching starts on group 0 while the later groups are still being copied
            sub = MatchResult(offsets=out.offsets[:len(my_pairs) + 1], ok=out.ok[:len(my_pairs)], matches=out.matches, good=out.good)
            res = cur.match_pairs(my_pairs, RATIO_ALL, out=sub, **kw)
            list_off[:] = sub.offsets[:len(my_pairs) + 1]
            join_stager()
            stamps.append(time.perf_counter() - t_begin)
            if trace:
                print(f"[trace rank {rank}] f32={use_f32} staging enqueued at {1e3 * stamps[0]:.2f} ms, done at {1e3 * stamps[1]:.2f} ms, "
                      f"{cur.timing()['match_launches']} matching launches", file=sys.stderr, flush=True)
            return h2d + my_pairs.nbytes, cur.timing()["d2h_bytes"], len(res.matches)
        for g in range(n_groups):
            a, b = sub_bounds[g], sub_bounds[g + 1]
            replicate_group(g, metas[g], cx)             # queued on the main stream: runs before sub-list g's launches
            if b == a:
                continue
            sub = MatchResult(offsets=out.offsets[a + g:b + g + 1], ok=out.ok[a:b], matches=out.matches[done:], good=out.good[done:])
            res = cur.match_pairs(my_pairs[a:b], RATIO_ALL, out=sub, **kw)
            list_off[a:b + 1] = done + sub.offsets[:b - a + 1]
            done += len(res.matches)
            d2h += cur.timing()["d2h_bytes"]
            stamps.append(time.perf_counter() - t_begin)
        join_stager()
        if trace:
            print(f"[trace rank {rank}] f32={use_f32} staging enqueued at {1e3 * stamps[0]:.2f} ms, sub-lists done at "
                  + ", ".join(f"{1e3 * t:.2f}" for t in stamps[1:]) + " ms", file=sys.stderr, flush=True)
        return h2d + my_pairs.nbytes, d2h, done

    if not args.no_e2e:
        e2e_steps = max(1, args.e2e_steps)
        e2e_step(e2e_f32, 0, m_alt is None)                 # warm-up (allocations, NCCL channels) ...
        if m_alt is not None:
            e2e_step(e2e_f32, 1, True)                      # ... of both contexts
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            h2d, d2h, n_e2e = e2e_step(e2e_f32, k, k == e2e_steps - 1)
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        e2e = {"value": (len(pairs) * e2e_steps) / dt, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "steps": e2e_steps, "host_rows": "float32 (CV_32FC1, the reference's container)" if e2e_f32 else "uint8",
               "pipeline": f"{n_groups} staging groups on the upload streams" + (" + one NCCL all-gather per group between matching launches; one "
                                                                                      "msfm_match_pairs call per group" if world > 1 else
                                                                                      "; ONE msfm_match_pairs call, batches cut where uploads have not landed")
                           + "; the pairs of groups <= g are matched while group g+1 is copied"
                           + ("; two contexts alternate: step k+1's host rows are copied + packed while step k is matched" if m_alt is not None else ""),
               "timer": "host wall clock between barriers + cuda synchronize, max over ranks", "matches_per_step_this_rank": int(n_e2e),
               "match_lists": "page-locked host buffers of the rank that matched the pair"}
        if e2e_f32:                                         # the same pipeline fed with pre-quantised uint8 rows, for comparison
            e2e_step(False, 0, m_alt is None)
            if m_alt is not None:
                e2e_step(False, 1, True)
            barrier()
            t0 = time.perf_counter()
            for k in range(e2e_steps):
                h2d_u8, _, _ = e2e_step(False, k, k == e2e_steps - 1)
            barrier()
            dt8 = time.perf_counter() - t0
            if world > 1:
                tt = torch.tensor([dt8], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt8 = float(tt.item())
            e2e["uint8_rows"] = {"value": (len(pairs) * e2e_steps) / dt8, "h2d_bytes_per_step": int(h2d_u8)}
    else:
        e2e_step(False)                                     # the parity check below needs lists in host memory

    # ---- parity inside the run: sampled pairs of EVERY rank's shard against the CPU oracle (rank 0 re-generates the images)
    n_par = wl["parity_pairs"]
    per_rank = (n_par + world - 1) // world if n_par > 0 else 0
    rng = np.random.default_rng(1234 + rank)
    if per_rank and len(my_pairs):
        # prefer pairs that read rows received over NCCL
        cand = np.nonzero((owner[my_pairs[:, 0]] != rank) | (owner[my_pairs[:, 1]] != rank))[0] if world > 1 else np.arange(len(my_pairs))
        if len(cand) == 0:
            cand = np.arange(len(my_pairs))
        for k in rng.choice(cand, size=min(per_rank, len(cand)), replace=False):
            a, b = int(list_off[k]), int(list_off[k + 1])
            sampled_local.append((int(my_pairs[k, 0]), int(my_pairs[k, 1]), out.matches[a:b].copy(), out.good[a:b].copy()))
    gathered = [sampled_local]
    if world > 1:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(sampled_local, gathered, dst=0)
    parity = None
    if rank == 0 and n_par > 0:
        sampled = [s for part in gathered for s in part][:max(n_par, 1)]
        regen = lambda i: col.image_u8(i).cpu().numpy()     # noqa: E731  (deterministic in the image id)
        checked, ok, bad = parity_check(sampled, regen, bool(args.mutual))
        # rows this rank received over NCCL equal the re-generated bytes
        nccl_ok, nccl_checked = True, 0
        for i in [i for i in range(n_images) if owner[i] != rank][:: max(1, n_images // 16)][:8]:
            got, _ = m.download_packed(i)
            nccl_ok = nccl_ok and np.array_equal(got, regen(i))
            nccl_checked += 1
        parity = {"parity_checked": checked, "parity_ok": bool(ok and nccl_ok), "first_mismatch": bad,
                  "nccl_received_images_checked": nccl_checked, "nccl_received_images_ok": bool(nccl_ok),
                  "how": "match lists of sampled pairs from every rank's shard (pairs reading NCCL-received rows first) == CPU oracle "
                         "on the re-generated images, bit for bit"}

    # ---- CPU baseline (rank 0, N = 1 only): the reference's exact engine on a bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        need = sorted({int(i) for p in pairs[: args.cpu_sample_pairs] for i in p})
        images = {i: host_u8[slot_of[i]].numpy() for i in need}
        sel = [tuple(int(x) for x in p) for p in pairs[: args.cpu_sample_pairs]]
        v, kind, cores, secs = cpu_reference_sample(images, sel, len(sel))
        cpu = {"value": v, "unit": "pairs/s", "cores": cores, "kind": kind,
               "sample": f"first {len(sel)} pairs of the workload ({rows}x{rows}), {secs:.1f} s: nanoflann exact KD-tree on idx1 + 2-NN of "
                         f"idx2 rows + ratio {RATIO_ALL}, OpenMP over queries (reference engine compiled from its own headers)"}
        forest = flann_forest_sample(images, sel, 2)
        if forest is not None:
            forest["extrapolated_pairs_per_s_one_query_per_core"] = cores / forest["kd_forest_query_s_per_pair"]
            cpu["production_kd_forest"] = forest

    if m_alt is not None:
        m_alt.close()
        m_alt, cx_alt = None, None
    int8_peak = None
    if rank == 0 and world == 1 and not args.no_int8_peak:
        m.close()                      # the library's scratch is not needed any more
        del desc_arena, norm_arena
        int8_peak = measure_int8_peak(dev)
    if rank == 0:
        kern_avg_ms = float(np.mean(kern_ms))
        emit_line(args, wl, world, value, total_ms, ops, kern_avg_ms, float(np.mean(step_ms)), clocks, launches, match_launches, wall_s,
                  e2e, cpu, int8_peak, parity, engine="ranks: one process per GPU, torch.distributed/NCCL",
                  extra_cfg={"matches_per_step_rank0": int(n_matches), "host_numa_pinning_rank0": numa,
                             "pairs_rank0": int(len(my_pairs)), "foreign_image_reads_rank0": foreign_reads,
                             "mutual_pairs_needing_tensor_twin_pass_rank0": int(twin_pairs)})
    m.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def emit_line(args, wl, world, value, total_ms, ops_rank0, kern_avg_ms, step_avg_ms, clocks, launches, match_launches, wall_s, e2e, cpu,
              int8_peak, parity, engine, extra_cfg):
    peaks, peaks_src = measured_peaks()
    achieved_tops = ops_rank0 / (kern_avg_ms * 1e-3) / 1e12 if kern_avg_ms > 0 else 0.0
    sustained = 2.0 * float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    burst = 2.0 * float(peaks.get("bf16_tflops", 1650.0))
    ipg = (args.images or WORKLOADS[2]["images_per_gpu"]) if args.workload == 2 else wl["n_images"]
    traffic, traffic_src = ncu_traffic(args.workload, wl["rows"], ipg, world)
    line = {
        "metric": f"image-pairs/sec ({wl['rows']} x {wl['rows']} SIFT-128)", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": wl["scaling"],
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": wl["label"] + f"; 2-NN + ratio {RATIO_ALL}/{RATIO_GOOD}" + (" + mutual cross-check" if args.mutual else " (no mutual check)"),
                   "pairs_per_step_all_gpus": int(len(wl["pairs"])), "images": int(wl["n_images"]),
                   "parallelism": f"ONE pair list sharded x{world} by cost (msfm_sched_shard), table replicated over NCCL", "engine": engine,
                   "l2": "flushed between timed steps (256 MiB write)", **extra_cfg},
        "roofline": {"bound": "tensor", "achieved": achieved_tops, "peak": INT8_SPEC_PEAK_TOPS, "unit": "TFLOP/s",
                     "frac": achieved_tops / INT8_SPEC_PEAK_TOPS, "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": "match_pairs_kernel<4,64,8,1,2> (4 strips x N=64 tiles, 8 B stages, 2 TMEM buffers per strip), rank 0's launches",
                     "note": "int8 tensor ops (2 per MAC), i.e. TOP/s; algorithmic ops = 2*M*N*128 per pair; peak = B200 dense int8 spec "
                             "(north_star's denominator; MEASURED_PEAKS.json has no int8 figure): the fractions of 2 x the measured bf16 "
                             "rates and of the cuBLAS int8 GEMM measured in this run are given beside it",
                     "frac_of_2x_bf16_sustained": achieved_tops / sustained, "frac_of_2x_bf16_burst": achieved_tops / burst,
                     "peaks_file": peaks_src, "kernel_ms_per_step": kern_avg_ms, "kernel_share_of_step": kern_avg_ms / step_avg_ms if step_avg_ms else None},
        "clocks": clocks,
        "gpu_launches": int(launches),
        "match_kernel_launches": int(match_launches),
        "wall_s_timed_region": wall_s,
    }
    if int8_peak is not None:
        line["roofline"]["int8_gemm_measured"] = int8_peak
        if "sustained_tops" in int8_peak:
            line["roofline"]["frac_of_measured_int8_sustained"] = achieved_tops / int8_peak["sustained_tops"]
    if parity is not None:
        line.update({"parity_checked": parity["parity_checked"], "parity_ok": parity["parity_ok"], "parity": parity})
    if e2e is not None:
        line["e2e"] = e2e
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), file=JSON_OUT, flush=True)


# ====================================================================================================== native arm: single process
def run_native_single(args):
    """ONE host process, every GPU of the box behind the C ABI of include/msfm_multi.h (no torch.distributed): staging with
    NCCL broadcast, LPT sharding, per-device matching threads and the stitched result all live in csrc/msfm_multi.cc."""
    import torch
    from metricsfm_b200.matcher import MatchResult
    from metricsfm_b200.multi import MultiMatcher
    from metricsfm_b200.synth_gpu import GpuCollection

    world = args.gpus
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        raise SystemExit(f"--engine single --gpus {world} needs {world} visible CUDA devices")
    wl = build_workload(args, world)
    n_images, rows, pairs = wl["n_images"], wl["rows"], wl["pairs"]
    rows_padded = (rows + 255) // 256 * 256
    n_groups = wl["groups"]
    # every image generated on GPU 0, kept in page-locked host memory (the single process owns all host rows)
    dev0 = torch.device("cuda", 0)
    col = GpuCollection(rows, dev0, seed=0)
    host_u8 = torch.empty((n_images, rows, 128), dtype=torch.uint8).pin_memory()
    for i in range(n_images):
        host_u8[i].copy_(col.image_u8(i))
    e2e_f32 = wl["e2e_dtype"] == "f32" and not args.no_e2e
    host_f32 = None
    if e2e_f32:
        host_f32 = torch.empty((n_images, rows, 128), dtype=torch.float32).pin_memory()
        host_f32.copy_(host_u8)
    per = (n_images + n_groups - 1) // n_groups
    groups = [list(range(g * per, min(n_images, (g + 1) * per))) for g in range(n_groups)]
    group_of = np.minimum(np.arange(n_images) // per, n_groups - 1)
    pg = np.maximum(group_of[pairs[:, 0]], group_of[pairs[:, 1]])
    order = np.argsort(pg, kind="stable")
    pairs_sorted = np.ascontiguousarray(pairs[order])
    pg = pg[order]
    bounds = [int(np.searchsorted(pg, g, side="left")) for g in range(n_groups)] + [len(pairs)]

    mm = MultiMatcher(list(range(world)), max_images=n_images, arena_rows=n_images * rows_padded)
    kw = dict(ratio_good=RATIO_GOOD, mutual=bool(args.mutual), min_keypoints=20, orientation=0)
    cap = int(min(len(pairs) * min(rows, 4096), 1 << 28)) + 1024
    out = MatchResult(offsets=np.zeros((len(pairs) + n_groups + 1,), np.int64), ok=np.zeros((len(pairs) + 1,), np.int32),
                      matches=torch.empty((cap, 2), dtype=torch.int32).pin_memory().numpy(),
                      good=torch.empty((cap,), dtype=torch.uint8).pin_memory().numpy())

    def stage(use_f32):
        mm.release_all()
        h2d = 0
        for ids in groups:
            if use_f32:
                mm.upload_f32(ids, [host_f32[i] for i in ids], scale=1.0)
                h2d += len(ids) * rows * 512
            else:
                mm.upload_u8(ids, [host_u8[i] for i in ids])
                h2d += len(ids) * rows * 128
        return h2d

    # ---- device-resident: table staged once; a step = msfm_multi_match_pairs over the whole list (lists stitched on the host)
    stage(False)
    mm.sync()
    sampler = ClockSampler(0)
    sampler.start()
    full = MatchResult(offsets=np.zeros((len(pairs) + 1,), np.int64), ok=np.zeros((len(pairs),), np.int32), matches=out.matches, good=out.good)
    for _ in range(args.warmup):
        mm.match_pairs(pairs_sorted, RATIO_ALL, capacity=cap, out=full, **kw)
    sampler.mark_begin()
    dev_ms, wall_ms, kern_ms, launches, match_launches, ops0 = [], [], [], 0, 0, 0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        res = mm.match_pairs(pairs_sorted, RATIO_ALL, capacity=cap, out=full, **kw)
        t, per_dev = mm.timing()
        dev_ms.append(t["device_ms_max"])
        wall_ms.append(t["wall_ms"])
        kern_ms.append(per_dev[0]["match_kernel_ms"])
        ops0 = per_dev[0]["int8_ops"]
        launches += sum(p["total_launches"] for p in per_dev)
        match_launches += sum(p["match_launches"] for p in per_dev)
    sampler.mark_end()
    wall_s = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    total_ms = float(sum(dev_ms))
    value = len(pairs) * args.steps / (total_ms * 1e-3)
    n_matches = len(res.matches)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pairs_sorted, res)   # before the e2e steps reuse the result buffers

    list_off = np.zeros((len(pairs) + 1,), np.int64)

    def e2e_step(use_f32):
        h2d = stage(use_f32)
        done = 0
        for g in range(n_groups):
            a, b = bounds[g], bounds[g + 1]
            if b == a:
                continue
            sub = MatchResult(offsets=out.offsets[a + g:b + g + 1], ok=out.ok[a:b], matches=out.matches[done:], good=out.good[done:])
            r = mm.match_pairs(pairs_sorted[a:b], RATIO_ALL, capacity=cap, out=sub, **kw)
            list_off[a:b + 1] = done + sub.offsets[:b - a + 1]
            done += len(r.matches)
        return h2d + pairs.nbytes, done * 9, done

    e2e = None
    if not args.no_e2e:
        e2e_steps = max(1, args.e2e_steps)
        e2e_step(e2e_f32)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            h2d, d2h, n_e2e = e2e_step(e2e_f32)
        mm.sync()
        dt = time.perf_counter() - t0
        e2e = {"value": len(pairs) * e2e_steps / dt, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "steps": e2e_steps, "host_rows": "float32 (CV_32FC1, the reference's container)" if e2e_f32 else "uint8",
               "pipeline": f"{n_groups} staging groups (owner H2D + NCCL broadcast); the pairs of groups <= g are matched while group g+1 lands",
               "timer": "host wall clock of the single process", "matches_per_step": int(n_e2e),
               "match_lists": "stitched into ONE result in the caller's pair order (msfm_multi_match_pairs)"}
    else:
        e2e_step(False)

    parity = None
    n_par = wl["parity_pairs"]
    if n_par > 0:
        rng = np.random.default_rng(1234)
        sampled = []
        for k in rng.choice(len(pairs), size=min(n_par, len(pairs)), replace=False):
            a, b = int(list_off[k]), int(list_off[k + 1])
            sampled.append((int(pairs_sorted[k, 0]), int(pairs_sorted[k, 1]), out.matches[a:b].copy(), out.good[a:b].copy()))
        regen = lambda i: host_u8[i].numpy()     # noqa: E731
        checked, ok, bad = parity_check(sampled, regen, bool(args.mutual))
        nccl_ok, nccl_checked = True, 0
        for d in range(world):
            for i in (0, n_images // 2, n_images - 1):
                got, _ = mm.download_packed(d, i)
                nccl_ok = nccl_ok and np.array_equal(got, host_u8[i].numpy())
                nccl_checked += 1
        parity = {"parity_checked": checked, "parity_ok": bool(ok and nccl_ok), "first_mismatch": bad,
                  "nccl_received_images_checked": nccl_checked, "nccl_received_images_ok": bool(nccl_ok),
                  "how": "stitched match lists of sampled pairs == CPU oracle, bit for bit; every device's replica of sampled images == host rows"}
    mm.close()
    emit_line(args, wl, world, value, total_ms, ops0, float(np.mean(kern_ms)), float(np.mean(dev_ms)), clocks, launches, match_launches, wall_s,
              e2e, None, None, parity, engine="single: one host process, C++ multi-GPU engine (include/msfm_multi.h), NCCL via ncclCommInitAll",
              extra_cfg={"matches_per_step": int(n_matches), "host_wall_ms_per_step_incl_stitch": float(np.mean(wall_ms)),
                         "value_timer": "max over devices of the CUDA-event time of each device's msfm_match_pairs call"})


JSON_OUT = sys.stdout


def claim_stdout():
    """Rank 0 prints exactly ONE JSON line on stdout.  Native libraries (NCCL's version banner, ...) write to file
    descriptor 1 directly, so keep a private copy of the real stdout for the JSON line and point fd 1 at stderr."""
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
        return
    under_torchrun = int(os.environ.get("WORLD_SIZE", "1")) > 1
    engine = args.engine
    if engine == "auto":
        engine = "ranks" if (under_torchrun or args.gpus == 1) else "single"
    if engine == "single":
        if int(os.environ.get("RANK", "0")) == 0:
            run_native_single(args)
    else:
        run_native_ranks(args)


if __name__ == "__main__":
    main()
