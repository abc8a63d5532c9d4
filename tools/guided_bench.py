"""Cost of guided re-matching (msfm_match_pairs_guided) against the unconstrained matcher (msfm_match_pairs) on one GPU.

Workload: --pairs independent two-view scene pairs of --rows-row images (oracle.guided_oracle.decoy_scene: true
correspondences, a quarter of them with a planted look-alike off the epipolar line, the rest unrelated rows), every image
distinct, so that the descriptor table (2 * pairs * rows * 128 B, 420 MB at the defaults) is well above the 126 MB L2.
Ratio 0.85 with ratio_good 0.6, mutual off and on, th_epipolar 3 px with the scene's F.  The two calls alternate in one
process after a warm-up of each; per call the host wall time, msfm_last_timing's total_ms and match_kernel_ms, and the
match counts (all, and planted true correspondences) are recorded, medians reported.  A second pass runs each call once
in a child process with MSFM_DEBUG_FLAGS=8 and reads the kernel's hot-group count (groups of 8 columns scored exactly)
from the context's debug summary.  The card's name and power limit are read in the same run.

    python tools/guided_bench.py --out profiles/guided_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _scene(args):
    from oracle.guided_oracle import decoy_scene
    seed, rows = args
    return decoy_scene(seed, rows, rows, decoy_frac=0.25, dups=False)


def make_scenes(n_pairs: int, rows: int, seed: int):
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        scenes = list(ex.map(_scene, [(seed + i, rows) for i in range(n_pairs)]))
    desc = np.stack([d for s in scenes for d in (s["ref"], s["qry"])])
    xy = np.stack([x for s in scenes for x in (s["xy_ref"], s["xy_qry"])])
    F = np.stack([s["F"] for s in scenes])
    true = [np.array(sorted(s["true"]), np.int32).reshape(-1, 2) for s in scenes]
    return desc, xy, F, true


def open_matcher(desc):
    from metricsfm_b200.matcher import Matcher
    n_img, rows = desc.shape[0], desc.shape[1]
    m = Matcher(device=0, max_images=n_img, arena_rows=n_img * rows + (1 << 16))
    m.upload_batch(list(range(n_img)), list(desc))
    return m


def run_call(m, kind, pairs, F, xy_map, mutual):
    if kind == "plain":
        return m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mutual)
    return m.match_pairs_guided(pairs, F, xy_map, th_epipolar=3.0, ratio=0.85, ratio_good=0.6, mutual=mutual)


def true_accepted(res, true):
    n = 0
    for p, t in enumerate(true):
        got = res.pair(p)
        if len(got) and len(t):
            a = got[:, 0].astype(np.int64) << 32 | got[:, 1].astype(np.int64)
            b = t[:, 0].astype(np.int64) << 32 | t[:, 1].astype(np.int64)
            n += int(np.isin(a, b).sum())
    return n


def child(path: str, kind: str, mutual: bool) -> None:
    """One call with MSFM_DEBUG_FLAGS=8 set by the parent; the summary is printed to stderr when the context closes."""
    z = np.load(path)
    desc, xy, F = z["desc"], z["xy"], z["F"]
    m = open_matcher(desc)
    pairs = np.arange(desc.shape[0], dtype=np.int32).reshape(-1, 2)
    run_call(m, kind, pairs, F, {i: xy[i] for i in range(xy.shape[0])}, mutual)
    m.close()


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [x.strip() for x in line.split(",")]
    return dict(name=parts[0] if parts else None, power_limit=parts[1] if len(parts) > 1 else None,
                max_sm_clock=parts[2] if len(parts) > 2 else None)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--seed", type=int, default=1000)
    ap.add_argument("--out", default="")
    ap.add_argument("--child", nargs=3, metavar=("NPZ", "KIND", "MUTUAL"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.child[0], a.child[1], a.child[2] == "1")
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("guided_bench needs a GPU")
    t0 = time.time()
    desc, xy, F, true = make_scenes(a.pairs, a.rows, a.seed)
    gen_s = time.time() - t0
    pairs = np.arange(desc.shape[0], dtype=np.int32).reshape(-1, 2)
    xy_map = {i: xy[i] for i in range(xy.shape[0])}
    m = open_matcher(desc)
    out = dict(workload=dict(pairs=a.pairs, rows=a.rows, images=int(desc.shape[0]), table_mb=round(desc.nbytes / 1e6, 1),
                             ratio=0.85, ratio_good=0.6, th_epipolar=3.0, decoy_frac=0.25, seed=a.seed),
               card=card_info(), scene_gen_s=round(gen_s, 1), results={})
    for mutual in (False, True):
        for kind in ("plain", "guided"):  # warm-up
            run_call(m, kind, pairs, F, xy_map, mutual)
        rec = {k: dict(wall_ms=[], total_ms=[], match_kernel_ms=[], finalize_ms=[]) for k in ("plain", "guided")}
        counts = {}
        for _ in range(a.reps):
            for kind in ("plain", "guided"):
                w0 = time.perf_counter()
                res = run_call(m, kind, pairs, F, xy_map, mutual)
                wall = (time.perf_counter() - w0) * 1e3
                t = m.timing()
                rec[kind]["wall_ms"].append(wall)
                for k in ("total_ms", "match_kernel_ms", "finalize_ms"):
                    rec[kind][k].append(t[k])
                counts[kind] = dict(matches=int(len(res.matches)), good=int(res.good.sum()), true_accepted=true_accepted(res, true),
                                    twin_pairs=int(t["twin_pairs"]), match_launches=int(t["match_launches"]))
        summ = {}
        for kind in ("plain", "guided"):
            med = {k: float(np.median(v)) for k, v in rec[kind].items()}
            summ[kind] = dict(**{f"{k}_median": round(v, 3) for k, v in med.items()},
                              **{f"{k}_all": [round(x, 3) for x in v] for k, v in rec[kind].items()},
                              pairs_per_s_total=round(a.pairs / (med["total_ms"] / 1e3), 1),
                              pairs_per_s_wall=round(a.pairs / (med["wall_ms"] / 1e3), 1), **counts[kind])
        summ["guided_over_plain"] = dict(
            total_ms=round(summ["guided"]["total_ms_median"] / summ["plain"]["total_ms_median"], 4),
            match_kernel_ms=round(summ["guided"]["match_kernel_ms_median"] / summ["plain"]["match_kernel_ms_median"], 4))
        out["results"][f"mutual{int(mutual)}"] = summ
        print(json.dumps({f"mutual{int(mutual)}": {k: (v if k == "guided_over_plain" else
                                                      {x: v[x] for x in v if not x.endswith("_all")}) for k, v in summ.items()}}), flush=True)
    m.close()
    # hot groups: each call once in a child process with the debug counters on (a separate run of the kernel's debug build)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "scenes.npz")
        np.savez(path, desc=desc, xy=xy, F=F)
        env = dict(os.environ, MSFM_DEBUG_FLAGS="8")
        hot = {}
        for mutual in (False, True):
            for kind in ("plain", "guided"):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path, kind, str(int(mutual))],
                                   env=env, capture_output=True, text=True)
                if p.returncode != 0:
                    raise SystemExit(p.stdout + p.stderr)
                mt = re.search(r"warp-tiles (\d+) \| hot groups/warp-tile ([0-9.]+)", p.stderr)
                wt, per = int(mt.group(1)), float(mt.group(2))
                hot[f"mutual{int(mutual)}_{kind}"] = dict(warp_tiles=wt, hot_groups_per_warp_tile=per, hot_groups=int(round(wt * per)))
        out["debug_hot_groups"] = hot
        print(json.dumps(dict(debug_hot_groups=hot)), flush=True)
    out["card_after"] = card_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(dict(card=out["card"], written=a.out or None)))


if __name__ == "__main__":
    main()
