"""Cost of homography-guided re-matching (msfm_match_pairs_guided_homography) against the F-guided call
(msfm_match_pairs_guided) and the unconstrained matcher (msfm_match_pairs) on one GPU, and of msfm_geo_homography.

Workload: --pairs independent planar pairs of --rows-row images (oracle.homography_oracle.planar_decoy_scene: true
correspondences on a ground plane, a quarter of them with a planted look-alike on the epipolar line, the rest unrelated
rows), every image distinct, so that the descriptor table (2 * pairs * rows * 128 B, 420 MB at the defaults) is well
above the 126 MB L2.  Two variants of the scenes are measured.  "with_companions": every true reference keypoint has a
companion reference row at exactly the same position with an unrelated descriptor, so the H gate's disc around a true
match holds a second neighbour (HOMOG-SPEC rejects a row with fewer than two allowed reference rows).
"without_companions": those rows sit at random positions, so at th = 4 px almost every row has fewer than two allowed
reference rows and the H gate rejects it.  Ratio 0.85 with ratio_good 0.6, mutual off and on, th = 4 px with the
scene's H and F.  The three calls alternate in one process after a warm-up of each; per call the host wall time, msfm_last_timing's total_ms and
match_kernel_ms, and the match counts (all, planted true correspondences, decoyed true correspondences) are recorded,
medians reported.  msfm_geo_homography is timed on the unconstrained lists of the same pairs.  The card's name and power
limit are read in the same run.

    python tools/guided_homography_bench.py --out profiles/guided_homography_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _scene(args):
    from oracle.homography_oracle import planar_decoy_scene
    seed, rows, companions = args
    return planar_decoy_scene(seed, rows, rows, decoy_frac=0.25, dups=False, companions=companions)


def make_scenes(n_pairs: int, rows: int, seed: int, companions: bool):
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        scenes = list(ex.map(_scene, [(seed + i, rows, companions) for i in range(n_pairs)]))
    desc = np.stack([d for s in scenes for d in (s["ref"], s["qry"])])
    xy = np.stack([x for s in scenes for x in (s["xy_ref"], s["xy_qry"])])
    H = np.stack([s["H"] for s in scenes])
    F = np.stack([s["F"] for s in scenes])
    return desc, xy, H, F, [s["true"] for s in scenes], [s["decoyed"] for s in scenes]


def kept(res, sets) -> int:
    from oracle.homography_oracle import kept as k
    return sum(k(res.pair(p), s) for p, s in enumerate(sets))


def card() -> dict:
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      text=True).strip().splitlines()[0]
        name, power, clk = (x.strip() for x in out.split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except (OSError, subprocess.CalledProcessError) as e:
        return dict(error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--th", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=9000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from metricsfm_b200.matcher import Matcher
    out = dict(card=card(), workloads={})
    n_img = 2 * a.pairs
    pairs = [(2 * p, 2 * p + 1) for p in range(a.pairs)]
    with Matcher(device=0, max_images=n_img, arena_rows=n_img * a.rows + (1 << 16)) as m:
        for companions in (True, False):
            name = "with_companions" if companions else "without_companions"
            t0 = time.time()
            desc, xy, H, F, true, decoyed = make_scenes(a.pairs, a.rows, a.seed, companions)
            wl = dict(pairs=a.pairs, rows=a.rows, th=a.th, ratio=0.85, ratio_good=0.6, decoy_frac=0.25,
                      true_per_pair=len(true[0]), decoyed_per_pair=len(decoyed[0]),
                      companion_rows_at_true_keypoints=companions, scene_seconds=round(time.time() - t0, 1))
            out["workloads"][name] = dict(workload=wl, results={})
            xy_map = {i: xy[i] for i in range(n_img)}
            m.release_all()
            m.upload_batch(list(range(n_img)), list(desc))
            calls = {
                "plain": lambda mu: m.match_pairs(pairs, 0.85, ratio_good=0.6, mutual=mu),
                "f_guided": lambda mu: m.match_pairs_guided(pairs, F, xy_map, th_epipolar=a.th, ratio=0.85, ratio_good=0.6,
                                                            mutual=mu),
                "h_guided": lambda mu: m.match_pairs_guided_homography(pairs, H, xy_map, th_transfer=a.th, ratio=0.85,
                                                                       ratio_good=0.6, mutual=mu),
            }
            for mutual in (False, True):
                rec = {k: dict(wall_ms=[], total_ms=[], kernel_ms=[]) for k in calls}
                last = {}
                for k, fn in calls.items():  # warm-up
                    fn(mutual)
                for _ in range(a.reps):
                    for k, fn in calls.items():
                        t = time.perf_counter()
                        r = fn(mutual)
                        w = (time.perf_counter() - t) * 1e3
                        tm = m.timing()
                        rec[k]["wall_ms"].append(w)
                        rec[k]["total_ms"].append(tm["total_ms"])
                        rec[k]["kernel_ms"].append(tm["match_kernel_ms"])
                        last[k] = r
                res = {}
                for k in calls:
                    r = last[k]
                    res[k] = dict(wall_ms=float(np.median(rec[k]["wall_ms"])), total_ms=float(np.median(rec[k]["total_ms"])),
                                  kernel_ms=float(np.median(rec[k]["kernel_ms"])), matches=int(len(r.matches)),
                                  true_kept=kept(r, true), decoyed_kept=kept(r, decoyed),
                                  samples_total_ms=rec[k]["total_ms"])
                for k in ("f_guided", "h_guided"):
                    res[k]["total_vs_plain"] = res[k]["total_ms"] / res["plain"]["total_ms"]
                out["workloads"][name]["results"][f"mutual{int(mutual)}"] = res
                print(json.dumps({name: {f"mutual{int(mutual)}": {k: {kk: v for kk, v in d.items() if kk != "samples_total_ms"}
                                                                  for k, d in res.items()}}}), flush=True)
            if companions:
                # geometric verification with the homography model on the unconstrained lists
                first = m.match_pairs(pairs, 0.85, ratio_good=0.6)
                m.geo_homography(pairs, first, xy_map, th=a.th, seed=1)
                ms, wall = [], []
                for r in range(a.reps):
                    t = time.perf_counter()
                    ok, inl, _, _ = m.geo_homography(pairs, first, xy_map, th=a.th, seed=1 + r)
                    wall.append((time.perf_counter() - t) * 1e3)
                    ms.append(m.timing()["finalize_ms"])
                out["geo_homography"] = dict(workload=name, kernel_ms=float(np.median(ms)), wall_ms=float(np.median(wall)),
                                             pairs_ok=int(ok.sum()), median_inliers=float(np.median(inl)),
                                             samples_kernel_ms=ms)
                print(json.dumps({"geo_homography": {k: v for k, v in out["geo_homography"].items()
                                                     if k != "samples_kernel_ms"}}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
