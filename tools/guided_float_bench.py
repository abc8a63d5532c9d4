"""Cost and decision flips of guided re-matching in the float regime (msfm_match_pairs_guided with rescore_band) on one
GPU.

Workload: --pairs independent two-view scene pairs of --rows-row unit-norm float images
(oracle.guided_float_oracle.float_decoy_scene: true correspondences, a quarter with a planted look-alike off the
epipolar line, the rest unrelated rows; float noise, not quantised), uploaded at scale 512 on a keep_float context, every
image distinct (float rows 2 * pairs * rows * 512 B = 1.7 GB at the defaults, well above the 126 MB L2).  th_epipolar
3 px with the scene's F, ratio 0.85 with ratio_good 0.6, mutual off and on.  The two arms, guided on quantised distances
(band 0) and guided with the band rows re-scored in fp32 (band --band), alternate in one process after a warm-up of each;
per call msfm_last_timing's total_ms, match_kernel_ms and finalize_ms, and the collect path's events and brute-force
batches (msfm_test_last_knn_stats) are recorded, medians reported.
On --sample pairs, each arm's one-way list is compared row by row with an fp32 guided matcher (every row decided on its
fp32 top-2 among the allowed reference rows): a flip is a query row whose (kept, reference row, good) differs.  The same
pairs give the band rows (counted by the restatement, which the tests hold equal to the GPU) and, from per-pair calls,
the events per band row.  The card's name and power limit are read in the same run.

    python tools/guided_float_bench.py --out profiles/guided_float_bench_1gpu.json
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

TH, RATIO, RATIO_GOOD, SCALE = 3.0, 0.85, 0.6, 512.0


def _scene(args):
    from oracle.guided_float_oracle import float_decoy_scene
    seed, rows = args
    return float_decoy_scene(seed, rows, rows, decoy_frac=0.25, dups=False)


def make_scenes(n_pairs: int, rows: int, seed: int):
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        scenes = list(ex.map(_scene, [(seed + i, rows) for i in range(n_pairs)]))
    desc = np.stack([d for s in scenes for d in (s["ref"], s["qry"])])
    xy = np.stack([x for s in scenes for x in (s["xy_ref"], s["xy_qry"])])
    F = np.stack([s["F"] for s in scenes])
    return scenes, desc, xy, F


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [x.strip() for x in line.split(",")]
    return dict(name=parts[0] if parts else None, power_limit=parts[1] if len(parts) > 1 else None,
                max_sm_clock=parts[2] if len(parts) > 2 else None)


def fp32_guided_rows(s, allowed=None):
    """Per query row of an fp32 guided matcher: (kept, reference row, good); `allowed` defaults to the epipolar gate.
    The fp32 top-2 among the allowed rows is found exactly in index order among the allowed rows whose float64 distance
    is within a relative 2^-14 of the float64 second distance (the fp32 sum is within 130 * 2^-24 of it), so only a few
    rows per query are summed in fp32."""
    from oracle import guided_float_oracle as gfo
    from oracle import guided_oracle as gdo
    ref, qry = s["ref"].astype(np.float64), s["qry"].astype(np.float64)
    if allowed is None:
        allowed = gdo.gate_f32(s["F"], s["xy_ref"], s["xy_qry"], TH)
    D = (qry * qry).sum(1)[:, None] + (ref * ref).sum(1)[None, :] - 2.0 * (qry @ ref.T)
    D[~allowed] = np.inf
    n = len(qry)
    keep = np.zeros(n, bool)
    good = np.zeros(n, bool)
    j0 = np.full(n, -1, np.int64)
    part = np.partition(D, 1, axis=1)[:, 1] if D.shape[1] > 1 else np.full(n, np.inf)
    for q in np.nonzero(np.isfinite(part))[0]:
        cand = np.nonzero(D[q] <= part[q] * (1 + 2.0 ** -14) + 1e-12)[0]
        ids, d = gfo.masked_knn2_f32(s["ref"][cand], s["qry"][q:q + 1], np.ones((1, len(cand)), bool))
        r = d[0, 0] / d[0, 1] if d[0, 1] > 0 else np.float32(np.nan)
        keep[q] = r < np.float32(RATIO)
        good[q] = keep[q] and r < np.float32(RATIO_GOOD)
        j0[q] = cand[ids[0, 0]]
    return keep, j0, good


def rows_of(res, p, n):
    keep = np.zeros(n, bool)
    j = np.full(n, -1, np.int64)
    good = np.zeros(n, bool)
    m, g = res.pair(p), res.pair_good(p)
    keep[m[:, 1]] = True
    j[m[:, 1]] = m[:, 0]
    good[m[:, 1]] = g.astype(bool)
    return keep, j, good


def flips(a, b):
    ka, ja, ga = a
    kb, jb, gb = b
    return int(((ka != kb) | (ka & kb & ((ja != jb) | (ga != gb)))).sum())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--band", type=float, default=0.02)
    ap.add_argument("--sample", type=int, default=8)
    ap.add_argument("--seed", type=int, default=3000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("guided_float_bench needs a GPU")
    from metricsfm_b200.matcher import Matcher
    from oracle import guided_float_oracle as gfo
    card = card_info()
    t0 = time.time()
    scenes, desc, xy, F = make_scenes(a.pairs, a.rows, a.seed)
    gen_s = time.time() - t0
    n_img = desc.shape[0]
    pairs = np.arange(n_img, dtype=np.int32).reshape(-1, 2)
    xy_map = {i: xy[i] for i in range(n_img)}
    m = Matcher(device=0, max_images=n_img, arena_rows=n_img * a.rows + (1 << 16), keep_float=True)
    for i in range(n_img):
        m.upload(i, desc[i], scale=SCALE)
    arms = {"quantised": 0.0, "rescored": a.band}

    def call(band, mutual, sel=slice(None)):
        return m.match_pairs_guided(pairs[sel], F[sel], xy_map, th_epipolar=TH, ratio=RATIO, ratio_good=RATIO_GOOD,
                                    mutual=mutual, rescore_band=band)

    out = dict(workload=dict(pairs=a.pairs, rows=a.rows, images=n_img, float_table_mb=round(desc.nbytes / 1e6, 1),
                             scale=SCALE, ratio=RATIO, ratio_good=RATIO_GOOD, th_epipolar=TH, band=a.band, decoy_frac=0.25,
                             seed=a.seed, reps=a.reps),
               card=card, scene_gen_s=round(gen_s, 1), results={})
    lists = {}
    for mutual in (False, True):
        for band in arms.values():  # warm-up
            call(band, mutual)
        rec = {k: dict(total_ms=[], match_kernel_ms=[], finalize_ms=[], events=[], brute_force_batches=[]) for k in arms}
        for _ in range(a.reps):
            for kind, band in arms.items():
                res = call(band, mutual)
                t = m.timing()
                for k in ("total_ms", "match_kernel_ms", "finalize_ms"):
                    rec[kind][k].append(t[k])
                if band > 0:
                    ev, bf = m._test_last_knn_stats()
                    rec[kind]["events"].append(ev)
                    rec[kind]["brute_force_batches"].append(bf)
                lists[(kind, mutual)] = res
        summ = {}
        for kind in arms:
            summ[kind] = {f"{k}_median": round(float(np.median(v)), 3) for k, v in rec[kind].items() if v}
            summ[kind].update({f"{k}_all": [round(float(x), 3) for x in v] for k, v in rec[kind].items() if v})
            summ[kind]["matches"] = int(len(lists[(kind, mutual)].matches))
        summ["rescored_over_quantised"] = {k: round(summ["rescored"][f"{k}_median"] / summ["quantised"][f"{k}_median"], 4)
                                           for k in ("total_ms", "match_kernel_ms", "finalize_ms")}
        out["results"][f"mutual{int(mutual)}"] = summ
        print(json.dumps({f"mutual{int(mutual)}": {k: {x: y for x, y in v.items() if not x.endswith("_all")}
                                                  for k, v in summ.items()}}), flush=True)
    # sample: flips of the one-way lists against an fp32 guided matcher, band rows, events per band row
    sample = list(range(min(a.sample, a.pairs)))
    fl = {k: 0 for k in arms}
    rows = band_rows = events = 0
    for p in sample:
        s = scenes[p]
        ref_rows = fp32_guided_rows(s)
        n = len(s["qry"])
        rows += n
        for kind in arms:
            fl[kind] += flips(rows_of(lists[(kind, False)], p, n), ref_rows)
        exp = gfo.match_pair_guided_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["F"], TH, RATIO, band=a.band,
                                          ratio_good=RATIO_GOOD)
        band_rows += int(exp["band"].sum())
        call(a.band, False, slice(p, p + 1))
        events += m._test_last_knn_stats()[0]
    out["sample"] = dict(pairs=len(sample), query_rows=rows, band_rows=band_rows,
                         band_row_fraction=round(band_rows / max(rows, 1), 5),
                         events=events, events_per_band_row=round(events / max(band_rows, 1), 3),
                         flips={k: v for k, v in fl.items()}, flip_rate={k: v / max(rows, 1) for k, v in fl.items()})
    print(json.dumps(dict(sample=out["sample"])), flush=True)
    m.close()
    out["card_after"] = card_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(dict(card=out["card"], written=a.out or None)))


if __name__ == "__main__":
    main()
