"""Cost and decision flips of homography-guided re-matching in the float regime (msfm_match_pairs_guided_homography with
rescore_band) on one GPU.

Workload: --pairs independent planar pairs of --rows-row unit-norm float images
(oracle.homography_float_oracle.float_planar_decoy_scene: true correspondences related by the plane's H, a quarter with
a planted look-alike on the epipolar line, a companion row at every true reference keypoint whose descriptor is a noisy
copy of the true one (--companion-sigma, a second orientation at the same location), the rest unrelated rows; float noise,
not quantised), uploaded at scale 512 on a keep_float context, every image distinct (float rows 2 * pairs * rows * 512 B
= 1.7 GB at the defaults, well above the 126 MB L2).  th_transfer 3 px with the scene's H, ratio 0.85 with ratio_good
0.6, mutual off and on.  The arms, H-guided on quantised distances (band 0) and H-guided with the band rows re-scored
in fp32 (one arm per --bands value), alternate in one process after a warm-up of each; per call msfm_last_timing's total_ms,
match_kernel_ms and finalize_ms, and the collect path's events and brute-force batches (msfm_test_last_knn_stats) are
recorded, medians reported.
On --sample pairs, each arm's one-way list is compared row by row with an fp32 H-guided matcher (every row decided on
its fp32 top-2 among the reference rows the H gate allows): a flip is a query row whose (kept, reference row, good)
differs.  The same pairs give the band rows (counted by the restatement, which the tests hold equal to the GPU) and,
from per-pair calls, the events per band row.  The card's name, power limit and SM clock are read in the same run.

    python tools/guided_homography_float_bench.py --out profiles/guided_homography_float_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from guided_float_bench import card_info, flips, fp32_guided_rows, rows_of  # noqa: E402

TH, RATIO, RATIO_GOOD, SCALE, DECOY_FRAC = 3.0, 0.85, 0.6, 512.0, 0.25


def _scene(args):
    from oracle.homography_float_oracle import float_planar_decoy_scene
    seed, rows, comp = args
    return float_planar_decoy_scene(seed, rows, rows, decoy_frac=DECOY_FRAC, dups=False, companion_sigma=comp)


def make_scenes(n_pairs: int, rows: int, seed: int, comp: float):
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        scenes = list(ex.map(_scene, [(seed + i, rows, comp) for i in range(n_pairs)]))
    desc = np.stack([d for s in scenes for d in (s["ref"], s["qry"])])
    xy = np.stack([x for s in scenes for x in (s["xy_ref"], s["xy_qry"])])
    H = np.stack([s["H"] for s in scenes])
    return scenes, desc, xy, H


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--bands", type=float, nargs="+", default=[0.02, 0.05])
    ap.add_argument("--companion-sigma", type=float, default=2.5)
    ap.add_argument("--sample", type=int, default=8)
    ap.add_argument("--seed", type=int, default=5000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("guided_homography_float_bench needs a GPU")
    from metricsfm_b200.matcher import Matcher
    from oracle import homography_float_oracle as hfo
    from oracle import homography_oracle as ho
    card = card_info()
    t0 = time.time()
    scenes, desc, xy, H = make_scenes(a.pairs, a.rows, a.seed, a.companion_sigma)
    gen_s = time.time() - t0
    n_img = desc.shape[0]
    pairs = np.arange(n_img, dtype=np.int32).reshape(-1, 2)
    xy_map = {i: xy[i] for i in range(n_img)}
    m = Matcher(device=0, max_images=n_img, arena_rows=n_img * a.rows + (1 << 16), keep_float=True)
    for i in range(n_img):
        m.upload(i, desc[i], scale=SCALE)
    arms = {"quantised": 0.0, **{f"band{b:g}": b for b in a.bands}}

    def call(band, mutual, sel=slice(None)):
        return m.match_pairs_guided_homography(pairs[sel], H[sel], xy_map, th_transfer=TH, ratio=RATIO,
                                               ratio_good=RATIO_GOOD, mutual=mutual, rescore_band=band)

    out = dict(workload=dict(pairs=a.pairs, rows=a.rows, images=n_img, float_table_mb=round(desc.nbytes / 1e6, 1),
                             scale=SCALE, ratio=RATIO, ratio_good=RATIO_GOOD, th_transfer=TH, bands=a.bands,
                             decoy_frac=DECOY_FRAC, companion_sigma=a.companion_sigma, seed=a.seed, reps=a.reps),
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
        for kind in arms:
            if kind != "quantised":
                summ[f"{kind}_over_quantised"] = {k: round(summ[kind][f"{k}_median"] / summ["quantised"][f"{k}_median"], 4)
                                                  for k in ("total_ms", "match_kernel_ms", "finalize_ms")}
        out["results"][f"mutual{int(mutual)}"] = summ
        print(json.dumps({f"mutual{int(mutual)}": {k: {x: y for x, y in v.items() if not x.endswith("_all")}
                                                  for k, v in summ.items()}}), flush=True)
    # sample: flips of the one-way lists against an fp32 H-guided matcher, band rows, events per band row
    sample = list(range(min(a.sample, a.pairs)))
    fl = {k: 0 for k in arms}
    rows = 0
    band_rows = {b: 0 for b in a.bands}
    events = {b: 0 for b in a.bands}
    for p in sample:
        s = scenes[p]
        ref_rows = fp32_guided_rows(s, ho.gate_h32(s["H"], s["xy_ref"], s["xy_qry"], TH))
        n = len(s["qry"])
        rows += n
        for kind in arms:
            fl[kind] += flips(rows_of(lists[(kind, False)], p, n), ref_rows)
        for b in a.bands:
            exp = hfo.match_pair_guided_h_float(s["ref"], s["qry"], s["xy_ref"], s["xy_qry"], s["H"], TH, RATIO, band=b,
                                                ratio_good=RATIO_GOOD)
            band_rows[b] += int(exp["band"].sum())
            call(b, False, slice(p, p + 1))
            events[b] += m._test_last_knn_stats()[0]
    out["sample"] = dict(pairs=len(sample), query_rows=rows,
                         band_rows={f"band{b:g}": v for b, v in band_rows.items()},
                         band_row_fraction={f"band{b:g}": round(v / max(rows, 1), 5) for b, v in band_rows.items()},
                         events={f"band{b:g}": v for b, v in events.items()},
                         events_per_band_row={f"band{b:g}": round(events[b] / max(band_rows[b], 1), 3) for b in a.bands},
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
