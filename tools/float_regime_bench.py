"""Float-regime throughput: unit-norm float rows (scale 512) matched with and without fp32 re-scoring of the rows near
a ratio threshold (msfm_params.rescore_band).  Device time of msfm_match_pairs over all pairs of `--images` images.
The re-scored arms also report the events the collect pass scored and the batches the brute force decided (the
library's test hook), and `band_rows` the query rows in the band (from the integer 2-NN of msfm_knn2_pairs).
Run on a GPU box: `python tools/float_regime_bench.py [--images 40] [--rows 8192] [--band 0.02]`; prints one JSON line."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from metricsfm_b200 import synth  # noqa: E402
from metricsfm_b200.matcher import Matcher  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=40)
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--band", type=float, default=0.02)
    ap.add_argument("--ratio", type=float, default=0.85)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    col = synth.Collection(args.rows, seed=0)
    pairs = [(i, j) for i in range(args.images) for j in range(i + 1, args.images)]
    out = {"images": args.images, "rows": args.rows, "pairs": len(pairs), "ratio": args.ratio, "band": args.band}
    with Matcher(device=0, max_images=args.images, arena_rows=args.images * (args.rows + 256), keep_float=True) as m:
        for i in range(args.images):
            m.upload(i, col.image_unit(i), scale=512.0)
        _, _, d = m.knn2_pairs(pairs)
        with np.errstate(divide="ignore", invalid="ignore"):
            r = d[:, 0] / d[:, 1]
        out["band_rows"] = int((np.abs(r - np.float32(args.ratio)) <= np.float32(args.band) * np.float32(args.ratio)).sum())
        for mutual in (False, True):
            for band in (0.0, args.band):
                ms = []
                for _ in range(args.repeats + 1):
                    res = m.match_pairs(pairs, args.ratio, mutual=mutual, rescore_band=band)
                    ms.append(m.timing()["total_ms"])
                best = min(ms[1:])
                arm = {"device_ms": best, "pairs_per_s": len(pairs) / best * 1e3, "matches": int(res.offsets[-1])}
                if band > 0:
                    arm["collect_events"], arm["brute_force_batches"] = m._test_last_knn_stats()
                    arm["events_per_band_row"] = arm["collect_events"] / max(out["band_rows"], 1)
                out[f"{'mutual' if mutual else 'oneway'}_{'rescored' if band > 0 else 'quantised'}"] = arm
    print(json.dumps(out))


if __name__ == "__main__":
    main()
