"""CPU tests of the host-side logic: synthetic collections, candidate pair lists, the multi-GPU pair scheduler."""
import os

import numpy as np
import pytest

from metricsfm_b200 import scheduler, synth


def test_synth_is_deterministic_and_sift_like():
    a = synth.Collection(512, seed=3)
    b = synth.Collection(512, seed=3)
    x, y = a.image_u8(7), b.image_u8(7)
    np.testing.assert_array_equal(x, y)
    assert x.dtype == np.uint8 and x.shape == (512, 128)
    norms = (x.astype(np.int64) ** 2).sum(1)
    assert 2.3e5 < norms.mean() < 2.7e5            # ||q||^2 ~ 512^2, the real-SIFT regime (SURVEY §8d)
    assert not np.array_equal(a.image_u8(8), x)
    u = a.image_unit(7)
    np.testing.assert_allclose(np.linalg.norm(u, axis=1), 1.0, atol=1e-5)
    np.testing.assert_array_equal(synth.quantize_512(u), x)


def test_pair_lists():
    p = synth.exhaustive_pairs(100)
    assert p.shape == (4950, 2) and (p[:, 0] < p[:, 1]).all()
    assert (np.diff(p[:, 0]) >= 0).all()            # grouped by the first image like the reference's idx1 loop
    g = synth.gps_neighbour_pairs(400, k=30)
    assert (g[:, 0] < g[:, 1]).all() and len(np.unique(g, axis=0)) == len(g)
    assert 400 * 15 <= len(g) <= 400 * 30
    r = synth.retrieval_pairs(500, partners=40)
    assert (r[:, 0] < r[:, 1]).all() and len(np.unique(r, axis=0)) == len(r)


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_shard_pairs_partitions_and_balances(world):
    rng = np.random.default_rng(world)
    rows = rng.integers(1000, 33000, size=300)
    pairs = synth.gps_neighbour_pairs(300, k=20)
    shards = scheduler.shard_pairs(pairs, rows, world)
    assert len(shards) == world
    allidx = np.concatenate(shards)
    np.testing.assert_array_equal(np.sort(allidx), np.arange(len(pairs)))     # a partition: nothing lost, nothing twice
    cost = scheduler.pair_costs(pairs, rows).astype(np.float64)
    loads = np.array([cost[s].sum() for s in shards])
    assert loads.max() <= 1.08 * loads.mean() + cost.max()                    # LPT balance
    for s in shards:
        assert (np.diff(s) > 0).all()                                         # original order kept inside a rank


def test_shard_pairs_degenerate():
    rows = np.array([100, 200, 300])
    assert [len(s) for s in scheduler.shard_pairs(np.zeros((0, 2), np.int32), rows, 4)] == [0, 0, 0, 0]
    one = scheduler.shard_pairs(np.array([[0, 1]]), rows, 4)
    assert sorted(len(s) for s in one) == [0, 0, 0, 1]


def test_stitch_results_roundtrip():
    rng = np.random.default_rng(0)
    n = 37
    counts = rng.integers(0, 6, size=n)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    matches = rng.integers(0, 1000, size=(offsets[-1], 2)).astype(np.int32)
    good = rng.integers(0, 2, size=offsets[-1]).astype(np.uint8)
    ok = rng.integers(0, 2, size=n).astype(np.int32)
    shards = [np.sort(rng.choice(n, size=n // 3, replace=False))]
    rest = np.setdiff1d(np.arange(n), shards[0])
    shards += [rest[::2], rest[1::2]]
    results = []
    for idx in shards:
        so = np.concatenate([[0], np.cumsum(counts[idx])])
        m = np.concatenate([matches[offsets[p]:offsets[p + 1]] for p in idx]) if len(idx) else np.zeros((0, 2), np.int32)
        g = np.concatenate([good[offsets[p]:offsets[p + 1]] for p in idx]) if len(idx) else np.zeros((0,), np.uint8)
        results.append(dict(offsets=so, ok=ok[idx], matches=m, good=g))
    o2, ok2, m2, g2 = scheduler.stitch_results(n, shards, results)
    np.testing.assert_array_equal(o2, offsets)
    np.testing.assert_array_equal(ok2, ok)
    np.testing.assert_array_equal(m2, matches)
    np.testing.assert_array_equal(g2, good)


def test_image_owner_blocks():
    own = scheduler.image_owner(10, 4)
    assert own.tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 2, 3]


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the native one) prints one JSON line with the
    contract's keys; tiny shape so that it runs in seconds without a GPU."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.check_output([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--rows", "512", "--images", "4",
                                   "--steps", "1", "--warmup", "0"], text=True, timeout=300)
    line = json.loads(out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "pairs/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


@pytest.mark.parametrize("budget", [64 << 20, 1 << 20])
def test_bench_dump_outputs(tmp_path, monkeypatch, budget):
    """`bench.py --dump-outputs`: whole match lists of every pair, or of a seeded sample of pairs when they exceed the
    budget; float files only, within the budget, every written list equal to its source, the same bytes whatever the
    order the pairs were matched in."""
    import bench
    from metricsfm_b200.matcher import MatchResult
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    rng = np.random.default_rng(5)
    n = 200
    pairs = np.stack([np.arange(n), np.arange(n) + 1], 1).astype(np.int32)
    counts = rng.integers(0, 4000, size=n)
    counts[::7] = 0
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    res = MatchResult(offs, (counts > 0).astype(np.int32), rng.integers(0, 8192, size=(offs[-1], 2)).astype(np.int32),
                      rng.integers(0, 2, size=offs[-1]).astype(np.uint8))
    bench.dump_outputs(str(tmp_path / "a"), pairs, res)
    order = rng.permutation(n)                                        # the same lists, matched in another order
    rows = np.concatenate([np.arange(offs[p], offs[p + 1]) for p in order])
    shuffled = MatchResult(np.concatenate([[0], np.cumsum(counts[order])]), res.ok[order], res.matches[rows], res.good[rows])
    bench.dump_outputs(str(tmp_path / "b"), pairs[order], shuffled)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["good.npy", "matches.npy", "offsets.npy", "ok.npy", "pairs.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= budget
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    p = got["pairs"][:, 0].astype(np.int64)                          # pair p of the list is (p, p + 1)
    assert (np.diff(p) > 0).all() and (len(p) == n) == (budget == 64 << 20) and len(p) > 0
    o = got["offsets"].astype(np.int64)
    for k, src in enumerate(p):
        np.testing.assert_array_equal(got["matches"][o[k]:o[k + 1]], res.pair(src))
        np.testing.assert_array_equal(got["good"][o[k]:o[k + 1]], res.pair_good(src))
        assert got["ok"][k] == res.ok[src]


def test_numa_pinning_helper_never_raises():
    """pin_to_gpu_numa_node() reports what it did and leaves the process alone when NVML / the device is missing."""
    import os
    from metricsfm_b200 import distributed as D
    before = os.sched_getaffinity(0)
    info = D.pin_to_gpu_numa_node(0)
    assert isinstance(info, dict) and "pinned" in info
    if not info["pinned"]:
        assert os.sched_getaffinity(0) == before
    os.sched_setaffinity(0, before)


def _dead_row_stream(Q, R, rho8, tile=64, group=8, warp=32):
    """numpy restatement of the matching kernel's epilogue with the dead-row rule (metricsfm_b200/csrc/match_kernel.cuh):
    tiles of `tile` reference rows, a group of `group` columns is scored exactly (by every row of the warp) iff some row of
    the warp has a raw accumulator above T = (theta + min norm of the tile) >> 1; theta = best score of a dead row
    (d0 > ((d1 >> 8) + 1) * rho8), second best otherwise; refreshed after a tile that scored something.
    Returns per row (d0, j0, d1_reported, j1, dead_at_end)."""
    N, M = Q.shape[0], R.shape[0]
    acc = Q.astype(np.int64) @ R.astype(np.int64).T
    nb = (R.astype(np.int64) ** 2).sum(1)
    na = (Q.astype(np.int64) ** 2).sum(1)
    score = 2 * acc - nb[None, :]
    NEG = -(1 << 40)
    S0 = np.full(N, NEG); S1 = np.full(N, NEG); J0 = np.full(N, -1); J1 = np.full(N, -1)

    def prune_score():
        d0, d1 = na - S0, na - S1
        dead = (S1 > NEG) & (d0 > ((d1 >> 8) * rho8 + rho8))
        return np.where(dead, S0, S1), dead

    theta, _ = prune_score()
    for t0 in range(0, M, tile):
        cols = np.arange(t0, min(t0 + tile, M))
        T = np.where(theta > NEG, (theta + nb[cols].min()) >> 1, NEG)
        touched = False
        for g0 in range(0, len(cols), group):
            gc = cols[g0:g0 + group]
            flag = acc[:, gc].max(1) > T
            hot = flag.reshape(-1, warp).any(1).repeat(warp)          # warp-wide decision
            if not hot.any():
                continue
            touched = True
            for j in gc:                                              # ascending columns, strict > (lowest index on ties)
                s = score[:, j]
                b0 = hot & (s > S0)
                b1 = hot & ~b0 & (s > S1)
                S1 = np.where(b0, S0, np.where(b1, s, S1)); J1 = np.where(b0, J0, np.where(b1, j, J1))
                S0 = np.where(b0, s, S0); J0 = np.where(b0, j, J0)
        if touched:
            theta, _ = prune_score()
    _, dead = prune_score()
    d1 = np.where(dead, na - S0, na - S1)                             # a row that ends dead reports d1 := d0
    return na - S0, J0, d1, J1, dead


@pytest.mark.parametrize("kind", ["sift", "clusters", "late_match"])
@pytest.mark.parametrize("ratio", [0.5, 0.85])
def test_dead_row_rule_restatement_keeps_every_verdict(kind, ratio):
    """The rule the forward pass uses to skip second-best updates of rows that already fail the ratio test: against the
    exact 2-NN it must keep d0 / nn0 of EVERY row, the exact (d1, nn1) of every row that passes the ratio test, reject
    exactly the rows the exact test rejects, and report for the others a d1 that is a lower bound of the row's distance to
    every reference row but nn0 (what the mutual check's dangerous-row bound relies on, aux_kernels.cuh)."""
    from metricsfm_b200 import synth
    rng = np.random.default_rng(7)
    if kind == "sift":
        col = synth.Collection(768, seed=3)
        R, Q = col.image_u8(0, 768), col.image_u8(1, 512)
    elif kind == "clusters":
        c = rng.integers(0, 100, size=(12, 128))
        R = np.clip(c[rng.integers(0, 12, 640)] + rng.integers(-3, 4, size=(640, 128)), 0, 255).astype(np.uint8)
        Q = np.clip(c[rng.integers(0, 12, 512)] + rng.integers(-3, 4, size=(512, 128)), 0, 255).astype(np.uint8)
    else:
        col = synth.Collection(768, seed=4)
        R, Q = col.image_u8(2, 704), col.image_u8(3, 512)
        Q[:200] = np.clip(R[-200:].astype(np.int32) + rng.integers(-2, 3, size=(200, 128)), 0, 255).astype(np.uint8)  # match in the last tiles
    rho8 = int(np.floor(ratio * 256.0)) + 2                          # msfm_api.cu: ratio rounded up to 1/256 plus one step
    d0, j0, d1, j1, dead = _dead_row_stream(Q, R, rho8)
    D = ((Q.astype(np.int64)[:, None, :] - R.astype(np.int64)[None, :, :]) ** 2).sum(2)
    order = np.argsort(D, axis=1, kind="stable")                     # stable: lowest index on ties
    e0, e1 = order[:, 0], order[:, 1]
    x0, x1 = D[np.arange(len(Q)), e0], D[np.arange(len(Q)), e1]
    np.testing.assert_array_equal(d0, x0)
    np.testing.assert_array_equal(j0, e0)
    accept = (x0.astype(np.float32) / np.maximum(x1, 1).astype(np.float32) < np.float32(ratio)) & (x1 > 0)
    got = (d0.astype(np.float32) / np.maximum(d1, 1).astype(np.float32) < np.float32(ratio)) & (d1 > 0)
    np.testing.assert_array_equal(got, accept)
    np.testing.assert_array_equal(d1[accept], x1[accept])
    np.testing.assert_array_equal(j1[accept], e1[accept])
    assert not (dead & accept).any()
    assert dead.sum() > (len(Q) // 2 if kind == "sift" else 0)          # the rule is at work (on most rows of SIFT-like images)
    Dm = D.copy()
    Dm[np.arange(len(Q)), e0] = np.iinfo(np.int64).max
    assert (d1 <= Dm.min(1)).all()                                    # reported d1 bounds every other distance from below


@pytest.mark.parametrize("kind", ["sift", "clusters"])
def test_mutual_check_from_forward_results_restatement(kind):
    """select_candidates_kernel's mutual cross-check (aux_kernels.cuh) restated in numpy on the rows the dead-row stream
    reports: (A) a per-column table of the nearest claimant among the rows whose nn0 is that column, (B) exact distances
    only for 'dangerous' rows, i.e. rows whose reported d1 (a lower bound of their distance to every column but nn0) does
    not exceed the candidate's d0.  The survivors must be exactly the brute-force mutual matches (lowest index on ties)."""
    from metricsfm_b200 import synth
    rng = np.random.default_rng(11)
    ratio = 0.85
    if kind == "sift":
        col = synth.Collection(768, seed=6)
        R, Q = col.image_u8(0, 640), col.image_u8(1, 512)
    else:
        c = rng.integers(0, 100, size=(10, 128))
        R = np.clip(c[rng.integers(0, 10, 576)] + rng.integers(-3, 4, size=(576, 128)), 0, 255).astype(np.uint8)
        Q = np.clip(c[rng.integers(0, 10, 512)] + rng.integers(-3, 4, size=(512, 128)), 0, 255).astype(np.uint8)
        Q[:40] = R[:40]                                              # exact duplicates: distance ties between query rows
        Q[40:80] = R[:40]
    d0, j0, d1, _, _ = _dead_row_stream(Q, R, int(np.floor(ratio * 256.0)) + 2)
    D = ((Q.astype(np.int64)[:, None, :] - R.astype(np.int64)[None, :, :]) ** 2).sum(2)
    n = len(Q)
    accept = (d0.astype(np.float32) / np.maximum(d1, 1).astype(np.float32) < np.float32(ratio)) & (d1 > 0)
    cand = np.nonzero(accept)[0]
    # (A) column table: (d0, q) minimum over ALL rows, keyed by nn0
    table = {}
    for q in range(n):
        key = (int(d0[q]), q)
        if j0[q] not in table or key < table[j0[q]]:
            table[int(j0[q])] = key
    d0max = int(d0[cand].max()) if len(cand) else -1
    danger = [q for q in range(n) if d1[q] <= d0max]                 # (B) rows that could interfere with some candidate
    survivors, exact_evals = [], 0
    for q in cand:
        j = int(j0[q])
        if table[j] != (int(d0[q]), int(q)):
            continue                                                 # a kind-(A) rival is closer (or ties with a lower index)
        killed = False
        for r in danger:
            if r != q and d1[r] <= d0[q]:
                exact_evals += 1
                d = int(D[r, j])
                if d < d0[q] or (d == d0[q] and r < q):
                    killed = True
        if not killed:
            survivors.append((j, int(q)))
    best_q = np.argmin(D, axis=0)                                     # numpy argmin: lowest index on ties
    expect = [(int(j0[q]), int(q)) for q in cand if best_q[j0[q]] == q]
    assert survivors == expect and len(expect) > 20
    assert exact_evals < n * len(cand) // 4                           # the bound prunes most (row, candidate) combinations
