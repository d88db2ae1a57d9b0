"""Paired-end best-hit search against the route to the same answer through the existing entry points, timed end to end
(host arrays in -> host arrays out) in one process on one GPU, in alternating rounds, on the config-2 segments (8
synthetic influenza-A segments) with synthetic FR read pairs of 150-nt mates (synth.paired_reads):

  A  the paired align entry point (align_paired_best_hit_arrays);
  B  four single-strand score calls (mate 1, rc(mate 1), mate 2, rc(mate 2)), the pair selection in numpy, one
     align_arrays call per segment on the host-gathered selected mates (a one-sequence context per segment), and
     tlen / proper in numpy.

A and B must return identical arrays.  Also reports assignment quality against the generator's truth, next to two
independent both-strand best-hit calls (one per mate file).

    python scripts/bench_paired.py [--n 1000000] [--rounds 3] [--out profiles/paired_cfg2.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402

from ab_gap_imm import gpu_info  # noqa: E402
from zoe_b200 import CudaProfiles, WeightMatrix, _lib, synth  # noqa: E402
from zoe_b200.alignment import _COMPLEMENT  # noqa: E402

PAIR_KEYS = ("hit", "proper", "tlen")
MATE_KEYS = ("strand", "score", "status", "tier", "runner_up", "ref_start", "ref_end", "query_start", "query_end",
             "hazard", "cigar_off")
MIN_INSERT, MAX_INSERT = 200, 500  # the generator's insert mean 350 +- 3 sd
COMP = np.frombuffer(_COMPLEMENT, dtype=np.uint8)


def rc2d(m):
    return np.ascontiguousarray(COMP[m[:, ::-1]])


def pair_rule(status, score, tier):
    """[n, 2 (mate), P, 2 (strand)] -> hit [n], per-mate strand / score / status / tier / runner_up [2n]."""
    n, _, P, _ = status.shape
    st1, sc1 = status[:, 0], score[:, 0].astype(np.int64)
    st2, sc2 = status[:, 1, :, ::-1], score[:, 1, :, ::-1].astype(np.int64)
    key = (((st1 == _lib.OVERFLOWED).astype(np.int64) + (st2 == _lib.OVERFLOWED)) << 40)
    key += np.where(st1 == _lib.SOME, sc1, 0) + np.where(st2 == _lib.SOME, sc2, 0)
    c = np.argmax(key.reshape(n, 2 * P), axis=1)
    hit, o = c // 2, c % 2
    rows = np.arange(n)
    other = np.ones((n, P), bool)
    other[rows, hit] = False
    out = {k: np.zeros((n, 2), dtype=dt) for k, dt in
           (("strand", np.uint8), ("score", np.uint32), ("status", np.uint8), ("tier", np.uint8), ("runner_up", np.uint32))}
    for m in range(2):
        s = o if m == 0 else 1 - o
        st = status[rows, m, hit, s]
        out["strand"][:, m], out["status"][:, m] = s, st
        out["score"][:, m], out["tier"][:, m] = score[rows, m, hit, s], tier[rows, m, hit, s]
        ru = np.where((status[:, m] == _lib.SOME) & other[:, :, None], score[:, m], 0).reshape(n, -1).max(axis=1)
        out["runner_up"][:, m] = np.where(st == _lib.SOME, ru, 0)
    return hit.astype(np.uint32), {k: v.reshape(-1) for k, v in out.items()}


def pair_outputs(status, strand, start, end):
    st, sd = status.reshape(-1, 2), strand.reshape(-1, 2)
    s, e = start.reshape(-1, 2).astype(np.int64), end.reshape(-1, 2).astype(np.int64)
    both = (st == _lib.SOME).all(axis=1)
    extent = e.max(axis=1) - s.min(axis=1)
    o = sd[:, 0]
    tlen = np.where((s[:, 0] < s[:, 1]) | ((s[:, 0] == s[:, 1]) & (o == 0)), extent, -extent)
    fwd, rev = np.where(o == 0, s[:, 0], s[:, 1]), np.where(o == 0, s[:, 1], s[:, 0])
    proper = both & (fwd <= rev) & (extent >= MIN_INSERT) & (extent <= MAX_INSERT)
    return np.where(both, tlen, 0).astype(np.int32), proper.astype(np.uint8)


def run_a(prof, m1, m2):
    (b1, o1), (b2, o2) = synth.fixed_len_batch(m1), synth.fixed_len_batch(m2)
    return prof.align_paired_best_hit_arrays(b1, o1, b2, o2, min_insert=MIN_INSERT, max_insert=MAX_INSERT)


def run_b(prof, singles, m1, m2):
    n, L = m1.shape
    calls = [[prof.sw_score_arrays(*synth.fixed_len_batch(x)) for x in (m, rc2d(m))] for m in (m1, m2)]
    st, sc, ti = (np.stack([np.stack([calls[m][s][k] for s in range(2)], axis=2) for m in range(2)], axis=1)
                  for k in (1, 0, 2))
    hit, out = pair_rule(st, sc, ti)
    mates = np.stack([m1, m2], axis=1).reshape(2 * n, L)              # mate order 2i + m
    sel = np.where(out["strand"][:, None] == 1, COMP[mates[:, ::-1]], mates)
    mhit = np.repeat(hit, 2)
    some = out["status"] == _lib.SOME
    for k in ("ref_start", "ref_end", "query_start", "query_end"):
        out[k] = np.zeros(2 * n, dtype=np.uint32)
    out["hazard"] = np.zeros(2 * n, dtype=np.uint8)
    lens = np.zeros(2 * n, dtype=np.int64)
    words = {}
    for j, pj in enumerate(singles):
        idx = np.nonzero(some & (mhit == j))[0]
        if idx.size == 0:
            continue
        a = pj.align_arrays(*synth.fixed_len_batch(sel[idx]))
        for k in ("ref_start", "ref_end", "query_start", "query_end", "hazard"):
            out[k][idx] = a[k][:idx.size]
        lens[idx] = np.diff(a["cigar_off"][:idx.size + 1].astype(np.int64))
        words[j] = (idx, a["cigar"], a["cigar_off"])
    off = np.zeros(2 * n + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    cigar = np.zeros(int(off[-1]), dtype=np.uint32)
    for idx, cw, co in words.values():
        ln = lens[idx]
        src = np.repeat(co[:idx.size].astype(np.int64), ln) + (np.arange(int(ln.sum())) - np.repeat(np.cumsum(ln) - ln, ln))
        dst = np.repeat(off[idx].astype(np.int64), ln) + (np.arange(int(ln.sum())) - np.repeat(np.cumsum(ln) - ln, ln))
        cigar[dst] = cw[src]
    out["cigar_off"], out["cigar"], out["hit"] = off, cigar, hit
    out["tlen"], out["proper"] = pair_outputs(out["status"], out["strand"], out["ref_start"], out["ref_end"])
    return out


def same(a, b):
    for k in PAIR_KEYS + MATE_KEYS:
        if not np.array_equal(np.asarray(a[k]), np.asarray(b[k])):
            return False, k
    t = int(b["cigar_off"][-1])
    return bool(np.array_equal(a["cigar"][:t], b["cigar"][:t])), "cigar"


def quality(a, truth):
    """Pairs whose mates land on the true segment in the true orientation (both Some), and the proper fraction."""
    some = (a["status"].reshape(-1, 2) == _lib.SOME).all(axis=1)
    on_true = some & (a["hit"] == truth["target"]) & (a["strand"][0::2] == truth["strand"])
    return {"pairs_on_true_segment_and_orientation": float(on_true.mean()), "proper_fraction": float(a["proper"].mean())}


def independent(prof, m1, m2, truth):
    """Two independent both-strand best-hit calls, one per mate file, scored with the same pair rule."""
    r = [prof.align_best_hit_arrays(*synth.fixed_len_batch(m), both_strands=True) for m in (m1, m2)]
    some = (r[0]["status"] == _lib.SOME) & (r[1]["status"] == _lib.SOME)
    same_seg = some & (r[0]["hit"] == r[1]["hit"])
    opposite = same_seg & (r[0]["strand"] != r[1]["strand"])
    status = np.stack([np.where(opposite, r[0]["status"], _lib.UNMAPPED), r[1]["status"]], axis=1).reshape(-1)
    inter = {k: np.stack([r[0][k], r[1][k]], axis=1).reshape(-1) for k in ("strand", "ref_start", "ref_end")}
    _, proper = pair_outputs(status, inter["strand"], inter["ref_start"], inter["ref_end"])
    on_true = opposite & (r[0]["hit"] == truth["target"]) & (r[0]["strand"] == truth["strand"])
    return {"pairs_on_true_segment_and_orientation": float(on_true.mean()),
            "pairs_mates_on_different_segments": float((some & ~same_seg).mean()),
            "pairs_mates_on_same_strand": float((same_seg & ~opposite).mean()),
            "proper_fraction": float(proper.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "paired_cfg2.json"))
    args = ap.parse_args()
    w25 = WeightMatrix.new_dna_matrix(2, -5, b"N")  # bench.py's scoring: +2 / -5, gap open -10, gap extend -1
    targets = synth.config2(n_reads=0)[0]
    m1, m2, truth = synth.paired_reads(np.random.default_rng(51), targets, args.n)
    prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], w25, -10, -1, devices=[0])
    singles = [CudaProfiles.new_with_w256([bytes(t)], w25, -10, -1, devices=[0]) for t in targets]
    res = {"gpu": gpu_info(), "n_pairs": args.n, "mate_len": 150, "insert": "normal(350, 50)",
           "insert_bounds": [MIN_INSERT, MAX_INSERT], "rounds": args.rounds,
           "timing": "host clock around each call (host arrays in -> host arrays out), median of alternating rounds"}
    a, b = run_a(prof, m1, m2), run_b(prof, singles, m1, m2)  # warm-up, and the outputs compared
    ok, key = same(a, b)
    times = {"A": [], "B": []}
    for _ in range(args.rounds):
        for w in ("A", "B"):
            t0 = time.perf_counter()
            run_a(prof, m1, m2) if w == "A" else run_b(prof, singles, m1, m2)
            times[w].append((time.perf_counter() - t0) * 1e3)
    run_a(prof, m1, m2)
    res["identical_A_B"] = ok if ok else f"differ at {key}"
    res["ms_median"] = {w: statistics.median(v) for w, v in times.items()}
    res["ms_range"] = {w: [min(v), max(v)] for w, v in times.items()}
    res["B_over_A"] = res["ms_median"]["B"] / res["ms_median"]["A"]
    res["stats_A"] = prof.last_stats()
    res["quality_paired"] = quality(a, truth)
    res["quality_two_independent_best_hit_calls"] = independent(prof, m1, m2, truth)
    for p in [prof] + singles:
        p.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
