"""Both-strand search, three ways, timed end to end (host arrays in -> host arrays out) in one process on one GPU:

  A  the both-strand entry point (strand expansion and selection on the device);
  B  a forward call plus a call on the batch reverse-complemented on the host, selection in numpy;
  C  one call on a batch doubled on the host (read, reverse complement, interleaved), selection in numpy;

plus the forward-only call for reference, in alternating rounds.  Config 2 (score, 1M x 150 nt reads x 8 segments) and
config 3 (align, 1M x 150 nt reads x the HA).  The three ways must return identical arrays.  Also reports, on config 3,
how many reads reach a Some score of at least 200 forward-only and with both strands.

    python scripts/bench_strands.py [--n 1000000] [--rounds 5] [--out profiles/both_strands_cfg2_cfg3.json]
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

COMP = np.frombuffer(_COMPLEMENT, dtype=np.uint8)
PAIR_KEYS = ("score", "status", "tier", "ref_start", "ref_end", "query_start", "query_end", "hazard")


def rank(status, score):
    return np.where(status == _lib.OVERFLOWED, np.int64(1) << 40, np.where(status == _lib.SOME, score.astype(np.int64) + 1, 0))


def select(f, r, keys, cigar):
    """The selection rule on two strands' flat outputs; f / r carry "lo" / "ln" (CIGAR start, length) and "cigar"."""
    rev = rank(r["status"], r["score"]) > rank(f["status"], f["score"])
    out = {k: np.where(rev, r[k], f[k]) for k in keys}
    out["strand"] = rev.astype(np.uint8)
    if cigar:
        ln = np.where(rev, r["ln"], f["ln"])
        off = np.zeros(len(ln) + 1, dtype=np.uint64)
        np.cumsum(ln, out=off[1:])
        lo = np.where(rev, r["lo"], f["lo"]).astype(np.int64)
        src = np.repeat(lo - off[:-1].astype(np.int64), ln) + np.arange(int(off[-1]))
        from_rev = np.repeat(rev, ln)
        words = f["cigar"][np.where(from_rev, 0, src)]
        words[from_rev] = r["cigar"][src[from_rev]]
        out["cigar_off"], out["cigar"] = off, words
    return out


def strand_view(a, rows, pairs, cigar):
    """The outputs of the given pair rows (a slice of a flat result) as a selection input."""
    v = {k: a[k][rows] for k in PAIR_KEYS if k in a}
    if cigar:
        v["lo"] = a["cigar_off"][:-1][rows]
        v["ln"] = np.diff(a["cigar_off"])[rows].astype(np.int64)
        v["cigar"] = a["cigar"]
    return v


def run(prof, kind, reads, way):
    """One end-to-end call: reads is an [n, L] uint8 array; returns flat host arrays."""
    n, L = reads.shape
    np_ = prof.n_profiled
    cigar = kind == "align"
    keys = [k for k in PAIR_KEYS if cigar or k in ("score", "status", "tier")]

    def call(batch, both=False):
        buf, offs = synth.fixed_len_batch(batch)
        if kind == "score":
            res = (prof.sw_score_both_strands_arrays if both else prof.sw_score_arrays)(buf, offs)
            return dict(zip(("score", "status", "tier", "strand"), (x.ravel() for x in res)))
        return (prof.align_both_strands_arrays if both else prof.align_arrays)(buf, offs)

    if way == "fwd":
        return call(reads)
    if way == "A":
        return call(reads, both=True)
    if way == "B":
        f = call(reads)
        r = call(COMP[reads[:, ::-1]])
        rows = np.arange(n * np_)
        return select(strand_view(f, rows, n * np_, cigar), strand_view(r, rows, n * np_, cigar), keys, cigar)
    doubled = np.empty((2 * n, L), dtype=np.uint8)
    doubled[0::2] = reads
    doubled[1::2] = COMP[reads[:, ::-1]]
    d = call(doubled)
    idx = (np.arange(n)[:, None] * 2 * np_ + np.arange(np_)[None, :]).ravel()
    return select(strand_view(d, idx, n * np_, cigar), strand_view(d, idx + np_, n * np_, cigar), keys, cigar)


def same(a, b, pairs):
    for k, v in a.items():
        if k in ("hazard",) and k not in b:
            continue
        n = int(a["cigar_off"][pairs]) if k == "cigar" else (pairs + 1 if k == "cigar_off" else pairs)
        if k in b and not np.array_equal(np.asarray(v)[:n], np.asarray(b[k])[:n]):
            return False
    return True


def bench(name, kind, prof, reads, rounds):
    n = reads.shape[0]
    pairs = n * prof.n_profiled
    ways = ["fwd", "A", "B", "C"]
    outs = {w: run(prof, kind, reads, w) for w in ways}  # warm-up, and the outputs compared below
    parity = all(same(outs["A"], outs[w], pairs) for w in ("B", "C"))
    times = {w: [] for w in ways}
    for _ in range(rounds):
        for w in ways:
            t0 = time.perf_counter()
            run(prof, kind, reads, w)
            times[w].append((time.perf_counter() - t0) * 1e3)
    rec = {"workload": name, "n_reads": n, "n_profiled": prof.n_profiled, "parity_A_B_C": parity,
           "ms_median": {w: statistics.median(t) for w, t in times.items()},
           "ms_range": {w: [min(t), max(t)] for w, t in times.items()},
           "A_over_fwd": statistics.median(times["A"]) / statistics.median(times["fwd"]),
           "stats_A": (run(prof, kind, reads, "A"), prof.last_stats())[1]}
    if kind == "align":
        hit = lambda a: int(((a["status"][:pairs] == _lib.SOME) & (a["score"][:pairs] >= 200)).reshape(n, -1).any(1).sum())
        rec["reads_some_score_ge_200"] = {"forward_only": hit(outs["fwd"]), "both_strands": hit(outs["A"])}
        rec["reverse_strand_pairs"] = int(outs["A"]["strand"][:pairs].sum())
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "both_strands_cfg2_cfg3.json"))
    args = ap.parse_args()
    w25 = WeightMatrix.new_dna_matrix(2, -5, b"N")  # bench.py's scoring: +2 / -5, gap open -10, gap extend -1
    res = {"gpu": gpu_info(), "rounds": args.rounds, "timing": "host clock around each call (host in -> host out)"}
    targets, reads = synth.config2(n_reads=args.n)
    prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], w25, -10, -1, devices=[0])
    res["cfg2_score"] = bench("cfg2", "score", prof, reads, args.rounds)
    prof.close()
    targets, reads = synth.config3(ROOT, n_reads=args.n)
    prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], w25, -10, -1, devices=[0])
    res["cfg3_align"] = bench("cfg3", "align", prof, reads, args.rounds)
    prof.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
