"""Best-hit search against the host-side route to the same answer, timed end to end (host arrays in -> host arrays out)
in one process on one GPU, in alternating rounds, on config 2 (1M x 150 nt reads x 8 segments), forward only and with
both strands:

  align  A  the best-hit align entry point;
         B  the all-pairs align (both strands: align_both_strands), then the selection in numpy and a gather of the
            winners' CIGARs;
  score  A  the best-hit score entry point;
         B  the all-pairs score (both strands: score_both_strands), then the selection in numpy.

Every A/B pair must return identical arrays.  Also reports how many reads are assigned to the segment the generator drew
them from, and, from a separate torch.profiler run, the device time of the best-hit kernels.

    python scripts/bench_best_hit.py [--n 1000000] [--rounds 3] [--out profiles/best_hit_cfg2.json]
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

OUT_KEYS = ("hit", "strand", "score", "status", "tier", "runner_up")
ALIGN_KEYS = ("ref_start", "ref_end", "query_start", "query_end", "hazard")


def rank(status, score):
    return np.where(status == _lib.OVERFLOWED, np.int64(1) << 40, np.where(status == _lib.SOME, score.astype(np.int64) + 1, 0))


def select(a, n, P, strand_of_pair):
    """The best-hit rule on all-pairs outputs (flat, pair index i P + j).  With both strands each pair already holds its
    better strand (ties to forward), so the winner is the first pair of highest rank."""
    st, sc = a["status"][:n * P].reshape(n, P), a["score"][:n * P].reshape(n, P)
    hit = np.argmax(rank(st, sc), axis=1)
    k = np.arange(n) * P + hit
    out = {"hit": hit.astype(np.uint32), "strand": strand_of_pair[k] if strand_of_pair is not None else np.zeros(n, np.uint8),
           "score": a["score"][k], "status": a["status"][k], "tier": a["tier"][k]}
    some_other = (st == _lib.SOME)
    some_other[np.arange(n), hit] = False
    ru = np.where(some_other, sc, 0).max(axis=1)
    out["runner_up"] = np.where(out["status"] == _lib.SOME, ru, 0).astype(np.uint32)
    return out, k


def run(prof, kind, both, reads, way):
    n, P = reads.shape[0], prof.n_profiled
    buf, offs = synth.fixed_len_batch(reads)
    if way == "A":
        if kind == "score":
            return prof.sw_score_best_hit_arrays(buf, offs, both_strands=both)
        return prof.align_best_hit_arrays(buf, offs, both_strands=both)
    if kind == "score":
        res = (prof.sw_score_both_strands_arrays if both else prof.sw_score_arrays)(buf, offs)
        a = dict(zip(("score", "status", "tier", "strand"), (x.ravel() for x in res)))
        return select(a, n, P, a.get("strand"))[0]
    a = (prof.align_both_strands_arrays if both else prof.align_arrays)(buf, offs)
    out, k = select(a, n, P, a.get("strand"))
    some = out["status"] == _lib.SOME
    for key in ALIGN_KEYS:
        out[key] = np.where(some, a[key][k], 0)
    lo = a["cigar_off"][k].astype(np.int64)
    ln = np.where(some, (a["cigar_off"][k + 1] - a["cigar_off"][k]).astype(np.int64), 0)
    off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(ln, out=off[1:])
    src = np.repeat(lo - off[:-1].astype(np.int64), ln) + np.arange(int(off[-1]))
    out["cigar_off"], out["cigar"] = off, a["cigar"][src]
    return out


def same(a, b, n):
    for k in OUT_KEYS + (ALIGN_KEYS + ("cigar_off",) if "cigar_off" in b else ()):
        m = n + 1 if k == "cigar_off" else n
        if not np.array_equal(np.asarray(a[k])[:m], np.asarray(b[k])[:m]):
            return False
    if "cigar" in b:
        t = int(b["cigar_off"][n])
        return np.array_equal(a["cigar"][:t], b["cigar"][:t])
    return True


def bench(prof, reads, which, rounds):
    n = reads.shape[0]
    legs = [(kind, both) for kind in ("align", "score") for both in (False, True)]
    res = {}
    outs = {}
    for kind, both in legs:  # warm-up, and the outputs compared below
        outs[(kind, both)] = {w: run(prof, kind, both, reads, w) for w in ("A", "B")}
    times = {leg: {"A": [], "B": []} for leg in legs}
    for _ in range(rounds):
        for leg in legs:
            for w in ("A", "B"):
                t0 = time.perf_counter()
                run(prof, leg[0], leg[1], reads, w)
                times[leg][w].append((time.perf_counter() - t0) * 1e3)
    for (kind, both) in legs:
        a = outs[(kind, both)]["A"]
        run(prof, kind, both, reads, "A")
        stats = prof.last_stats()
        some = a["status"] == _lib.SOME
        t = times[(kind, both)]
        res[f"{kind}_{'both' if both else 'fwd'}"] = {
            "identical_A_B": same(a, outs[(kind, both)]["B"], n),
            "ms_median": {w: statistics.median(v) for w, v in t.items()},
            "ms_range": {w: [min(v), max(v)] for w, v in t.items()},
            "B_over_A": statistics.median(t["B"]) / statistics.median(t["A"]),
            "reads_some": int(some.sum()),
            "assigned_to_true_segment": int((a["hit"] == which).sum()),
            "assigned_to_true_segment_score_ge_200": [int(((a["hit"] == which) & some & (a["score"] >= 200)).sum()),
                                                      int((some & (a["score"] >= 200)).sum())],
            "reverse_strand_winners": int(a["strand"].sum()),
            "stats_A": stats,
        }
    return res


def kernel_times(prof, reads):
    """Device time per best-hit kernel (and the total) in one both-strand align call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    buf, offs = synth.fixed_len_batch(reads)
    prof.align_best_hit_arrays(buf, offs, both_strands=True)
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        prof.align_best_hit_arrays(buf, offs, both_strands=True)
        torch.cuda.synchronize()
    out, total = {}, 0.0
    for e in p.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        total += us
        if "best_hit" in e.key:
            name = e.key.split("(")[0].replace("void zoe_cuda::", "")
            out[name] = {"ms": us / 1e3, "calls": e.count}
    return {"kernels": out, "all_device_ms": total / 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "best_hit_cfg2.json"))
    args = ap.parse_args()
    w25 = WeightMatrix.new_dna_matrix(2, -5, b"N")  # bench.py's scoring: +2 / -5, gap open -10, gap extend -1
    res = {"gpu": gpu_info(), "rounds": args.rounds, "timing": "host clock around each call (host in -> host out)"}
    targets, reads = synth.config2(n_reads=args.n)
    which = np.random.default_rng(3).integers(0, len(targets), args.n)  # illumina_reads' first draw (5 % become random)
    prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], w25, -10, -1, devices=[0])
    res["cfg2"] = bench(prof, reads, which, args.rounds)
    res["cfg2_profiler_align_both"] = kernel_times(prof, reads)
    prof.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
