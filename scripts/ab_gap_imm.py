"""A/B of the score kernels with the gap penalties compiled in (GapImm) against the run-time-penalty kernels (GapRt), in
one process on one GPU: two contexts over the same staged batch, one created with ZOE_CUDA_NO_GAP_IMM set; both are
warmed up, then timed in alternating rounds with CUDA events on the library stream; their score / status / tier arrays
must be identical.  ZOE_CUDA_LIB=<path> loads another build of the library (e.g. the other form of the "- go" step).

    python scripts/ab_gap_imm.py [--n 1000000] [--rounds 7] [--steps 5] [--warmup 3] [--out profiles/ab_gap_imm_cfg2.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import zoe_b200._lib as L  # noqa: E402
from zoe_b200 import CudaProfiles, WeightMatrix, synth  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))


def make_ctx(targets, no_imm: bool):
    if no_imm:
        os.environ["ZOE_CUDA_NO_GAP_IMM"] = "1"
    else:
        os.environ.pop("ZOE_CUDA_NO_GAP_IMM", None)
    try:
        # the scoring of bench.py's config 2: DNA +2 / -5, gap open -10, gap extend -1
        return CudaProfiles.new_with_w256([bytes(t) for t in targets], WeightMatrix.new_dna_matrix(2, -5, b"N"), -10, -1,
                                          devices=[0])
    finally:
        os.environ.pop("ZOE_CUDA_NO_GAP_IMM", None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ab_gap_imm_cfg2.json"))
    args = ap.parse_args()
    if args.rounds < 5:
        ap.error("--rounds must be at least 5")

    targets, reads = synth.config2(n_reads=args.n, seed_reads=3)
    buf, offs = synth.fixed_len_batch(reads)
    cells = int(offs[-1]) * sum(len(t) for t in targets)
    variants = {"imm": make_ctx(targets, False), "rt": make_ctx(targets, True)}
    streams = {}
    for name, prof in variants.items():
        prof.stage(buf, offs)
        streams[name] = torch.cuda.ExternalStream(prof.stream_handle(0), device=0)
    info_before = gpu_info()

    for name, prof in variants.items():
        for _ in range(args.warmup):
            prof.run_score_staged()
        torch.cuda.synchronize()
    outs = {name: prof.fetch_scores() for name, prof in variants.items()}
    for a, b, what in zip(outs["imm"], outs["rt"], ("score", "status", "tier")):
        assert np.array_equal(a, b), f"{what} differs between the two variants"

    ms = {name: [] for name in variants}
    for r in range(args.rounds):
        for name in (("imm", "rt") if r % 2 == 0 else ("rt", "imm")):
            prof = variants[name]
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(streams[name])
            for _ in range(args.steps):
                prof.run_score_staged()
            ev1.record(streams[name])
            ev1.synchronize()
            ms[name].append(ev0.elapsed_time(ev1) / args.steps)
    info_after = gpu_info()
    outs2 = {name: prof.fetch_scores() for name, prof in variants.items()}
    for name in variants:
        for a, b in zip(outs[name], outs2[name]):
            assert np.array_equal(a, b), f"{name}: results changed between the warm-up and the timed rounds"
    launches = {name: prof.last_timing()["kernel_launches"] for name, prof in variants.items()}
    for prof in variants.values():
        prof.close()

    summary = {name: {"min_ms": min(v), "median_ms": statistics.median(v), "max_ms": max(v),
                      "gcups_at_median": cells / (statistics.median(v) * 1e-3) / 1e9, "ms_per_step": v,
                      "launches_per_step": launches[name]} for name, v in ms.items()}
    rec = {
        "workload": f"cfg2: {args.n} x 150nt reads vs 8 flu-A-length segments, score-only (synth.config2 seed_reads=3), "
                    "DNA +2/-5, gap open 10, extend 1",
        "library": os.path.relpath(L.LIB_PATH, ROOT),
        "variants": {"imm": "gap penalties compiled in (GapImm<10,1>)", "rt": "ZOE_CUDA_NO_GAP_IMM: penalties from ScoreParams"},
        "rounds": args.rounds, "steps_per_round": args.steps, "warmup": args.warmup, "order": "imm, rt in even rounds; rt, imm in odd rounds",
        "results_identical": True,
        "median_gain": summary["rt"]["median_ms"] / summary["imm"]["median_ms"] - 1.0,
        "gpu_before": info_before, "gpu_after": info_after,
        **summary,
    }
    for name in ("imm", "rt"):
        s = summary[name]
        print(f"{name:4s} ms/step min {s['min_ms']:.2f} median {s['median_ms']:.2f} max {s['max_ms']:.2f} "
              f"({s['gcups_at_median']:.0f} GCUPS)")
    print(f"median gain {100 * rec['median_gain']:+.2f} %  gpu {info_before}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
