#!/usr/bin/env python
"""bench.py -- SW GCUPS of the B200 path on BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2] [--mode M] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input.  The headline workload is BASELINE.json
configs[1]: ONE fixed set of 1M x 150-nt reads (seed 3) vs 8 influenza-A-length segments, score only (2.04e12 cells per
step).  With N GPUs (one process per GPU under torchrun) rank r scores the contiguous shard
``zoe_b200.dist.shard_range(1_000_000, r, N)`` of that same set -- "scaling": "strong"; no collective on the data path;
the per-rank result checksums are summed (off the clock) and must equal the N = 1 checksum.

`value`  = whole-job GCUPS with the shard already resident in HBM (CUDA events on the library's stream, max over ranks).
`e2e`    = whole-job GCUPS through the host-buffer C-ABI call (pinned host -> device copies and the device -> host
           result copies inside the timed region, max over ranks).
`legs`   = the other half of the metric and the other configurations, timed by the same code in the same run:
           "align" (cfg 3: zoe_cuda_sw_align_batch, device traceback + CIGARs; at N = 1 checked pair by pair against the
           vectorised CPU restatement of sw_simd_align on the WHOLE set), and at N = 1 also "cfg1", "cfg4" (a stated
           slice), "cfg4_3pass" (CIGARs for the long reads), "align_tieheavy" (a scoring that sends 6.7 % of the pairs
           through the literal striped kernels), "cfg5".  `--legs none` skips them, `--config C` benches one alone.
`--impl reference` times the CPU restatement of zoe's striped path (oracle/zoe_sw_cpu.cpp) on all host threads; zoe
itself (Rust nightly) cannot be built in this image.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "sw_gcups"
UNIT = "GCUPS"
DPX_INSTR_PER_CELL = 2.25  # 4.5 DPX/ALU instructions per packed cell pair (DESIGN.md "score kernel")

# Result checksums of the default workloads at N = 1 (sum of scores [+ ranges + CIGAR words], mod 2^64).  A sharded
# run must reproduce them: the results do not depend on how the reads are split over GPUs.
EXPECTED_CHECKSUM = {("cfg2", "score", 1_000_000): 268486591, ("cfg3", "align", 1_000_000): 4405153473,
                     ("cfg5", "score", 1_000_000): 767435248, ("cfg1", "score", 10_000): 1466752,
                     ("cfg4", "score", 20_000): 23653328}
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much


def dump_outputs(out_dir: str, outs: dict, n: int, n_prof: int, mode: str):
    """Writes the result arrays of the last timed step as float64 ``out_dir/<name>.npy``: one value per pair (pair =
    read * n_prof + profiled sequence), and in the CIGAR modes ``cigar_len`` (words per pair) and the pairs' ``cigar``
    words back to back.  When that exceeds DUMP_BYTES a seeded sample of reads is written; ``read_index`` lists the
    reads kept.  The sample depends only on n and n_prof, so two builds of the project dump the same pairs.  CIGAR words
    past the size limit are cut off."""
    per_pair = ["score", "status", "tier"]
    if mode != "score":
        per_pair += ["ref_start", "ref_end", "query_start", "query_end"]
    if mode == "align":
        per_pair.append("hazard")
    has_cigar = "cigar" in outs
    limit = DUMP_BYTES - 4096  # room for the .npy headers
    row_bytes = 8 * (1 + n_prof * (len(per_pair) + has_cigar))
    k = min(n, (limit // 2 if has_cigar else limit) // row_bytes)
    rows = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    pairs = (rows[:, None] * n_prof + np.arange(n_prof)[None, :]).reshape(-1)
    arrays = {"read_index": rows}
    arrays.update({name: outs[name][pairs] for name in per_pair})
    if has_cigar:
        lo = outs["cigar_off"][pairs].astype(np.int64)
        lens = outs["cigar_off"][pairs + 1].astype(np.int64) - lo
        arrays["cigar_len"] = lens
        words = np.repeat(lo - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
        arrays["cigar"] = outs["cigar"][words[: (limit - 8 * sum(a.size for a in arrays.values())) // 8]]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


SCORING = None  # --scoring match,mismatch,gap_open,gap_extend (DNA configurations): e.g. 4,-2,-3,-1 = tie-heavy


def make_workload(config: int, n_override: int | None):
    """Returns (key, name, matrix, gap_open, gap_extend, targets, (buf, offs), mode).  The data depend on the
    configuration only -- never on the rank: every rank generates the same set and takes its shard of it."""
    w = _make_workload(config, n_override)
    if SCORING and config != 5:
        from zoe_b200 import WeightMatrix
        ma, mi, go, ge = SCORING
        key, name, _, _, _, t, batch, mode = w
        return (key + f"/scoring{ma},{mi},{go},{ge}", name + f" [scoring match {ma} mismatch {mi} open {go} extend {ge}]",
                WeightMatrix.new_dna_matrix(ma, mi, b"N"), go, ge, t, batch, mode)
    return w


def _make_workload(config: int, n_override: int | None):
    from zoe_b200 import BLOSUM_62, WeightMatrix, synth

    dna = WeightMatrix.new_dna_matrix(2, -5, b"N")
    if config == 1:
        n = n_override or 10_000
        t, r = synth.config1(ROOT, n_reads=n, seed=1)
        return ("cfg1", f"cfg1: {n} x 150nt reads vs 1704nt HA, score", dna, -10, -1, t, synth.fixed_len_batch(r), "score")
    if config == 2:
        n = n_override or 1_000_000
        t, r = synth.config2(n_reads=n, seed_reads=3)
        return ("cfg2", f"cfg2: {n} x 150nt reads vs 8 flu-A-length segments (13588nt), score-only", dna, -10, -1, t,
                synth.fixed_len_batch(r), "score")
    if config == 3:
        n = n_override or 1_000_000
        t, r = synth.config3(ROOT, n_reads=n, seed=4)
        return ("cfg3", f"cfg3: {n} x 150nt reads vs 1704nt HA, align with traceback", dna, -10, -1, t,
                synth.fixed_len_batch(r), "align")
    if config == 4:
        n = n_override or 100_000
        t, r = synth.config4(n_reads=n, seed_reads=6)
        return ("cfg4", f"cfg4: {n} x 1-5kb ONT-like reads vs 29903nt genome, score-only (long-row path)", dna, -10, -1, t,
                synth.pack(r), "score")
    if config == 5:
        n = n_override or 1_000_000
        t, q = synth.config5(n_queries=n, seed_queries=8)
        return ("cfg5", f"cfg5: {n} x 300aa queries vs 566aa target, BLOSUM62, score-only", BLOSUM_62, -10, -1, t,
                synth.fixed_len_batch(q), "score")
    raise SystemExit(f"config {config} is not a bench workload")


def shared_config(name: str, n_total: int, n_prof: int, mode: str, in_bytes: int):
    """The `config` object, identical in both arms (b200 / reference) for the same command line."""
    return {
        "workload": name, "sequences": n_total, "profiled": n_prof, "mode": mode,
        "sharding": "one fixed set; rank r takes the contiguous index range shard_range(n, r, n_gpus); no collective",
        "l2": ("inputs_exceed_l2" if in_bytes > 126e6 else
               "inputs_smaller_than_l2 (ALU-bound kernel; every sequence byte is read once per step)"),
        "orientation": "profile = reference side, reads streamed (SeqSrc::Query)", "lanes": "w256",
        "reference_arm_sample": "the CPU arm times a bounded prefix of this workload per step (GCUPS is a rate)",
    }


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")] + [time.time()])

    def window(self, t0: float, t1: float):
        """Keep only the samples taken inside [t0, t1] (the sampler is started before the warm-up so that the
        start-up cost of nvidia-smi -- tens of ms of driver lock -- never lands inside the timed region)."""
        rows = [r for r in self.rows if t0 <= r[-1] <= t1]
        if rows:
            self.rows = rows

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.rows = [r[:-1] for r in self.rows]
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU side (oracle/): the reported baseline and the parity checker.  Never inside a timed GPU region.
# ------------------------------------------------------------------------------------------------------------------
def cpu_port_run(matrix, go, ge, targets, buf, offs, n_sample, threads, width_bits=256):
    from oracle import cpu_baseline as CB
    from zoe_b200 import synth

    pbuf, poff = synth.pack([np.asarray(t, dtype=np.uint8) for t in targets])
    o = offs[: n_sample + 1]
    t0 = time.perf_counter()
    res = CB.score_batch(pbuf, poff, buf[: int(o[-1])], o, matrix.weights, matrix.mapping.index_map, go, ge,
                         width_bits=width_bits, n_threads=threads)
    dt = time.perf_counter() - t0
    cells = int(o[-1]) * int(poff[-1])
    return cells / dt / 1e9, dt, res


def cpu_align_run(matrix, go, ge, targets, buf, offs, n_sample, threads, width_bits=256):
    from oracle import cpu_baseline as CB
    from zoe_b200 import synth

    pbuf, poff = synth.pack([np.asarray(t, dtype=np.uint8) for t in targets])
    o = offs[: n_sample + 1]
    t0 = time.perf_counter()
    res = CB.align_batch(pbuf, poff, buf[: int(o[-1])], o, matrix.weights, matrix.mapping.index_map, go, ge,
                         width_bits=width_bits, n_threads=threads, streamed_is_query=True)
    dt = time.perf_counter() - t0
    cells = int(o[-1]) * int(poff[-1])
    return cells / dt / 1e9, dt, res


def run_threaded(check_range, n_items):
    """Runs ``check_range(lo, hi) -> mismatches`` over [0, n_items) on all host threads (the oracle is called through
    ctypes, which releases the GIL).  Returns (total mismatches, threads used)."""
    from concurrent.futures import ThreadPoolExecutor
    threads = max(1, min(os.cpu_count() or 1, 64))
    step = max(1, (n_items + 8 * threads - 1) // (8 * threads))
    spans = [(lo, min(lo + step, n_items)) for lo in range(0, n_items, step)]
    with ThreadPoolExecutor(max_workers=threads) as ex:
        return sum(ex.map(lambda sp: check_range(*sp), spans)), threads


def sized_sample(n_total, probe_fn, seconds):
    """Largest prefix of the workload the CPU port gets through in about `seconds` (probe: 2000 sequences)."""
    probe = min(n_total, 2000)
    _, dt0, _ = probe_fn(probe)
    return int(min(n_total, max(probe, probe * seconds / max(dt0, 1e-3))))


def run_reference(args):
    """`--impl reference`: the CPU restatement on all host threads, rank 0 only."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from oracle import cpu_baseline as CB

    key, name, matrix, go, ge, targets, (buf, offs), mode = make_workload(args.config, args.n)
    if args.mode:
        mode = args.mode
        name += f" [mode {mode}]"
    threads = CB.hardware_threads()
    n_total = len(offs) - 1
    n_prof = len(targets)
    align = mode in ("align", "3pass", "ranges")
    runner = cpu_align_run if align else cpu_port_run
    # a bounded sample: ~4 s of CPU work per step
    n_sample = sized_sample(n_total, lambda k: runner(matrix, go, ge, targets, buf, offs, k, threads), 4.0)
    for _ in range(args.warmup):
        runner(matrix, go, ge, targets, buf, offs, min(n_sample, 2000), threads)
    times = []
    for _ in range(args.steps):
        g, dt, _ = runner(matrix, go, ge, targets, buf, offs, n_sample, threads)
        times.append(dt)
    prof_total = sum(len(t) for t in targets)
    cells = int(offs[n_sample]) * prof_total
    value = cells * len(times) / sum(times) / 1e9
    what = ("sw_simd_align + to_alignment + invert" if align else "sw_simd_score") + " + i8->i16->i32 escalation"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "i8/i16/i32 (zoe tiers, w256 lanes)", "data": "synthetic",
        "config": shared_config(name, n_total, n_prof, mode, int(buf.nbytes + offs.nbytes)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"first {n_sample} sequences x {prof_total} profiled residues per step, {CB.isa()}, "
                                   f"C++ restatement of zoe's striped {what} "
                                   "(zoe itself needs nightly Rust: not buildable here)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# one leg = one configuration + mode, timed device-resident and end to end on this rank's shard
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide state of a bench run (ranks, barrier, reductions from zoe_b200.dist)."""

    def __init__(self, args):
        import torch
        from zoe_b200 import dist as zdist

        self.torch = torch
        self.zdist = zdist
        self.rank, self.world, self.local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        self.distributed = self.world > 1
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: zoe_b200 has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dist = None
        if self.distributed:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist
        self.in_process_devices = args.gpus if (not self.distributed and args.gpus > 1) else 1
        self.n_gpus = self.world if self.distributed else self.in_process_devices
        self.device = torch.device("cuda", self.local_rank)

    def barrier(self):
        if self.distributed:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        return self.zdist.max_over_ranks(x, device=self.device)

    def sum_over_ranks(self, x: float) -> float:
        return self.zdist.sum_over_ranks(x, device=self.device)

    def sum_u64_over_ranks(self, x: int) -> int:
        return self.zdist.sum_u64_over_ranks(x, device=self.device)


def pinned(torch, arr: np.ndarray):
    t = torch.from_numpy(arr).pin_memory()
    return t, t.numpy()


def run_leg(ctx: Ctx, config: int, mode_override, n_override, steps: int, warmup: int, cpu: bool, cpu_seconds: float,
            align_opts=None, sample_clocks: bool = False, full_parity: bool = True, scoring=None, dump_dir=None):
    """Times one configuration on this rank's shard; returns the record rank 0 prints (None on the other ranks).
    ``dump_dir``: rank 0 writes its shard's results of the last timed step there (dump_outputs)."""
    from zoe_b200 import CudaProfiles

    torch = ctx.torch
    global SCORING
    saved_scoring = SCORING
    if scoring is not None:
        SCORING = scoring
    try:
        key, name, matrix, go, ge, targets, (buf_all, offs_all), mode = make_workload(config, n_override)
    finally:
        SCORING = saved_scoring
    tie_heavy = scoring is not None or SCORING is not None
    if mode_override:
        mode = mode_override
        name += f" [mode {mode}]"
    n_total = len(offs_all) - 1
    n_prof = len(targets)
    prof_total = sum(len(t) for t in targets)
    total_cells = int(offs_all[-1]) * prof_total

    # ---- this rank's shard: contiguous index range of the one fixed set ----
    # (an in-process multi-device context shards inside the library by the same rule)
    _, buf, offs = ctx.zdist.shard_batch(buf_all, offs_all, ctx.rank if ctx.distributed else 0,
                                         ctx.world if ctx.distributed else 1)
    n = len(offs) - 1
    pairs = n * n_prof

    if ctx.in_process_devices > 1:
        prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], matrix, go, ge, n_devices=ctx.in_process_devices)
    else:
        prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], matrix, go, ge, devices=[ctx.local_rank])
    if align_opts:
        prof.set_align_options(*[int(x) for x in align_opts.split(",")])

    # pinned host buffers for the end-to-end leg
    t_buf, h_buf = pinned(torch, buf)
    t_offs, h_offs_i = pinned(torch, offs.view(np.int64))
    h_offs = h_offs_i.view(np.uint64)
    keep = [t_buf, t_offs]
    outs = {}
    for k in ("score", "ref_start", "ref_end", "query_start", "query_end"):
        if k == "score" or mode != "score":
            t, a = pinned(torch, np.zeros(max(pairs, 1), dtype=np.int32))
            keep.append(t)
            outs[k] = a.view(np.uint32)
    for k in ("status", "tier", "hazard"):
        if k != "hazard" or mode in ("align", "3pass"):
            t, a = pinned(torch, np.zeros(max(pairs, 1), dtype=np.uint8))
            keep.append(t)
            outs[k] = a
    if mode in ("align", "3pass"):
        # CIGAR words: <= 5 per short read; cheap gaps fragment them; long noisy reads need ~1 word per 15 bases
        cap = pairs * (64 if tie_heavy else 8) + int(offs[-1]) * n_prof // 6 + 1024
        t, a = pinned(torch, np.zeros(pairs + 1, dtype=np.int64))
        keep.append(t)
        outs["cigar_off"] = a.view(np.uint64)
        t, a = pinned(torch, np.zeros(cap, dtype=np.int32))
        keep.append(t)
        outs["cigar"] = a.view(np.uint32)

    stream = torch.cuda.ExternalStream(prof.stream_handle(0), device=ctx.device)
    run_staged = {"score": prof.run_score_staged, "align": prof.run_align_staged, "ranges": prof.run_ranges_staged,
                  "3pass": prof.run_3pass_staged}[mode]

    def e2e_call():
        if mode == "score":
            prof.sw_score_into(h_buf, h_offs, outs["score"], outs["status"], outs["tier"])
        elif mode == "ranges":
            prof.ranges_into(h_buf, h_offs, outs)
        else:
            prof.align_into(h_buf, h_offs, outs, three_pass=(mode == "3pass"))

    # ---------------- device-resident leg (`value`) ----------------
    prof.stage(h_buf, h_offs)
    sampler = ClockSampler(ctx.local_rank) if (sample_clocks and ctx.rank == 0) else None
    if sampler:
        sampler.start()
    for _ in range(warmup):
        run_staged()
    ctx.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dp_ms, launches = [], 0
    t_region0 = time.time()
    ev0.record(stream)
    for _ in range(steps):
        run_staged()
        tm = prof.last_timing()
        dp_ms.append(tm["dp_kernel_ms"])
        launches += tm["kernel_launches"]
    ev1.record(stream)
    ctx.barrier()
    if sampler:
        sampler.window(t_region0, time.time())
    clocks = sampler.stop() if sampler else None
    dev_ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    stats = prof.last_stats()
    value = total_cells * steps / (dev_ms * 1e-3) / 1e9

    # ---------------- end-to-end leg (`e2e`): host buffers in, host results out ----------------
    for _ in range(min(warmup, 2)):
        e2e_call()
    ctx.barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev2.record(stream)
    for _ in range(steps):
        e2e_call()
        launches += prof.last_timing()["kernel_launches"]
    ev3.record(stream)
    ctx.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = ctx.max_over_ranks(max(ev2.elapsed_time(ev3), wall_ms))
    e2e_stats = prof.last_stats()
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, outs, n, n_prof, mode)
    n_words = int(outs["cigar_off"][pairs]) if mode in ("align", "3pass") else 0
    d2h = {"score": pairs * 6, "ranges": pairs * 22}.get(mode, pairs * (5 * 4 + 3 + 8) + 8 + n_words * 4)
    # additive checksum: the per-rank values sum to the N = 1 value
    checksum = int(outs["score"][:pairs].sum(dtype=np.uint64))
    if mode != "score":
        for k in ("ref_start", "ref_end", "query_start", "query_end"):
            checksum += int(outs[k][:pairs].sum(dtype=np.uint64))
    if n_words:
        checksum += int(outs["cigar"][:n_words].sum(dtype=np.uint64))
    checksum = ctx.sum_u64_over_ranks(checksum & 0xFFFFFFFFFFFFFFFF)
    want = EXPECTED_CHECKSUM.get((key, mode, n_total))
    e2e = {"value": total_cells * steps / (e2e_ms * 1e-3) / 1e9, "unit": UNIT,
           "h2d_bytes_per_step": int(ctx.sum_over_ranks(float(h_buf.nbytes + h_offs.nbytes))),
           "d2h_bytes_per_step": int(ctx.sum_over_ranks(float(d2h))),
           "ms_per_step": e2e_ms / steps, "result_checksum": checksum,
           "checksum_expected_n1": want, "checksum_matches_n1": (checksum == want) if want is not None else None}

    # ---------------- roofline of the dominant kernel (this rank's launches) ----------------
    dpx_g, _ = prof.dpx_peak(0)  # G lane-instr/s, measured live on this GPU
    peak_gcups = dpx_g / DPX_INSTR_PER_CELL
    cells_rank = int(offs[-1]) * prof_total
    dp_mean = float(np.mean(dp_ms)) if dp_ms and np.mean(dp_ms) > 0 else float("nan")
    kernel_gcups = cells_rank / (dp_mean * 1e-3) / 1e9
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    in_bytes = float(h_buf.nbytes + h_offs.nbytes + pairs * 4)
    maxlen = int(np.max(np.diff(offs.astype(np.int64)))) if n else 0
    if mode == "score":
        if matrix.S > 8 and max(len(t) for t in targets) <= 1024 and 64 <= maxlen <= 1024:
            kname, instr = "sw_score_rows_stream_kernel (profiled sequence in registers, shared table)", "4.5 ALU + 2 FMA-pipe"
        elif maxlen > 1024:
            kname, instr = "sw_score_long_kernel (chunked rows, boundary rows through L2)", "4.5 ALU + 1 FMA-pipe"
        else:
            kname, instr = "sw_score_kernel (two column streams, ping-pong register sets)", "4.5 ALU + 1 FMA-pipe"
        frac_of = "the kernel alone"
    elif mode in ("ranges", "3pass"):
        kname = "sw_align_scan_kernel forward (+ pin sweep) and its REV instantiation (score + end / start cell, no traceback matrix)"
        instr = "4.5 ALU + 1 FMA-pipe per cell pair plus per-column bookkeeping; the reverse pass covers the truncated matrix"
        if mode == "3pass":
            kname += "; pass 3 = tp_classify / tp_dp kernels (no-gaps shortcut, banded box alignment)"
        frac_of = "all DP kernels of the step (forward scan, pin sweep, reverse scan)"
    else:
        kname = "sw_align_scan_kernel + sw_align_winfill_kernel (checkpointed window; DESIGN.md 4.3)"
        instr = "4.5 ALU per cell pair in the scan, 9.5 ALU + 11 FMA-pipe in the window fill"
        ck = (n / 2) * sum((len(t) - 1) // 64 for t in targets) * 40 * 8 * 4
        fl = (pairs / 2) * 216 * 8 * 8 * 4
        in_bytes += float(ck + fl)
        frac_of = "the DP kernels of the step (scan + pin + window fill), not the whole pipeline -- see `frac_step`"
    traffic, traffic_source = None, None
    try:  # measured DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(f"cfg{config}/{mode}")
        if tr and n_override is None and ctx.n_gpus == 1:
            traffic, traffic_source = tr["dram_read_bytes"] + tr["dram_write_bytes"], tr["source"]
    except Exception:
        pass
    roofline = {
        "bound": "alu", "achieved": kernel_gcups, "peak": peak_gcups, "unit": "GCUPS", "frac": kernel_gcups / peak_gcups,
        "frac_of": frac_of, "frac_step": value / ctx.n_gpus / peak_gcups,
        "traffic": traffic, "traffic_source": traffic_source,
        "note": ("integer max-plus (DPX on the ALU pipe) bound, not hbm/tensor: peak = live-measured "
                 "VIADDMNMX.S16x2 issue rate (%.0f G lane-instr/s) / %.2f ALU instr per cell (4.5 per packed s16x2 cell "
                 "pair: the score recurrence); kernel = %s, %s per cell pair; avg of %d steps on rank 0's shard, CUDA events "
                 "on the library stream" % (dpx_g, DPX_INSTR_PER_CELL, kname, instr, len(dp_ms))),
        "hbm": {"algorithmic_bytes_per_launch": in_bytes, "achieved_gbs": in_bytes / (dp_mean * 1e-3) / 1e9,
                "peak_gbs": hbm_peak, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                "frac": in_bytes / (dp_mean * 1e-3) / 1e9 / hbm_peak},
    }

    # ---------------- CPU baseline + parity (rank 0, N = 1 only) ----------------
    cpu_rec, parity = None, None
    if cpu and ctx.rank == 0 and ctx.n_gpus == 1:
        from oracle import cpu_baseline as CB
        threads = CB.hardware_threads()
        if mode == "score":
            full = full_parity and total_cells <= 4e11  # cfg 1 / 5: the whole set (SURVEY 8(d)); cfg 2 / 4: a sample
            n_sample = n if full else sized_sample(
                n, lambda k: cpu_port_run(matrix, go, ge, targets, buf, offs, k, threads), cpu_seconds)
            g, dt, (c_score, c_status, c_tier) = cpu_port_run(matrix, go, ge, targets, buf, offs, n_sample, threads)
            lazy, rows = CB.last_lazy_stats()
            cpu_rec = {"value": g, "unit": UNIT, "cores": threads, "kind": "port",
                       "sample": f"first {n_sample} of {n} sequences x all {n_prof} profiled ({dt:.1f} s, {CB.isa()}, w256 "
                                 f"lanes i8x32/i16x16/i32x8; lazy-F revisits {lazy / max(rows, 1):.1f} vectors per DP row)"}
            g_score = outs["score"].reshape(n, n_prof)[:n_sample]
            g_status = outs["status"].reshape(n, n_prof)[:n_sample]
            g_tier = outs["tier"].reshape(n, n_prof)[:n_sample]
            some = c_status == 0
            mism = int((g_status != c_status).sum() + (g_score[some] != c_score[some]).sum()
                       + (g_tier[some] != c_tier[some]).sum())
            parity = {"checked_pairs": int(n_sample * n_prof), "of_pairs": pairs, "mismatches": mism,
                      "against": "vectorised CPU port of sw_simd_score (oracle/zoe_sw_cpu.cpp)"}
        elif mode == "align":
            n_sample = n if full_parity else sized_sample(
                n, lambda k: cpu_align_run(matrix, go, ge, targets, buf, offs, k, threads), cpu_seconds)
            g, dt, want_res = cpu_align_run(matrix, go, ge, targets, buf, offs, n_sample, threads)
            t1 = time.perf_counter()
            mism = CB.compare_alignments(outs, want_res, n_sample * n_prof)
            cpu_rec = {"value": g, "unit": UNIT, "cores": threads, "kind": "port",
                       "sample": f"first {n_sample} of {n} sequences ({dt:.1f} s, {CB.isa()}, w256 lanes): vectorised C++ "
                                 "restatement of sw_simd_align + to_alignment + invert + i8->i16->i32 escalation"}
            parity = {"checked_pairs": int(n_sample * n_prof), "of_pairs": pairs, "mismatches": mism,
                      "compare_s": round(time.perf_counter() - t1, 2),
                      "against": "vectorised CPU port of sw_simd_align (oracle/zoe_sw_cpu.cpp; itself pinned to "
                                 "oracle/zoe_sw_oracle.c in tests/): status, score, tier, ranges, CIGAR"}
        else:  # ranges / 3pass: the plain-C oracle on a sample
            from oracle import oracle as O
            sc = O.Scoring(matrix.weights, matrix.mapping.index_map, go, ge)
            # the scalar-loop oracle does ~1 GCUPS on 16 threads: a prefix of at most 20000 sequences and ~2e10 cells
            cum = np.cumsum(np.diff(offs.astype(np.int64))) * prof_total
            n_sample = int(min(n, 20000, max(1, np.searchsorted(cum, 2e10) + 1)))
            t0 = time.perf_counter()

            def check_range(lo_, hi_):
                bad = 0
                for i in range(lo_, hi_):
                    s_i = bytes(buf[int(offs[i]):int(offs[i + 1])])
                    for j, tg in enumerate(targets):
                        k = i * n_prof + j
                        if mode == "3pass":
                            rc, w, _, _ = O.sw_align_3pass_from(bytes(tg), s_i, sc, streamed_is_query=True)
                            ok = int(outs["status"][k]) == rc
                            if ok and rc == 0:
                                lo_w, hi_w = int(outs["cigar_off"][k]), int(outs["cigar_off"][k + 1])
                                cig = "".join(f"{int(x) >> 4}{'MID?S'[int(x) & 15]}" for x in outs["cigar"][lo_w:hi_w])
                                ok = (int(outs["score"][k]), int(outs["ref_start"][k]), int(outs["ref_end"][k]),
                                      int(outs["query_start"][k]), int(outs["query_end"][k]), cig) == \
                                     (w.score, w.ref_range[0], w.ref_range[1], w.query_range[0], w.query_range[1], w.cigar)
                        else:
                            rc, score, rr, qr, _ = O.sw_score_ranges_from(bytes(tg), s_i, sc, streamed_is_query=True)
                            ok = int(outs["status"][k]) == rc
                            if ok and rc == 0:
                                ok = (int(outs["score"][k]), int(outs["ref_start"][k]), int(outs["ref_end"][k]),
                                      int(outs["query_start"][k]), int(outs["query_end"][k])) == (score, rr[0], rr[1], qr[0], qr[1])
                        bad += 0 if ok else 1
                return bad

            mism, oracle_threads = run_threaded(check_range, n_sample)
            dt = time.perf_counter() - t0
            cpu_rec = {"value": int(offs[n_sample]) * prof_total / dt / 1e9, "unit": UNIT, "cores": oracle_threads,
                       "kind": "port",
                       "sample": f"first {n_sample} sequences, plain-C scalar-loop oracle of "
                                 f"{'sw_align_3pass' if mode == '3pass' else 'sw_simd_score_ranges'} + escalation ({dt:.1f} s); "
                                 "not vectorised -- a checker, not a tuned baseline"}
            parity = {"checked_pairs": n_sample * n_prof, "of_pairs": pairs, "mismatches": mism,
                      "against": "oracle/zoe_sw_oracle.c"}

    rec = None
    if ctx.rank == 0:
        rec = {
            "value": value, "unit": UNIT, "ms_per_step": dev_ms / steps, "steps": steps, "warmup": warmup,
            "config": shared_config(name, n_total, n_prof, mode, int(buf_all.nbytes + offs_all.nbytes)),
            "sequences_per_rank": n, "cells_per_step": total_cells,
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu_rec, "parity": parity, "tiers": stats,
            "hazard_pairs": int(e2e_stats.get("hazard", 0)),
        }
    prof.close()
    del keep
    return rec


def sneaky_leg(ctx: Ctx, cpu: bool, n: int = 1_000_000, threshold: float = 0.1):
    """SURVEY 8(f).4: the SneakySnake pre-alignment filter on 1M (150-nt window, 150-nt read) pairs -- an HBM-light
    byte-compare kernel, reported in pairs/s with the bytes it has to move against the measured HBM peak."""
    from zoe_b200 import SneakySnake

    torch = ctx.torch
    rng = np.random.default_rng(9)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    refs = acgt[rng.integers(0, 4, (n, 150))]
    qs = refs.copy()
    nerr = rng.integers(0, 30, n)  # 0..29 substitutions per read: both outcomes occur at threshold 0.1 (15 edits)
    pos = rng.integers(0, 150, (n, 30))
    mask = np.arange(30)[None, :] < nerr[:, None]
    rows = np.repeat(np.arange(n), 30).reshape(n, 30)[mask]
    qs[rows, pos[mask]] = acgt[rng.integers(0, 4, int(mask.sum()))]
    offs = (np.arange(n + 1, dtype=np.uint64) * np.uint64(150)).astype(np.uint64)
    t_r, h_r = pinned(torch, np.ascontiguousarray(refs.reshape(-1)))
    t_q, h_q = pinned(torch, np.ascontiguousarray(qs.reshape(-1)))
    snake = SneakySnake()
    for _ in range(2):
        out = snake.filter_arrays(h_r, offs, h_q, offs, threshold)
    tot, ker = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        out = snake.filter_arrays(h_r, offs, h_q, offs, threshold)
        wall = (time.perf_counter() - t0) * 1e3
        a, b = snake.last_timing()
        tot.append(max(a, wall))
        ker.append(b)
    snake.close()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    bytes_moved = float(h_r.nbytes + h_q.nbytes + 2 * offs.nbytes + n)
    k_ms, e_ms = float(np.mean(ker)), float(np.mean(tot))
    rec = {"workload": f"{n} pairs of (150-nt window, 150-nt read with 0-29 substitutions), threshold {threshold}",
           "value": n / (k_ms * 1e-3) / 1e6, "unit": "Mpairs/s", "ms_per_step": k_ms,
           "e2e": {"value": n / (e_ms * 1e-3) / 1e6, "unit": "Mpairs/s", "ms_per_step": e_ms,
                   "h2d_bytes_per_step": int(h_r.nbytes + h_q.nbytes + 2 * offs.nbytes), "d2h_bytes_per_step": n},
           "roofline": {"bound": "hbm", "achieved": bytes_moved / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": bytes_moved / (k_ms * 1e-3) / 1e9 / hbm_peak,
                        "note": "algorithmic bytes = both sequences + offsets + 1 result byte per pair, each read once; the "
                                "kernel is a chain of dependent byte compares per pair (latency, not bandwidth, bound)"},
           "outcomes": {"some_true": int((out == 1).sum()), "some_false": int((out == 0).sum()), "none": int((out == 2).sum())}}
    if cpu:
        from oracle import oracle as O
        m = 20000
        t0 = time.perf_counter()
        want = [O.sneaky_snake(bytes(refs[i]), bytes(qs[i]), threshold) for i in range(m)]
        dt = time.perf_counter() - t0
        code = {False: 0, True: 1, None: 2}
        mism = int(sum(1 for i in range(m) if code[want[i]] != int(out[i])))
        rec["parity"] = {"checked_pairs": m, "of_pairs": n, "mismatches": mism, "against": "oracle/zoe_sw_oracle.c zo_sneaky_snake"}
        rec["cpu_baseline"] = {"value": m / dt / 1e6, "unit": "Mpairs/s", "cores": 1, "kind": "port",
                               "sample": f"first {m} pairs, plain-C restatement called pair by pair through ctypes ({dt:.1f} s)"}
    return rec


def compact(rec):
    """An extra leg's record inside the headline line: the same keys, minus the long prose."""
    if rec is None:
        return None
    out = {k: rec[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "sequences_per_rank", "cells_per_step",
                               "gpu_launches", "cpu_baseline", "parity", "tiers", "hazard_pairs")}
    out["workload"] = rec["config"]["workload"]
    out["mode"] = rec["config"]["mode"]
    out["e2e"] = rec["e2e"]
    r = rec["roofline"]
    out["roofline"] = {k: r[k] for k in ("bound", "achieved", "peak", "unit", "frac", "frac_of", "frac_step", "traffic")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=None, help="bench ONE configuration (1..5) alone; default: cfg 2 + legs")
    ap.add_argument("--n", type=int, default=None, help="override the number of streamed sequences of the whole job")
    ap.add_argument("--mode", default=None, choices=["score", "align", "ranges", "3pass"],
                    help="override the workload's mode (ranges = sw_score_ranges: score + alignment ranges, no traceback matrix; "
                         "3pass = sw_align_from_i8_3pass: ranges + banded alignment of the bounding box)")
    ap.add_argument("--align-opts", default=None, help="mode,checkpoint_log2,slack for zoe_cuda_set_align_options (tuning)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--legs", default="auto", help="auto | none | comma list of align,cfg1,cfg4,cfg4_3pass,align_tieheavy,cfg5,w512")
    ap.add_argument("--leg-steps", type=int, default=5)
    ap.add_argument("--parity", default="full", choices=["full", "sample"],
                    help="full: cfg 1 / 3 / 5 are checked on the whole set (SURVEY 8(d)); sample: a bounded prefix")
    ap.add_argument("--scoring", default=None, help="match,mismatch,gap_open,gap_extend for the DNA configurations "
                                                    "(e.g. 4,-2,-3,-1: many E == H == F ties -> literal striped kernels)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline workload's results of the last timed step to DIR/<name>.npy (float64, "
                         "at most 64 MB: a seeded sample of reads when larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; the reference arm times a prefix of the workload")
    if args.scoring:
        global SCORING
        SCORING = tuple(int(v) for v in args.scoring.split(","))
    args.warmup = max(args.warmup, 0)
    headline_alone = args.config is not None
    if args.config is None:
        args.config = 2

    if args.impl == "reference":
        run_reference(args)
        return

    ctx = Ctx(args)
    cpu = not args.no_cpu_baseline
    full = args.parity == "full"
    head = run_leg(ctx, args.config, args.mode, args.n, args.steps, args.warmup, cpu, 12.0, args.align_opts,
                   sample_clocks=True, full_parity=full, dump_dir=args.dump_outputs)

    legs = {}
    want = []
    if args.legs == "auto":
        if not headline_alone and args.n is None:
            want = (["align", "cfg5", "cfg4", "cfg4_3pass", "align_tieheavy", "cfg1", "sneaky", "w512"] if ctx.n_gpus == 1 else ["align"])
    elif args.legs != "none":
        want = [x for x in args.legs.split(",") if x]
    for leg in want:
        ls, lw = args.leg_steps, 3
        if leg == "align":
            legs["align"] = compact(run_leg(ctx, 3, "align", None, ls, lw, cpu, 6.0, args.align_opts, full_parity=full))
        elif leg == "cfg5":
            legs["cfg5"] = compact(run_leg(ctx, 5, None, None, ls, lw, cpu, 6.0, full_parity=full))
        elif leg == "cfg4":
            r = run_leg(ctx, 4, None, 20_000, 3, 3, cpu, 5.0, full_parity=full)
            if r:
                r["config"]["workload"] += " [the first 20000 reads of the 100k-read set]"
            legs["cfg4"] = compact(r)
        elif leg == "cfg4_3pass":
            # SURVEY 8(f).1: CIGARs for long reads through the memory-light 3-pass alignment (long-row ranges + banded pass 3)
            r = run_leg(ctx, 4, "3pass", 20_000, 3, 2, cpu, 5.0, full_parity=full)
            if r:
                r["config"]["workload"] += " [the first 20000 reads of the 100k-read set]"
            legs["cfg4_3pass"] = compact(r)
        elif leg == "align_tieheavy":
            # VERDICT r1 #4: a scoring whose walks meet E == H == F ties (6.7 % of the pairs go through the literal striped
            # kernels) -- the cost of zoe's lane-layout-dependent tie-breaks, checked on every pair against the CPU port
            legs["align_tieheavy"] = compact(run_leg(ctx, 3, "align", 200_000, 3, 2, cpu, 6.0, full_parity=full,
                                                     scoring=(2, -3, -4, -1)))
        elif leg == "sneaky" and ctx.rank == 0 and ctx.n_gpus == 1:
            legs["sneaky_snake"] = sneaky_leg(ctx, cpu)
        elif leg == "cfg1":
            legs["cfg1"] = compact(run_leg(ctx, 1, None, None, max(ls, 20), lw, cpu, 2.0, full_parity=full))
        elif leg == "w512" and cpu and ctx.rank == 0 and ctx.n_gpus == 1:
            # SURVEY 8(d): the score-only CPU baseline with zoe's w512 preset (i8 x 64; sw/mod.rs:285-286) beside w256
            from oracle import cpu_baseline as CB
            key, name, matrix, go, ge, targets, (buf, offs), _ = make_workload(2, 200_000)
            threads = CB.hardware_threads()
            n_s = sized_sample(len(offs) - 1, lambda k: cpu_port_run(matrix, go, ge, targets, buf, offs, k, threads, 512), 5.0)
            g, dt, _ = cpu_port_run(matrix, go, ge, targets, buf, offs, n_s, threads, 512)
            legs["cpu_w512"] = {"value": g, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"cfg2, first {n_s} sequences x 8 profiled, score-only, w512 lanes i8x64/i16x32/i32x16 "
                                          f"({dt:.1f} s, {CB.isa()})"}

    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": ctx.n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "s16x2 packed (s32 on overflow)", "data": "synthetic",
            "config": head["config"], "sequences_per_rank": head["sequences_per_rank"],
            "cells_per_step": head["cells_per_step"],
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "roofline": head["roofline"],
            "cpu_baseline": head["cpu_baseline"], "parity": head["parity"], "tiers": head["tiers"],
        }
        if legs:
            line["legs"] = legs
            if "align" in legs:
                line["align"] = legs["align"]  # the "with traceback" half of the metric, also at top level
        print(json.dumps(line), flush=True)
    if ctx.distributed:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
