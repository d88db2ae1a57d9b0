"""Seeded synthetic workloads for the five BASELINE.json configurations (SURVEY.md 8(d)).

Pure host-side data generation (numpy, PCG64 with fixed seeds); nothing here is timed.
"""
from __future__ import annotations

import os

import numpy as np

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = np.zeros(256, dtype=np.uint8)
_COMP[list(b"ACGT")] = list(b"TGCA")
_AA20 = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)

#: synthetic influenza-A segment lengths (PB2, PB1, PA, HA, NP, NA, M, NS)
FLU_SEGMENT_LENGTHS = (2341, 2341, 2233, 1778, 1565, 1413, 1027, 890)
SARS2_LENGTH = 29903


def random_dna(rng: np.random.Generator, n: int) -> np.ndarray:
    return _ACGT[rng.integers(0, 4, n)]


def pack(seqs):
    """list of uint8 arrays -> (concatenated buffer, uint64 offsets)."""
    offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    buf = np.concatenate(seqs) if len(seqs) else np.zeros(1, dtype=np.uint8)
    return np.ascontiguousarray(buf, dtype=np.uint8), offs


def _mutate(rng, frag, sub, ins, dele, alphabet):
    """Apply substitutions / insertions / deletions (geometric insertion length, p = 0.5); vectorised."""
    n = len(frag)
    if n == 0:
        return np.zeros(0, dtype=np.uint8)
    r = rng.random(n)
    deleted = r < dele
    inserted = (~deleted) & (r < dele + ins)
    substituted = (~deleted) & (r < dele + ins + sub)
    ins_len = np.where(inserted, rng.geometric(0.5, n), 0)
    out_len = ins_len + (~deleted)
    total = int(out_len.sum())
    if total == 0:
        return np.zeros(0, dtype=np.uint8)
    idx = np.repeat(np.arange(n), out_len)
    first = np.cumsum(out_len) - out_len
    within = np.arange(total) - np.repeat(first, out_len)
    is_ins = within < np.repeat(ins_len, out_len)
    out = np.asarray(frag, dtype=np.uint8)[idx]
    rnd = is_ins | substituted[idx]
    out[rnd] = alphabet[rng.integers(0, len(alphabet), int(rnd.sum()))]
    return out


def _read_errors(rng, frag, read_len, sub, indel):
    """The read error model: an indel in ~``2*indel*read_len`` of the reads, then substitutions.  ``frag`` is
    ``[n, span]`` with some slack past ``read_len`` so that deletions still leave ``read_len`` bases; returns
    ``[n, read_len]``."""
    span = frag.shape[1]
    has_indel = rng.random(len(frag)) < (2 * indel * read_len)
    for k in np.nonzero(has_indel)[0]:
        f = frag[k]
        pos = int(rng.integers(10, read_len - 10))
        ln = int(rng.geometric(0.5))
        if rng.random() < 0.5:
            f2 = np.concatenate([f[:pos], random_dna(rng, ln), f[pos:]])[:span]
        else:
            f2 = np.concatenate([f[:pos], f[pos + ln:], random_dna(rng, ln)])[:span]
        frag[k] = f2
    frag = frag[:, :read_len].copy()
    subs = rng.random(frag.shape) < sub
    frag[subs] = _ACGT[rng.integers(0, 4, int(subs.sum()))]
    return frag


def illumina_reads(rng: np.random.Generator, targets, n_reads: int, read_len: int = 150, sub: float = 0.01,
                   indel: float = 0.001, random_frac: float = 0.05):
    """Fixed-length reads drawn from uniformly chosen targets, both strands, with a few errors.

    Vectorised: substitutions everywhere, indels only on the ~``2*indel*read_len`` fraction of reads that get one.
    Returns a ``[n_reads, read_len]`` uint8 array.
    """
    lens = np.array([len(t) for t in targets])
    which = rng.integers(0, len(targets), n_reads)
    reads = np.empty((n_reads, read_len), dtype=np.uint8)
    span = read_len + 8  # a little slack so deletions still leave read_len bases
    for ti, t in enumerate(targets):
        idx = np.nonzero(which == ti)[0]
        if idx.size == 0:
            continue
        tt = np.concatenate([t, random_dna(rng, span)])  # reads may run off the 3' end into noise
        start = rng.integers(0, max(1, lens[ti] - read_len + 1), idx.size)
        frag = _read_errors(rng, tt[start[:, None] + np.arange(span)[None, :]], read_len, sub, indel)
        rc = rng.random(idx.size) < 0.5
        frag[rc] = _COMP[frag[rc][:, ::-1]]
        reads[idx] = frag
    rnd = rng.random(n_reads) < random_frac
    reads[rnd] = _ACGT[rng.integers(0, 4, (int(rnd.sum()), read_len))]
    return reads


def paired_reads(rng: np.random.Generator, targets, n_pairs: int, read_len: int = 150, insert_mean: float = 350.0,
                 insert_sd: float = 50.0, sub: float = 0.01, indel: float = 0.001, random_frac: float = 0.05):
    """Illumina-like FR read pairs.  Each pair's fragment comes from a uniformly chosen target, on a random strand, with
    an insert length drawn from a normal distribution (at least ``read_len``, at most the target).  Mate 1 is the
    fragment's first ``read_len`` bases, mate 2 the reverse complement of its last ``read_len`` bases; each mate then
    gets the error model of :func:`illumina_reads`, and a ``random_frac`` of the mates are replaced by random reads.

    Returns ``(mates1, mates2, truth)``: two ``[n_pairs, read_len]`` uint8 arrays and a dict of per-pair arrays,
    ``target``, ``start`` (the fragment's first target position), ``insert`` and ``strand`` (1: the fragment is the
    reverse complement of ``target[start:start + insert]``)."""
    lens = np.array([len(t) for t in targets])
    which = rng.integers(0, len(targets), n_pairs)
    strand = rng.integers(0, 2, n_pairs).astype(np.uint8)
    insert = np.minimum(np.maximum(np.rint(rng.normal(insert_mean, insert_sd, n_pairs)), read_len).astype(np.int64),
                        lens[which])
    start = (rng.random(n_pairs) * (lens[which] - insert + 1)).astype(np.int64)
    mates = [np.empty((n_pairs, read_len), dtype=np.uint8) for _ in range(2)]
    span = read_len + 8
    for ti, t in enumerate(targets):
        idx = np.nonzero(which == ti)[0]
        if idx.size == 0:
            continue
        tt = np.concatenate([random_dna(rng, span), t, random_dna(rng, span)])  # reads may run off either end
        s, e = start[idx] + span, start[idx] + insert[idx] + span
        fwd = tt[s[:, None] + np.arange(span)[None, :]]            # the target's strand, read from the fragment start
        rev = _COMP[tt[(e - 1)[:, None] - np.arange(span)[None, :]]]  # the other strand, read from the fragment end
        rc = strand[idx] == 1
        first, second = np.where(rc[:, None], rev, fwd), np.where(rc[:, None], fwd, rev)
        mates[0][idx] = _read_errors(rng, first, read_len, sub, indel)
        mates[1][idx] = _read_errors(rng, second, read_len, sub, indel)
    for m in mates:
        rnd = rng.random(n_pairs) < random_frac
        m[rnd] = _ACGT[rng.integers(0, 4, (int(rnd.sum()), read_len))]
    return mates[0], mates[1], {"target": which, "start": start, "insert": insert, "strand": strand}


def fixed_len_batch(reads2d: np.ndarray):
    n, L = reads2d.shape
    offs = (np.arange(n + 1, dtype=np.uint64) * np.uint64(L)).astype(np.uint64)
    return np.ascontiguousarray(reads2d.reshape(-1)), offs


def golden_ha(root: str) -> np.ndarray:
    with open(os.path.join(root, "tests", "golden", "KJ907631.1.txt"), "rb") as f:
        return np.frombuffer(f.read(), dtype=np.uint8).copy()


def config1(root: str, n_reads: int = 10_000, seed: int = 1):
    """10k x 150 nt reads vs the 1704-nt H5 HA (the reference's CPU-runnable case)."""
    ha = golden_ha(root)
    rng = np.random.default_rng(seed)
    return [ha], illumina_reads(rng, [ha], n_reads)


def config2(n_reads: int = 1_000_000, seed_targets: int = 2, seed_reads: int = 3):
    """1M x 150 nt reads vs 8 synthetic influenza-A-length segments, score only."""
    rng = np.random.default_rng(seed_targets)
    targets = [random_dna(rng, L) for L in FLU_SEGMENT_LENGTHS]
    rng = np.random.default_rng(seed_reads)
    return targets, illumina_reads(rng, targets, n_reads)


def config3(root: str, n_reads: int = 1_000_000, seed: int = 4):
    """1M x 150 nt reads vs the 1704-nt HA, with traceback."""
    ha = golden_ha(root)
    rng = np.random.default_rng(seed)
    return [ha], illumina_reads(rng, [ha], n_reads)


def config4(n_reads: int = 100_000, seed_genome: int = 5, seed_reads: int = 6, min_len=1000, max_len=5000):
    """ONT-like 1-5 kb reads (6 % sub, 4 % ins, 4 % del) vs a 29 903-nt genome."""
    rng = np.random.default_rng(seed_genome)
    genome = random_dna(rng, SARS2_LENGTH)
    rng = np.random.default_rng(seed_reads)
    reads = []
    for _ in range(n_reads):
        L = int(rng.integers(min_len, max_len + 1))
        s = int(rng.integers(0, SARS2_LENGTH - L + 1))
        frag = genome[s:s + L]
        if rng.random() < 0.5:
            frag = _COMP[frag[::-1]]
        reads.append(_mutate(rng, frag, 0.06, 0.04, 0.04, _ACGT))
    return [genome], reads


def config5(n_queries: int = 1_000_000, seed_target: int = 7, seed_queries: int = 8, qlen: int = 300, tlen: int = 566):
    """300-aa queries vs a 566-aa target: 40 % random (stay in the i8 tier), 60 % diverged windows (i16)."""
    rng = np.random.default_rng(seed_target)
    target = _AA20[rng.integers(0, 20, tlen)]
    rng = np.random.default_rng(seed_queries)
    q = _AA20[rng.integers(0, 20, (n_queries, qlen))]
    related = np.nonzero(rng.random(n_queries) < 0.6)[0]
    start = rng.integers(0, tlen - qlen + 1, related.size)
    win = target[start[:, None] + np.arange(qlen)[None, :]]
    div = rng.uniform(0.10, 0.40, related.size)
    keep = rng.random(win.shape) >= div[:, None]
    q[related] = np.where(keep, win, q[related])
    return [target], q
