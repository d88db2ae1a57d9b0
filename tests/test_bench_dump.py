"""CPU-only: bench.py --dump-outputs writes the pairs' results exactly, within its size limit, and samples the same
reads whatever the results are (so the dumps of two builds compare pair for pair)."""
import os

import numpy as np

import bench


def _score_outs(rng, pairs):
    return {"score": rng.integers(0, 1 << 32, pairs, dtype=np.uint64).astype(np.uint32),
            "status": rng.integers(0, 3, pairs, dtype=np.uint8), "tier": rng.integers(8, 33, pairs, dtype=np.uint8)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _total_bytes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_small_score_dump_is_complete_and_exact(tmp_path):
    rng = np.random.default_rng(1)
    outs = _score_outs(rng, 50 * 8)
    bench.dump_outputs(str(tmp_path), outs, 50, 8, "score")
    got = _load(str(tmp_path))
    assert sorted(got) == ["read_index", "score", "status", "tier"]
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["read_index"], np.arange(50))
    for k in ("score", "status", "tier"):
        assert np.array_equal(got[k], outs[k].astype(np.float64)), k


def test_large_dump_is_a_fixed_sample_within_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    n, n_prof = 20_000, 8
    dirs = [str(tmp_path / "a"), str(tmp_path / "b")]
    for seed, d in zip((2, 3), dirs):
        outs = _score_outs(np.random.default_rng(seed), n * n_prof)
        bench.dump_outputs(d, outs, n, n_prof, "score")
        assert _total_bytes(d) <= 1 << 20
        got = _load(d)
        rows = got["read_index"].astype(np.int64)
        assert 0 < len(rows) < n and np.all(np.diff(rows) > 0)
        pairs = (rows[:, None] * n_prof + np.arange(n_prof)).reshape(-1)
        assert np.array_equal(got["score"], outs["score"][pairs].astype(np.float64))
    assert np.array_equal(np.load(os.path.join(dirs[0], "read_index.npy")), np.load(os.path.join(dirs[1], "read_index.npy")))


def _align_outs(rng, n, n_prof, max_words):
    pairs = n * n_prof
    outs = _score_outs(rng, pairs)
    for k in ("ref_start", "ref_end", "query_start", "query_end"):
        outs[k] = rng.integers(0, 5000, pairs, dtype=np.uint32)
    outs["hazard"] = rng.integers(0, 2, pairs, dtype=np.uint8)
    lens = rng.integers(0, max_words + 1, pairs)
    outs["cigar_off"] = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    outs["cigar"] = rng.integers(0, 1 << 32, int(lens.sum()) + 100, dtype=np.uint64).astype(np.uint32)  # + spare capacity
    return outs


def test_align_dump_keeps_each_pairs_cigar(tmp_path):
    n, n_prof = 300, 3
    outs = _align_outs(np.random.default_rng(4), n, n_prof, 12)
    bench.dump_outputs(str(tmp_path), outs, n, n_prof, "align")
    got = _load(str(tmp_path))
    assert sorted(got) == ["cigar", "cigar_len", "hazard", "query_end", "query_start", "read_index", "ref_end",
                           "ref_start", "score", "status", "tier"]
    off = outs["cigar_off"].astype(np.int64)
    assert np.array_equal(got["cigar_len"], np.diff(off).astype(np.float64))
    assert np.array_equal(got["cigar"], outs["cigar"][: off[-1]].astype(np.float64))


def test_sampled_align_dump_cuts_cigar_words_at_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    n, n_prof = 5000, 2
    outs = _align_outs(np.random.default_rng(5), n, n_prof, 200)
    bench.dump_outputs(str(tmp_path), outs, n, n_prof, "3pass")
    assert _total_bytes(str(tmp_path)) <= 1 << 20
    got = _load(str(tmp_path))
    assert "hazard" not in got
    rows = got["read_index"].astype(np.int64)
    pairs = (rows[:, None] * n_prof + np.arange(n_prof)).reshape(-1)
    lo, hi = outs["cigar_off"][pairs].astype(np.int64), outs["cigar_off"][pairs + 1].astype(np.int64)
    assert np.array_equal(got["cigar_len"], (hi - lo).astype(np.float64))
    want = np.concatenate([outs["cigar"][a:b] for a, b in zip(lo, hi)])
    assert 0 < len(got["cigar"]) < len(want)
    assert np.array_equal(got["cigar"], want[: len(got["cigar"])].astype(np.float64))
