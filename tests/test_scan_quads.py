"""GPU (-m gpu): the quad variant of the ungapped scan (four G = 8 queries per warp on one target, V-form profile words from tensor
memory) against the oracle, and against the one-query-per-group kernel (B200_SCAN_NO_QUADS=1) on the same inputs."""
import numpy as np
import pytest

from mmseqs2_b200 import synth
from oracle.pyoracle import pack_targets

pytestmark = pytest.mark.gpu

# capacities 2*8*K rows of the G = 8 classes (K = 4, 6, ..., 32): 64 .. 512 rows in 32-row steps
G8_CAPS = list(range(64, 513, 32))


def _db(rng, bg, qs, n=160):
    res, off = synth.random_seqs(rng, n, bg, mean=250, sigma=0.8, lo=1, hi=1500)
    synth.plant_homologs(rng, res, off, qs, bg, frac=0.5, subst=0.15, indel=0.01)
    seqs = synth.split(res, off)
    # near-identical targets saturate at 255 - bias in every group of a quad; short targets (1, < 8, < 16 residues) end mid-chunk
    for k, q in enumerate(qs):
        seqs[(7 * k) % len(seqs)] = q.copy()
    seqs[1] = seqs[1][:1]
    seqs[2] = seqs[2][:5]
    seqs[3] = seqs[3][:13]
    return pack_targets(seqs)


def _check(ctx, oracle, submat, qs, cbs, monkeypatch):
    td, to = _db(np.random.default_rng(len(qs)), synth.background(submat.pback), qs)
    ctx.load_db(td, to.astype(np.uint64), 21)
    profs = [submat.ssw_query(q, comp_bias=cb) for q, cb in zip(qs, cbs)]
    hits, n_hits, dense = ctx.ungapped_scan(profs, want_dense=True)
    for qi, (q, cb) in enumerate(zip(qs, cbs)):
        c, bias = oracle.query_cb(q, cb)
        exp = oracle.ungapped(q, c, bias, td, to)
        assert np.array_equal(dense[qi].astype(np.int32), exp), (qi, len(q), np.nonzero(dense[qi] != exp)[0][:5])
    monkeypatch.setenv("B200_SCAN_NO_QUADS", "1")
    hits1, n_hits1, dense1 = ctx.ungapped_scan(profs, want_dense=True)
    monkeypatch.delenv("B200_SCAN_NO_QUADS")
    assert np.array_equal(dense, dense1) and np.array_equal(n_hits, n_hits1) and np.array_equal(hits, hits1)


def _seqs(rng, bg, lens):
    return [synth.random_seqs(rng, 1, bg, mean=L, sigma=0, lo=L, hi=L, normal=True)[0] for L in lens]


def test_quads_every_g8_class_boundary(ctx, oracle, submat, monkeypatch):
    """qlen = capacity - 1 (last length of a class) and capacity (first of the next) for every G = 8 class, so that quads mix
    lengths across K classes and every quad K is instantiated; bias differs within quads (composition bias on / off)"""
    rng = np.random.default_rng(41)
    bg = synth.background(submat.pback)
    lens = sorted(set([c - 1 for c in G8_CAPS] + G8_CAPS[:-1] + [5, 20, 63]))
    qs = _seqs(rng, bg, lens)
    _check(ctx, oracle, submat, qs, [i % 3 != 0 for i in range(len(qs))], monkeypatch)


@pytest.mark.parametrize("n", [4, 5, 6, 7, 16])
def test_quads_equal_lengths_and_leftovers(ctx, oracle, submat, monkeypatch, n):
    """4k + 0 ... 4k + 3 queries of one length (the n mod 4 shortest go to the one-query kernel), and a 16-query batch of
    lengths around 350 as the benchmark runs it"""
    rng = np.random.default_rng(100 + n)
    bg = synth.background(submat.pback)
    lens = [350] * n if n < 16 else list(rng.integers(300, 420, n))
    qs = _seqs(rng, bg, lens)
    _check(ctx, oracle, submat, qs, [i % 2 == 0 for i in range(n)], monkeypatch)


def test_quads_next_to_longer_classes(ctx, oracle, submat, monkeypatch):
    """G = 8 quads in one batch with G = 16 / G = 32 and tiled queries, which keep the one-query kernel"""
    rng = np.random.default_rng(9)
    bg = synth.background(submat.pback)
    qs = _seqs(rng, bg, [120, 130, 140, 150, 511, 512, 700, 1500, 2100, 30])
    _check(ctx, oracle, submat, qs, [True] * len(qs), monkeypatch)
