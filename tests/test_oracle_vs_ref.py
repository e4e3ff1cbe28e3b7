"""CPU: oracle/oracle.c against the reference's own sources (oracle.pyoracle.Ref; the `ref` fixture answers from the recording of
the reference's outputs in tests/golden)."""
import numpy as np
import pytest

from oracle.pyoracle import pack_targets
from mmseqs2_b200 import synth


def _targets(rng, bg, q, n):
    tg = []
    for k in range(n):
        m = k % 3
        if m == 0 or len(q) < 4:
            tg.append(synth.random_seqs(rng, 1, bg, mean=200, sigma=0.8, lo=1, hi=900)[0])
        elif m == 1:
            tg.append(synth.mutate(rng, q, bg, 0.37, 0.08))
        else:
            a = int(rng.integers(0, len(q) - 1))
            b = int(rng.integers(a + 1, len(q) + 1))
            pre = synth.random_seqs(rng, 1, bg, mean=20, sigma=0.5, lo=1, hi=60)[0]
            tg.append(np.concatenate([pre, synth.mutate(rng, q[a:b], bg, 0.2, 0.04), pre[::-1]]))
    return pack_targets(tg)


def test_matrix_fixture_matches_reference(ref, blosum):
    mat, pb, _ = ref.matrix()
    assert np.array_equal(mat, blosum[0]) and np.array_equal(pb, blosum[1])


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_pairs_all_entry_points(ref, oracle, blosum, seed):
    rng = np.random.default_rng(seed)
    bg = synth.background(blosum[1])
    for it in range(5):
        qL = int(rng.integers(1, 40)) if it % 4 == 0 else int(rng.integers(20, 600))
        q = synth.random_seqs(rng, 1, bg, mean=qL, sigma=0, lo=qL, hi=qL, normal=True)[0]
        if it % 5 == 0:
            q[:: 5] = 20  # X
        td, to = _targets(rng, bg, q, 120)
        f = ref.comp_bias(q)
        assert np.array_equal(f.view(np.uint32), oracle.comp_bias(q).view(np.uint32))
        for cbf in (True, False):
            cb, bias = oracle.query_cb(q, cbf)
            assert np.array_equal(ref.ungapped(q, cbf, td, to), oracle.ungapped(q, cb, bias, td, to))
            assert np.array_equal(ref.sw_score_endpos(q, cbf, td, to), oracle.sw_score_endpos(q, cb, bias, td, to))
            a, _, _ = ref.ssw_align(q, cbf, td, to, mode=1)
            assert np.array_equal(a[:, :6], oracle.sw_align(q, cb, bias, td, to))
        ids = rng.integers(0, len(to) - 1, 500).astype(np.uint32)
        dg = rng.integers(-qL - 3, 700, 500).astype(np.int16).view(np.uint16)
        for use in (True, False):
            cb4 = oracle.round_bias_diag(f) if use else np.zeros(qL, np.int8)
            c1, r1 = ref.diag(q, f if use else None, td, to, ids, dg)
            c2, r2 = oracle.diag(q, cb4, td, to, ids, dg)
            assert np.array_equal(c1, c2) and np.array_equal(r1, r2)


def test_gap_penalty_variants(ref, oracle, blosum):
    rng = np.random.default_rng(99)
    bg = synth.background(blosum[1])
    q = synth.random_seqs(rng, 1, bg, mean=180, sigma=0, lo=180, hi=180, normal=True)[0]
    td, to = _targets(rng, bg, q, 90)
    cb, bias = oracle.query_cb(q, True)
    for go, ge in ((11, 1), (10, 2), (5, 5), (20, 1), (2, 1)):
        assert np.array_equal(ref.sw_score_endpos(q, True, td, to, go, ge), oracle.sw_score_endpos(q, cb, bias, td, to, go, ge))
        a, _, _ = ref.ssw_align(q, True, td, to, go, ge, mode=1)
        assert np.array_equal(a[:, :6], oracle.sw_align(q, cb, bias, td, to, go, ge))


def test_backtrace_gap_penalty_variants_and_wide_bands(ref, oracle, blosum):
    """banded_sw + computerBacktrace of the reference (ssw_align mode 2) against the restatement for several gap costs and for
    alignments whose band doubles far beyond |dbLen - qLen| + 1 -- the cases the GPU parity test of the warp backtrace kernel
    (tests/test_gpu_parity.py::test_backtrace_gap_penalties_and_wide_bands) checks against the oracle.
    Only go > ge: with go <= ge the reference's striped kernels stop being the Gotoh recurrence (on the 220-residue deletion below
    its forward pass scores 1316, its own reverse pass 1321, the textbook DP 1329, and ssw_align exits on its forward/backward
    check) -- there is no reference behaviour to pin there; the library and the oracle compute the textbook recurrence."""
    rng = np.random.default_rng(4242)
    bg = synth.background(blosum[1])
    q = synth.random_seqs(rng, 1, bg, mean=600, sigma=0, lo=600, hi=600, normal=True)[0]
    tg = [synth.mutate(rng, q, bg, s, i) for s, i in ((0.1, 0.02), (0.3, 0.05), (0.2, 0.0), (0.05, 0.1), (0.4, 0.03))]
    tg.append(np.concatenate([q[:200], q[420:]]))
    tg.append(np.concatenate([q[:100], synth.random_seqs(rng, 1, bg, mean=300, sigma=0, lo=300, hi=300, normal=True)[0], q[100:]]))
    tg.append(q[50:550].copy())
    tg += [synth.mutate(rng, q[a:a + 250], bg, 0.25, 0.04) for a in (0, 100, 350)]
    td, to = pack_targets(tg)
    cb, bias = oracle.query_cb(q, True)
    checked = 0
    for go, ge in ((11, 1), (5, 2), (20, 1), (10, 2), (4, 3)):
        a, _, bts = ref.ssw_align(q, True, td, to, go, ge, mode=2, want_bt=True)
        exp = oracle.sw_align(q, cb, bias, td, to, go, ge)
        assert np.array_equal(a[:, :6], exp), (go, ge)
        for k in range(len(tg)):
            if exp[k, 4] == -1:
                continue
            bt, ids = oracle.backtrace(q, cb, tg[k], exp[k], go, ge)
            assert bt == bts[k] and ids == a[k, 6], (go, ge, k)
            checked += 1
    assert checked >= 40


def test_rescore_diagonal_modes(ref, oracle):
    """groundwork for SURVEY 8f row 3 (no device path yet): the restatement of DistanceCalculator::computeUngappedAlignment equals
    the reference for all five rescore modes on ASCII sequences with lower case, ambiguity letters and '*' ends"""
    rng = np.random.default_rng(31337)
    m = ref.ascii_matrix()
    letters = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWYXBZUacdklmn", np.uint8)
    checked = 0
    for rep in range(60):
        qL, tL = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        q = bytearray(rng.choice(letters, qL).tobytes()); t = bytearray(rng.choice(letters, tL).tobytes())
        if rep % 3 == 0:                                   # a shared segment so that the scores are not all tiny
            n = int(rng.integers(1, min(qL, tL) + 1)); a = int(rng.integers(0, qL - n + 1)); b = int(rng.integers(0, tL - n + 1))
            t[b:b + n] = q[a:a + n]
            for k in rng.integers(0, n, n // 8):
                t[b + int(k)] = int(rng.choice(letters))
        if rep % 5 == 0:
            q[0] = ord("*"); t[-1] = ord("*")
        for diag in [0, 1, -1 & 0xffff, int(rng.integers(-tL, qL + 1)) & 0xffff, int(rng.integers(-tL, qL + 1)) & 0xffff, 5000, 60000]:
            for mode in range(5):
                exp = ref.rescore_diagonal(bytes(q), bytes(t), diag, mode)
                got = oracle.rescore_diagonal(bytes(q), bytes(t), diag, m, mode)
                assert np.array_equal(got, exp), (rep, diag, mode, got, exp)
                checked += 1
    assert checked == 60 * 7 * 5

