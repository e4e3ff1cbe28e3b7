"""Randomised differential checks of the host-side formats and statistics against the reference's own code: alignment records
(Matcher::resultToBuffer, all three identity formats, E-values over 300 decades, compressed and plain backtraces), prefilter records
(parsePrefilterHits / prefilterHitToBuffer round trip), E-values and bit scores (EvalueComputation, doubles compared exactly).
The reference's answers come from the `ref` fixture (recorded from oracle/_ref, tests/golden/ref_calls_v1.pkl.xz)."""
import numpy as np

from mmseqs2_b200 import alignment as al


def test_alignment_records_equal_result_to_buffer(ref):
    rng = np.random.default_rng(7)
    for t in range(420):
        key, score = int(rng.integers(0, 2 ** 32)), int(rng.integers(-50, 5000))
        seq_id = [1.0, float(rng.random()), 0.9995, 0.0995, float(np.float32(rng.integers(0, 1001)) / 1000), 0.0][t % 6]
        ev = float(10.0 ** rng.uniform(-300, 5)) if t % 7 else 0.0
        ql, dl = int(rng.integers(1, 70000)), int(rng.integers(1, 70000))
        qs, qe = sorted(int(x) for x in rng.integers(0, ql, 2))
        ds, de = sorted(int(x) for x in rng.integers(0, dl, 2))
        bt = bytes(rng.choice(list(b"MID"), int(rng.integers(0, 60))).astype(np.uint8)) if t % 3 == 0 else b""
        add, comp = bool(t % 2), bool(t % 4 < 2)
        r = np.zeros(1, al.RESULT_DTYPE)
        for f, v in (("db_key", key), ("score", score), ("seq_id", seq_id), ("eval", ev), ("q_start", qs), ("q_end", qe), ("q_len", ql),
                     ("db_start", ds), ("db_end", de), ("db_len", dl)):
            r[f] = v
        assert al.result_to_buffer(r[0], bt, add, comp) == ref.result_to_buffer(key, score, seq_id, ev, qs, qe, ql, ds, de, dl, bt, add, comp), t


def test_prefilter_records_round_trip(ref):
    rng = np.random.default_rng(8)
    for t in range(60):
        entry = b"".join(b"%d\t%d\t%d\n" % (int(rng.integers(0, 2 ** 32)), int(rng.integers(-3000, 3000)), int(rng.integers(-32768, 32768)))
                         for _ in range(int(rng.integers(0, 30))))
        ids, sc, dg, back = ref.prefilter_roundtrip(entry)
        h = al.parse_prefilter_hits(entry)
        assert np.array_equal(h["seq_id"], ids) and np.array_equal(h["pref_score"], sc) and np.array_equal(h["diagonal"], dg), t
        assert al.prefilter_hits_to_buffer(h) == back, t


def test_evalues_and_bit_scores_are_the_reference_doubles(ref):
    rng = np.random.default_rng(9)
    for t in range(400):
        dbres, score, ql = int(10 ** rng.uniform(3, 11)), float(rng.integers(0, 3000)), float(rng.integers(1, 40000))
        p = al.EvalueParams.defaults("blosum62.out", 11, 1, dbres, gapped=True)
        e, bits = ref.evalue_bits(11, 1, dbres, score, ql)
        assert p.evalue(score, ql) == e and p.bit_score(score) == bits, (t, dbres, score, ql)
    # the ungapped set rescorediagonal scores with (EvalueComputation(dbResCount, subMat))
    for t in range(400):
        dbres, score, ql = int(10 ** rng.uniform(3, 11)), float(rng.integers(0, 1500)), float(rng.integers(1, 40000))
        p = al.EvalueParams.defaults("blosum62.out", 0, 0, dbres, gapped=False)
        e, bits = ref.evalue_bits_ungapped(dbres, score, ql)
        assert p.evalue(score, ql) == e and p.bit_score(score) == bits, ("ungapped", t, dbres, score, ql)
