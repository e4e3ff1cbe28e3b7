"""Word-mode saturation: alignments whose exact local score passes 32767.

The reference's word-mode Smith-Waterman (sw_sse2_word, StripedSmithWaterman.cpp:301-476) adds scores with adds_epi16, so every
cell saturates at 32767.  Such a pair reports score 32767, ends at the first column in which a cell reaches 32767 (smallest row in
that column), takes its start from a reverse pass that stops at the first column whose maximum is 32767, and is backtraced inside
that rectangle.  Titin-sized proteins against themselves or close homologs get there.  Fixture: tests/golden/saturated_v1.npz,
written by the reference's own code (tests/golden/make_saturated_golden.py); it also records each pair's exact int32 score and end,
which lie elsewhere for every saturated pair.

CPU: the oracle (oracle/oracle.c) against the fixture and, on seeded inputs, against the recorded reference.
GPU (-m gpu): every device entry point that can see such a pair against the fixture, bit for bit."""
import importlib.util
import os

import numpy as np
import pytest

from mmseqs2_b200 import synth
from oracle.pyoracle import pack_targets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def sat():
    with np.load(os.path.join(GOLDEN, "saturated_v1.npz")) as d:
        return dict(d.items())          # read once: the lazy NpzFile is not safe to share between threads


def _maker():
    spec = importlib.util.spec_from_file_location("make_saturated_golden", os.path.join(GOLDEN, "make_saturated_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _seq(d, o, i):
    return d[int(o[i]):int(o[i + 1])]


def _groups(sat):
    """-> [(group, query, comp bias, go, ge, pool target ids, slice of the per-pair rows)]"""
    off = sat["grp_off"]
    out = []
    for g in range(len(off) - 1):
        q = _seq(sat["qdata"], sat["qoff"], int(sat["grp_query"][g]))
        out.append((g, q, bool(sat["grp_cb"][g]), int(sat["grp_go"][g]), int(sat["grp_ge"][g]),
                    sat["grp_targets"][off[g]:off[g + 1]], slice(int(off[g]), int(off[g + 1]))))
    return out


def _target(sat, t):
    return _seq(sat["tdata"], sat["toff"], int(t))


# ---- CPU ------------------------------------------------------------------------------------------------------------------
def test_fixture_exercises_saturation(sat, blosum, oracle):
    """enough pairs saturate, their exact scores really pass 32767 and their exact ends lie elsewhere; other pairs pin the
    boundary from below.  The exact ends of the two shortest saturated pairs are recomputed here."""
    e, x = sat["endpos"], sat["exact"]
    sat_rows = (e[:, 0] == 32767) & (e[:, 3] == 1)
    assert sat_rows.sum() >= 20
    assert (x[sat_rows, 0] > 32767).all()
    assert ((x[sat_rows, 1] != e[sat_rows, 1]) | (x[sat_rows, 2] != e[sat_rows, 2])).sum() >= 20
    assert np.array_equal(x[~sat_rows], e[~sat_rows, :3])
    assert ((e[:, 0] >= 31000) & (e[:, 0] < 32767)).sum() >= 8
    assert any(len(q) > 16384 for _, q, *_ in _groups(sat))
    assert sum(int(sat["pssm%d_align" % k][:, 0].tolist().count(32767)) for k in (0, 1)) >= 4
    exact_endpos = _maker().exact_endpos
    mat = blosum[0]
    cells = []
    for g, q, cbf, go, ge, tg, sl in _groups(sat):
        for k, t in enumerate(tg):
            if sat_rows[sl][k]:
                cells.append((len(q) * len(_target(sat, t)), g, k))
    for _, g, k in sorted(cells)[:2]:
        _, q, cbf, go, ge, tg, sl = _groups(sat)[g]
        cb, _ = oracle.query_cb(q, cbf)
        prof = mat[:, q].astype(np.int64) + cb.astype(np.int64)
        assert exact_endpos(prof, _target(sat, tg[k]), go, ge) == tuple(int(v) for v in x[sl][k]), (g, k)


def test_oracle_equals_saturated_fixture(sat, oracle):
    """score, ends, word flag, start positions, backtrace and identity count of every pair (one pair per worker thread: the
    oracle's ctypes calls release the GIL)"""
    from concurrent.futures import ThreadPoolExecutor
    jobs = [(g, q, cbf, go, ge, t, sl.start + k) for g, q, cbf, go, ge, tg, sl in _groups(sat) for k, t in enumerate(tg)]
    jobs.sort(key=lambda j: -len(j[1]) * len(_target(sat, j[5])))      # largest first

    def one(job):
        g, q, cbf, go, ge, t, row = job
        cb, bias = oracle.query_cb(q, cbf)
        sd, so = pack_targets([_target(sat, t)])
        got = oracle.sw_align(q, cb, bias, sd, so, go, ge, nthreads=1)[0]
        bt, ids = oracle.backtrace(q, cb, _target(sat, t), got, go, ge)
        return got, bt, ids

    with ThreadPoolExecutor(8) as pool:
        results = list(pool.map(one, jobs))
    for job, (got, bt, ids) in zip(jobs, results):
        g, row = job[0], job[6]
        assert np.array_equal(got[[0, 2, 4, 5]], sat["endpos"][row]), (g, row, got, sat["endpos"][row])
        assert np.array_equal(got, sat["align"][row]), (g, row, got, sat["align"][row])
        assert bt == str(sat["bt"][row]) and ids == sat["ident"][row], (g, row)
    assert len(jobs) == len(sat["endpos"])


def test_oracle_vs_reference_saturated_random(ref, oracle, blosum):
    """seeded long queries against mutated, extended and truncated copies: the oracle equals the reference (recorded) on score,
    ends and mode-1 start positions, saturated or not"""
    rng = np.random.default_rng(32767)
    bg = synth.background(blosum[1])
    n_sat = 0
    for case in range(4):
        L = int(rng.integers(6000, 8000))
        q = synth.random_seqs(rng, 1, bg, mean=L, sigma=0, lo=L, hi=L, normal=True)[0]
        cbf = bool(case % 2)
        go, ge = ((11, 1), (5, 2), (20, 1), (11, 1))[case]
        a = int(rng.integers(0, 1000))
        tg = [synth.mutate(rng, q, bg, float(rng.uniform(0.0, 0.12)), float(rng.uniform(0.0, 0.02))),
              np.concatenate([synth.random_seqs(rng, 1, bg, mean=300, sigma=0, lo=300, hi=300, normal=True)[0], q[a:]]),
              q[a:a + int(rng.integers(4000, 6500))].copy()]
        sd, so = pack_targets(tg)
        cb, bias = oracle.query_cb(q, cbf)
        exp_e = ref.sw_score_endpos(q, cbf, sd, so, go, ge)
        exp_a, _, _ = ref.ssw_align(q, cbf, sd, so, go, ge, mode=1)
        got = oracle.sw_align(q, cb, bias, sd, so, go, ge)
        assert np.array_equal(got[:, [0, 2, 4, 5]], exp_e), (case, got, exp_e)
        assert np.array_equal(got, exp_a[:, :6]), (case, got, exp_a[:, :6])
        n_sat += int((exp_e[:, 0] == 32767).sum())
    assert n_sat >= 4


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _sw_endpos(ctx, queries, pairs, scores, go, ge):
    """b200_sw_endpos: end positions for pairs whose score is already known"""
    from mmseqs2_b200.api import END_DTYPE, _cqueries, _p, _u64
    pa = ctx._pairs(pairs)
    sc = np.ascontiguousarray(scores, np.int32)
    out = np.zeros(len(pa), END_DTYPE)
    ctx._check(ctx.lib.b200_sw_endpos(ctx.h, _cqueries(queries), len(queries), _p(pa), _u64(len(pa)), go, ge, _p(sc), _p(out)))
    return out


def _ends(rows):
    from mmseqs2_b200.api import END_DTYPE
    out = np.zeros(len(rows), END_DTYPE)
    for k, f in enumerate(("score", "qend", "dbend", "word")):
        out[f] = rows[:, k]
    return out


def _aln(rows):
    from mmseqs2_b200.api import ALN_DTYPE
    out = np.zeros(len(rows), ALN_DTYPE)
    for k, f in enumerate(("score", "qstart", "qend", "dbstart", "dbend", "word")):
        out[f] = rows[:, k]
    return out


ALN_FIELDS = ("score", "qstart", "qend", "dbstart", "dbend", "word")


@pytest.mark.gpu
def test_device_sequence_entry_points(sat, ctx, submat):
    """sw_score, sw_score_job, sw_score_endpos, sw_job, sw_endpos, sw_startpos, sw_align and sw_backtrace on every pair"""
    ctx.load_db(sat["tdata"], sat["toff"].astype(np.uint64), 21)
    for g, q, cbf, go, ge, tg, sl in _groups(sat):
        prof = [submat.ssw_query(q, comp_bias=cbf)]
        pairs = np.array([(0, t) for t in tg], np.uint32)
        e, a = sat["endpos"][sl], sat["align"][sl]
        ends = ctx.sw_score_endpos(prof, pairs, go, ge)
        got = np.stack([ends[f] for f in ("score", "qend", "dbend", "word")], 1)
        assert np.array_equal(got, e), ("sw_score_endpos", g, got, e)
        assert np.array_equal(ctx.sw_score(prof, pairs, go, ge), e[:, 0]), ("sw_score", g)
        job = ctx.sw_score_job(prof, pairs, go, ge)
        job.run()
        assert np.array_equal(job.fetch(), e[:, 0]), ("sw_score_job", g)
        job.close()
        job = ctx.sw_job(prof, pairs, go, ge)
        job.run()
        got = job.fetch()
        job.close()
        assert np.array_equal(np.stack([got[f] for f in ("score", "qend", "dbend", "word")], 1), e), ("sw_job", g)
        got = _sw_endpos(ctx, prof, pairs, e[:, 0], go, ge)
        assert np.array_equal(np.stack([got[f] for f in ("score", "qend", "dbend", "word")], 1), e), ("sw_endpos", g)
        st = ctx.sw_startpos(prof, pairs, _ends(e), go, ge)
        assert np.array_equal(np.stack([st[f] for f in ALN_FIELDS], 1), a), ("sw_startpos", g, st, a)
        aln = ctx.sw_align(prof, pairs, go, ge)
        assert np.array_equal(np.stack([aln[f] for f in ALN_FIELDS], 1), a), ("sw_align", g)
        out, bts = ctx.sw_backtrace(prof, [q], pairs, _aln(a), go, ge)
        for k in range(len(tg)):
            assert out["ok"][k] == 1 and bts[k] == str(sat["bt"][sl][k]), ("sw_backtrace", g, k)
            assert out["identical"][k] == sat["ident"][sl][k] and out["bt_len"][k] == len(bts[k]), ("sw_backtrace", g, k)


@pytest.mark.gpu
def test_device_pssm_queries(sat, ctx, submat):
    """sharp profile queries (submat.pssm_query) against their consensus and mutated copies: positions, backtrace, identity"""
    ctx.load_db(sat["tdata"], sat["toff"].astype(np.uint64), 21)
    for k in (0, 1):
        p = sat["pssm%d" % k]
        prof = [submat.pssm_query(p)]
        cons = p.argmax(0).astype(np.uint8)
        tg = sat["pssm%d_targets" % k]
        pairs = np.array([(0, t) for t in tg], np.uint32)
        a = sat["pssm%d_align" % k]
        assert np.array_equal(ctx.sw_score(prof, pairs), a[:, 0]), k
        ends = ctx.sw_score_endpos(prof, pairs)
        assert np.array_equal(np.stack([ends[f] for f in ("score", "qend", "dbend", "word")], 1), a[:, [0, 2, 4, 5]]), k
        aln = ctx.sw_align(prof, pairs)
        assert np.array_equal(np.stack([aln[f] for f in ALN_FIELDS], 1), a), (k, aln, a)
        out, bts = ctx.sw_backtrace(prof, [cons], pairs, aln)
        for i in range(len(tg)):
            assert out["ok"][i] == 1 and bts[i] == sat["pssm%d_bt" % k][i].decode(), (k, i)
            assert out["identical"][i] == sat["pssm%d_ident" % k][i], (k, i)


def _align_inputs(sat):
    qs = [_seq(sat["aln_qdata"], sat["aln_qoff"], i) for i in range(len(sat["aln_qoff"]) - 1)]
    ho = sat["aln_hit_off"]
    lists = [sat["aln_hits"][int(ho[i]):int(ho[i + 1])] for i in range(len(qs))]
    return qs, lists


def _align_params(kw):
    from mmseqs2_b200 import alignment as al
    kw = dict(kw)
    add_bt, comp = kw.pop("add_backtrace", True), kw.pop("compress", True)
    return al.AlignParams(**kw), add_bt, comp


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sat_mode2", "sat_mode1_cov", "sat_identity"])
def test_device_align_batch_records(sat, ctx, submat, name):
    """b200_align_batch: saturated and ordinary hits in one batch give the reference's `align` records"""
    from mmseqs2_b200 import alignment as al
    ctx.load_db(sat["tdata"], sat["toff"].astype(np.uint64), 21)
    qs, lists = _align_inputs(sat)
    par, add_bt, comp = _align_params(_maker().ALIGN_CONFIGS[name])
    ev = al.EvalueParams.defaults("blosum62.out", 11, 1, int(sat["toff"][-1]))
    res, pool, _ = al.align_batch(ctx, submat, qs, lists, par, ev, query_keys=7000 + np.arange(len(qs)), target_keys=sat["target_keys"])
    texts = sat["cfg_%s_text" % name]
    for qi in range(len(qs)):
        assert al.records(res[qi], pool, add_bt, comp) == bytes(texts[qi]), (name, qi)
    assert sum(len(r) for r in res) >= 20


@pytest.mark.gpu
def test_device_multi_align_batch_split(sat, ctx, submat):
    """the multi-device align batch over two contexts equals the single-context result and the reference's records"""
    from mmseqs2_b200 import MultiContext, alignment as al, load_library
    n = load_library().b200_device_count()
    qs, lists = _align_inputs(sat)
    par, add_bt, comp = _align_params(_maker().ALIGN_CONFIGS["sat_mode2"])
    ev = al.EvalueParams.defaults("blosum62.out", 11, 1, int(sat["toff"][-1]))
    keys = dict(query_keys=7000 + np.arange(len(qs)), target_keys=sat["target_keys"])
    ctx.load_db(sat["tdata"], sat["toff"].astype(np.uint64), 21)
    r1, p1, a1 = al.align_batch(ctx, submat, qs, lists, par, ev, **keys)
    m = MultiContext([0, 1] if n >= 2 else [0, 0])
    try:
        m.load_db(sat["tdata"], sat["toff"].astype(np.uint64), 21)
        r2, p2, a2 = al.align_batch(m, submat, qs, lists, par, ev, **keys)
    finally:
        m.close()
    assert a1 == a2
    for qi in range(len(qs)):
        got = al.records(r2[qi], p2, add_bt, comp)
        assert got == al.records(r1[qi], p1, add_bt, comp) == bytes(sat["cfg_sat_mode2_text"][qi]), qi
