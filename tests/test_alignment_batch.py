"""The batched align step (include/b200_alignment.h): E-value statistics, record formats and -- on the GPU -- whole alignment-DB
entries, against fixtures written by the reference's own EvalueComputation / Matcher / QueryMatcher code
(tests/golden/make_align_golden.py).  Text is compared byte for byte, doubles bit for bit."""
import os

import numpy as np
import pytest

from mmseqs2_b200 import alignment as al

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(ROOT, "tests", "golden", "align_v1.npz"))


@pytest.fixture(scope="module")
def ex():
    return np.load(os.path.join(ROOT, "tests", "golden", "examples_v1.npz"))


def _params(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_align_golden_cfg", os.path.join(ROOT, "tests", "golden", "align_configs.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m.CONFIGS[name]


def _nucl_params(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_align_golden_cfg", os.path.join(ROOT, "tests", "golden", "align_configs.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m.NUCL_CONFIGS[name]


def _align_params(kw):
    kw = dict(kw)
    kw.pop("add_backtrace", None); kw.pop("compress", None)
    if "max_reject" in kw:
        kw["max_rejected"] = kw.pop("max_reject")
    return al.AlignParams(**kw)


# ---- CPU: statistics and formats ----------------------------------------------------------------------------------------
def test_evalue_and_bitscore_bit_exact(gold):
    g = gold["evalue_grid"]
    for s, ql, db, ev, bits in g:
        p = al.EvalueParams.defaults("blosum62.out", 11, 1, int(db))
        assert p.evalue(s, ql) == ev, (s, ql, db)
        assert p.bit_score(s) == bits, (s, db)


def test_evalue_defaults_error_path():
    with pytest.raises(al.B200Error):
        al.EvalueParams.defaults("blosum62.out", 10, 2, 1000)     # the reference would run ALP here
    assert al.EvalueParams.defaults("nucleotide.out", 5, 2, 10 ** 9).evalue(60, 150) > 0
    assert al.EvalueParams.defaults("blosum62.out", 0, 0, 10 ** 6, gapped=False).bit_score(50) > 0


def test_result_to_buffer_matches_reference_text(gold):
    cases, bts, texts = gold["record_cases"], gold["record_case_bt"], gold["record_case_text"]
    k = 0
    for c, bt in zip(cases, bts):
        r = np.zeros(1, al.RESULT_DTYPE)[0]
        r["db_key"], r["score"], r["seq_id"], r["eval"] = int(c[0]), int(c[1]), np.float32(c[2]), c[3]
        r["q_start"], r["q_end"], r["q_len"], r["db_start"], r["db_end"], r["db_len"] = [int(x) for x in c[4:10]]
        for add_bt, comp in ((False, True), (True, True), (True, False)):
            assert al.result_to_buffer(r, bytes(bt), add_bt, comp) == bytes(texts[k]), (c, add_bt, comp)
            k += 1


def test_prefilter_records_round_trip(gold):
    hits = al.parse_prefilter_hits(bytes(gold["pref_entry"]))
    assert np.array_equal(hits["seq_id"], gold["pref_ids"])
    assert np.array_equal(hits["pref_score"], gold["pref_scores"])
    assert np.array_equal(hits["diagonal"], gold["pref_diags"])
    assert al.prefilter_hits_to_buffer(hits) == bytes(gold["pref_text"])
    assert len(al.parse_prefilter_hits(b"")) == 0


def test_against_live_reference_when_present(ref):
    """random statistics / records against the reference's own code (the `ref` fixture)"""
    rng = np.random.default_rng(11)
    for _ in range(150):
        s = int(rng.integers(1, 3000)); ql = int(rng.integers(1, 5000)); db = int(rng.integers(1, 10 ** 10))
        p = al.EvalueParams.defaults("blosum62.out", 11, 1, db)
        assert p.evalue(s, ql) == ref.evalue(11, 1, db, s, ql)
        assert p.bit_score(s) == ref.bit_score(11, 1, db, s)
    for _ in range(100):
        r = np.zeros(1, al.RESULT_DTYPE)[0]
        sid = np.float32(rng.choice([rng.random(), 1.0, 0.0, 0.1, 0.01, 0.099999, 0.00999]))
        ev = float(10.0 ** rng.uniform(-200, 5))
        vals = [int(x) for x in rng.integers(-1, 70000, 6)]
        bt = bytes(rng.choice(list(b"MID"), int(rng.integers(0, 60))).astype(np.uint8))
        r["db_key"], r["score"], r["seq_id"], r["eval"] = int(rng.integers(0, 2 ** 32)), int(rng.integers(-5, 5000)), sid, ev
        r["q_start"], r["q_end"], r["q_len"], r["db_start"], r["db_end"], r["db_len"] = vals
        for add_bt, comp in ((False, True), (True, True), (True, False)):
            want = ref.result_to_buffer(int(r["db_key"]), int(r["score"]), float(sid), ev, *vals, backtrace=bt, add_backtrace=add_bt,
                                        compress=comp)
            assert al.result_to_buffer(r, bt, add_bt, comp) == want


# ---- GPU: whole alignment-DB entries ---------------------------------------------------------------------------------------
def _seqs(d, o):
    return [d[int(o[i]):int(o[i + 1])] for i in range(len(o) - 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["default_a", "mode1_cov", "mode0", "strict", "target_cov_nobias", "len_modes"])
def test_alignment_entries_equal_reference(gold, ex, ctx, submat, name):
    kw = _params(name)
    qs = _seqs(ex["qdata"], ex["qoff"])
    ctx.load_db(ex["tdata"], ex["toff"].astype(np.uint64), 21)
    ho = gold["hit_off"]
    lists = [gold["hit_targets"][int(ho[i]):int(ho[i + 1])] for i in range(len(qs))]
    ev = al.EvalueParams.defaults("blosum62.out", 11, 1, int(gold["db_residues"]))
    res, pool, n_aln = al.align_batch(ctx, submat, qs, lists, _align_params(kw), ev, query_keys=5000 + np.arange(len(qs)),
                                      target_keys=gold["target_keys"])
    texts = gold["cfg_%s_text" % name]
    for qi in range(len(qs)):
        got = al.records(res[qi], pool, kw.get("add_backtrace", True), kw.get("compress", True))
        assert got == bytes(texts[qi]), (name, qi)
    assert n_aln == int(gold["cfg_%s_naligned" % name].sum())
    assert sum(len(r) for r in res) > 50


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_identity_hits(gold, ctx, submat, mode):
    so = gold["self_off"]
    ctx.load_db(gold["self_data"], so.astype(np.uint64), 21)
    keys = gold["self_keys"]
    qs = _seqs(gold["self_data"], so)[:12]
    lists = [np.array([qi] + list(range(12, 72)) + [(qi + 1) % 12], np.uint32) for qi in range(12)]
    ev = al.EvalueParams.defaults("blosum62.out", 11, 1, int(so[-1]))
    par = al.AlignParams(sw_mode=mode, eval_thr=1e-3, include_identity=True)
    res, pool, _ = al.align_batch(ctx, submat, qs, lists, par, ev, query_keys=keys[:12], target_keys=keys)
    texts = gold["self_mode%d_text" % mode]
    for qi in range(12):
        assert al.records(res[qi], pool, mode == 2, True) == bytes(texts[qi]), (mode, qi)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["nucl_default", "nucl_strict", "nucl_loose"])
def test_nucleotide_alignment_entries_equal_reference(gold, ctx, name):
    """the BandedNucleotideAligner branch of getSWResult through b200_align_batch_nucl: forward and reverse-strand hits"""
    kw = _nucl_params(name)
    nv = np.load(os.path.join(ROOT, "tests", "golden", "nucl_v1.npz"))
    ctx.load_db(nv["tdata"], nv["toff"].astype(np.uint64), 5)
    ro = gold["nucl_read_off"]
    reads = [gold["nucl_reads"][int(ro[i]):int(ro[i + 1])] for i in range(len(ro) - 1)]
    per = 4
    lists = [gold["nucl_hit_targets"][per * i:per * (i + 1)] for i in range(len(reads))]
    diags = [gold["nucl_hit_diags"][per * i:per * (i + 1)] for i in range(len(reads))]
    revs = [gold["nucl_hit_rev"][per * i:per * (i + 1)] for i in range(len(reads))]
    ev = al.EvalueParams.defaults("nucleotide.out", 5, 2, int(nv["toff"][-1]))
    par = _align_params(dict(kw, gap_open=5, gap_extend=2))
    res, pool, n_aln = al.align_batch_nucl(ctx, reads, lists, diags, revs, par, ev, zdrop=40, query_keys=900 + np.arange(len(reads)),
                                           target_keys=gold["nucl_target_keys"])
    texts = gold["cfg_%s_text" % name]
    for k in range(len(reads)):
        got = al.records(res[k], pool, kw.get("add_backtrace", True), kw.get("compress", True))
        assert got == bytes(texts[k]), (name, k, got, bytes(texts[k]))
    assert n_aln == int(gold["cfg_%s_naligned" % name].sum())
    assert sum(len(r) for r in res) > 20
    if name == "nucl_default":
        assert sum(1 for k in range(len(reads)) if revs[k][0] and len(res[k])) >= 40      # reverse-strand hits are found


@pytest.mark.gpu
def test_align_batch_edge_cases(ex, ctx, submat):
    ctx.load_db(ex["tdata"], ex["toff"].astype(np.uint64), 21)
    qs = _seqs(ex["qdata"], ex["qoff"])[:3]
    ev = al.EvalueParams.defaults("blosum62.out", 11, 1, int(ex["toff"][-1]))
    # empty hit lists, an empty batch and a query without hits next to one with hits
    res, pool, n = al.align_batch(ctx, submat, qs, [[], [], []], al.AlignParams(), ev)
    assert [len(r) for r in res] == [0, 0, 0] and n == 0
    res, _, n = al.align_batch(ctx, submat, qs, [[], [0, 1, 2, 3], []], al.AlignParams(sw_mode=0, eval_thr=1e9), ev)
    assert len(res[0]) == 0 and len(res[2]) == 0 and n == 4
    with pytest.raises(al.B200Error):
        al.align_batch(ctx, submat, qs, [[10 ** 6], [], []], al.AlignParams(), ev)        # target id out of range
    with pytest.raises(al.B200Error):
        al.align_batch(ctx, submat, qs, [[0], [], []], al.AlignParams(sw_mode=3), ev)      # unknown mode
