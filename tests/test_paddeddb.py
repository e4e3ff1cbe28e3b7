"""Padded GPU sequence DB writer (`makepaddedseqdb`) and the repeat masker (Masker over tantan), include/b200_db.h, against files written
by the reference binary and values computed by oracle/_ref (tests/golden/make_paddeddb_golden.py).  Host code: no GPU needed."""
import importlib.util
import os

import numpy as np
import pytest

from mmseqs2_b200 import db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUFFIXES = ("", ".index", ".dbtype", "_h", "_h.index", "_h.dbtype", ".lookup", ".source")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(ROOT, "tests", "golden", "paddeddb_v1.npz"), allow_pickle=False)


@pytest.fixture(scope="module")
def alphabet():
    return np.load(os.path.join(ROOT, "tests", "golden", "blosum62.npz"))["alphabet"].tobytes()


def _param_sets():
    spec = importlib.util.spec_from_file_location("make_paddeddb_golden", os.path.join(ROOT, "tests", "golden", "make_paddeddb_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m.PARAM_SETS


def _write_src(gold, tmp_path):
    src = str(tmp_path / "T")
    for suf in SUFFIXES:
        if "src" + suf in gold.files:
            open(src + suf, "wb").write(gold["src" + suf].tobytes())
    return src


@pytest.mark.parametrize("name", ["default", "nomask", "lower_runs", "prob05_nolookup"])
def test_writer_reproduces_the_reference_files(gold, alphabet, tmp_path, name):
    src = _write_src(gold, tmp_path)
    dst = str(tmp_path / ("P_" + name))
    db.make_padded_db(src, dst, alphabet, gold["lr"], threads=3, **_param_sets()[name][1])
    for suf in SUFFIXES:
        key = name + suf
        assert os.path.exists(dst + suf) == (key in gold.files), suf
        if key in gold.files:
            assert open(dst + suf, "rb").read() == gold[key].tobytes(), suf
    # one thread writes the same files
    db.make_padded_db(src, dst + "_1", alphabet, gold["lr"], threads=1, **_param_sets()[name][1])
    assert open(dst + "_1", "rb").read() == gold[name].tobytes()


def test_writer_layout_properties(gold):
    """what Marv::loadDb relies on: 4-byte aligned entries in ascending length, index length = L + 2, dbtype carries the GPU flag"""
    idx = np.array([[int(x) for x in l.split()] for l in gold["default.index"].tobytes().decode().splitlines()], np.int64)
    assert np.array_equal(idx[:, 0], np.arange(len(idx))) and np.all(idx[:, 1] % 4 == 0) and np.all(np.diff(idx[:, 2]) >= 0)
    assert np.array_equal(np.diff(idx[:, 1]), ((idx[:-1, 2] - 2 + 3) // 4) * 4)
    ty = int(np.frombuffer(gold["default.dbtype"].tobytes(), np.int32)[0])
    assert (ty >> 16) & 0x7FFE == 8 and ty & 0xffff == 0


def test_writer_on_a_compressed_source(gold, alphabet, tmp_path, ref):
    """a source DB written with `createdb --compressed 1` gives the same padded DB (the reader inflates it)"""
    src = _write_src(gold, tmp_path)
    d, h = db.DB(src), db.DB(src + "_h")
    csrc = str(tmp_path / "C")
    ref.db_write(csrc, 0, [d.key(i) for i in range(len(d))], [d.data(i) for i in range(len(d))], compressed=True)
    ref.db_write(csrc + "_h", 12, [h.key(i) for i in range(len(h))], [h.data(i) for i in range(len(h))], compressed=True)
    d.close(); h.close()
    dst = str(tmp_path / "PC")
    db.make_padded_db(csrc, dst, alphabet, gold["lr"], write_lookup=0)
    for suf in ("", ".index", ".dbtype", "_h", "_h.index", "_h.dbtype"):
        assert open(dst + suf, "rb").read() == gold["default" + suf].tobytes(), suf


def test_tantan_posteriors_bitwise(gold):
    for i, s in enumerate(gold["seq_text"]):
        L = len(s)
        p = db.tantan_probabilities(gold["seq_codes"][i, :L], gold["lr"])
        assert np.array_equal(p.view(np.uint32), gold["seq_probs"][i, :L].view(np.uint32)), i


def test_mask_sequence_modes(gold):
    for k, (tt, pr, lc, nr) in enumerate(gold["seq_mask_modes"]):
        for i, s in enumerate(gold["seq_text"]):
            L = len(s)
            m, n = db.mask_sequence(gold["seq_codes"][i, :L], bytes(s), gold["lr"], bool(tt), float(pr), bool(lc), int(nr))
            assert np.array_equal(m, gold["seq_masked"][k, i, :L]), (k, i)
            if nr == 0:          # with run masking the reference counts letters that were X already; only the codes are the contract
                assert n == int(gold["seq_mask_counts"][k, i]), (k, i)


def test_masker_against_live_reference(ref):
    lr = ref.tantan_matrix()
    rng = np.random.default_rng(5)
    for t in range(12):
        L = int(rng.integers(1, 1500))
        if t % 3 == 0:
            s = rng.integers(0, 21, L)
        elif t % 3 == 1:
            s = np.resize(rng.integers(0, 20, int(rng.integers(1, 60))), L)
            hit = rng.random(L) < 0.08
            s[hit] = rng.integers(0, 20, int(hit.sum()))
        else:
            s = rng.integers(0, 20, L)
            a = int(rng.integers(0, L))
            s[a:a + 60] = rng.integers(0, 2, len(s[a:a + 60]))
        s = np.ascontiguousarray(s, np.uint8)
        exp = ref.tantan_probabilities(s)
        assert np.array_equal(db.tantan_probabilities(s, lr).view(np.uint32), exp.view(np.uint32)), t


def test_writer_refuses_bad_input(gold, alphabet, tmp_path):
    with pytest.raises(db.B200Error):
        db.make_padded_db(str(tmp_path / "missing"), str(tmp_path / "o"), alphabet, gold["lr"])
    src = _write_src(gold, tmp_path)
    with pytest.raises(db.B200Error):
        db.make_padded_db(src, str(tmp_path / "o"), alphabet, None, mask=1)          # masking without the matrix
    os.remove(src + "_h")
    with pytest.raises(db.B200Error):
        db.make_padded_db(src, str(tmp_path / "o"), alphabet, gold["lr"])
