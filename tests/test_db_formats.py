"""DB triple (data / .index / .dbtype), letter mapping and the `align` module over DB files (include/b200_db.h), against files
written by the reference's own DBWriter and tables of its BaseMatrix (tests/golden/make_align_golden.py)."""
import os

import numpy as np
import pytest

from mmseqs2_b200 import alignment as al
from mmseqs2_b200 import db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(ROOT, "tests", "golden", "align_v1.npz"), allow_pickle=False)


def _entries(gold):
    return [bytes(e)[:int(n)] if n else b"" for e, n in zip(gold["dbw_entries"], gold["dbw_entry_len"])]


def test_letter_mapping_equals_reference_tables(gold, blosum):
    b = np.load(os.path.join(ROOT, "tests", "golden", "blosum62.npz"))
    assert np.array_equal(db.aa2num_table(bytes(b["alphabet"]))[:255], gold["aa2num_aa"])
    assert np.array_equal(db.aa2num_table(bytes(b["nucl_alphabet"]), nucleotide=True)[:255], gold["aa2num_nt"])


def test_writer_produces_the_reference_files(gold, tmp_path):
    path = str(tmp_path / "w")
    db.write_db(path, 7, gold["dbw_keys"], _entries(gold))
    for suf, name in (("", "data"), (".index", "index"), (".dbtype", "dbtype")):
        assert open(path + suf, "rb").read() == gold["dbw_file_" + name].tobytes(), name


def test_reader_on_reference_files(gold, tmp_path):
    path = str(tmp_path / "r")
    for suf, name in (("", "data"), (".index", "index"), (".dbtype", "dbtype")):
        open(path + suf, "wb").write(gold["dbw_file_" + name].tobytes())
    d = db.DB(path)
    order = np.argsort(gold["dbw_keys"], kind="stable")
    ents = _entries(gold)
    assert len(d) == len(order) and d.dbtype == 7
    for i, k in enumerate(order):
        assert d.key(i) == int(gold["dbw_keys"][k]) and d.data(i) == ents[k] and d.entry_len(i) == len(ents[k]) + 1
        assert d.id_of(int(gold["dbw_keys"][k])) == i
    assert d.id_of(999) == -1
    d.close()
    # split data files <name>.0, <name>.1 read as one (FileUtil::findDatafiles)
    blob = gold["dbw_file_data"].tobytes()
    sp = str(tmp_path / "split")
    open(sp + ".0", "wb").write(blob[:300]); open(sp + ".1", "wb").write(blob[300:])
    open(sp + ".index", "wb").write(gold["dbw_file_index"].tobytes())
    d2 = db.DB(sp)
    assert [d2.data(i) for i in range(len(d2))] == [ents[k] for k in order] and d2.dbtype == -1
    d2.close()
    with pytest.raises(db.B200Error):
        db.DB(str(tmp_path / "missing"))


def test_reader_writer_against_live_reference(tmp_path, ref):
    rng = np.random.default_rng(8)
    keys = rng.permutation(5000)[:100].astype(np.uint32)
    ents = [bytes(rng.integers(32, 127, int(rng.integers(0, 300))).astype(np.uint8)) + b"\n" for _ in keys]
    ref.db_write(str(tmp_path / "r"), 0, keys, ents)
    db.write_db(str(tmp_path / "m"), 0, keys, ents)
    for suf in ("", ".index", ".dbtype"):
        assert open(str(tmp_path / "r") + suf, "rb").read() == open(str(tmp_path / "m") + suf, "rb").read(), suf
    k, l, o, ty = ref.db_read(str(tmp_path / "m"))
    d = db.DB(str(tmp_path / "r"))
    assert [d.key(i) for i in range(len(d))] == list(k) and [d.data(i) for i in range(len(d))] == o and d.dbtype == ty
    d.close()


def _compressed_gold():
    g = np.load(os.path.join(ROOT, "tests", "golden", "compressed_db_v1.npz"), allow_pickle=False)
    ents = [bytes(e)[:int(n)] for e, n in zip(g["entries"], g["entry_len"])]
    return g, ents


def test_reader_on_reference_compressed_files(tmp_path):
    """zstd-compressed DB written by the reference's DBWriter (tests/golden/make_compressed_db_golden.py): entries below 60 bytes
    are stored raw, the others as one zstd frame each; the reader hands out the plain text and the dbtype without bit 31"""
    g, ents = _compressed_gold()
    path = str(tmp_path / "c")
    for suf, name in (("", "data"), (".index", "index"), (".dbtype", "dbtype")):
        open(path + suf, "wb").write(g["file_" + name].tobytes())
    assert int(np.frombuffer(g["file_dbtype"].tobytes(), np.int32)[0]) < 0          # bit 31 set on disk
    d = db.DB(path)
    order = np.argsort(g["keys"], kind="stable")
    assert len(d) == len(ents) and d.dbtype == int(g["reader_dbtype"]) & 0x7fffffff
    for i, k in enumerate(order):
        assert d.key(i) == int(g["keys"][k]) and d.data(i) == ents[k] and d.entry_len(i) == len(ents[k]) + 1, i
    d.close()
    # a truncated frame and an index length that disagrees with the frame are refused, not misread
    blob = bytearray(g["file_data"].tobytes())
    idx = [l.split(b"\t") for l in g["file_index"].tobytes().splitlines()]
    big = max(idx, key=lambda f: int(f[2]))
    bad = str(tmp_path / "bad")
    blob2 = bytearray(blob); blob2[int(big[1]) + 4 + 20] ^= 0x5a
    open(bad, "wb").write(bytes(blob2)); open(bad + ".index", "wb").write(g["file_index"].tobytes()); open(bad + ".dbtype", "wb").write(g["file_dbtype"].tobytes())
    with pytest.raises(db.B200Error):
        db.DB(bad)
    open(bad, "wb").write(bytes(blob))
    open(bad + ".index", "wb").write(b"\n".join(b"\t".join([f[0], f[1], str(int(f[2]) + (7 if f is big else 0)).encode()]) for f in idx) + b"\n")
    with pytest.raises(db.B200Error):
        db.DB(bad)


def test_compressed_reader_against_live_reference(tmp_path, ref):
    rng = np.random.default_rng(9)
    keys = rng.permutation(5000)[:50].astype(np.uint32)
    aa = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", np.uint8)
    ents = [bytes(aa[rng.integers(0, 20, int(rng.integers(0, 900)))]) + b"\n" for _ in keys]
    ref.db_write(str(tmp_path / "c"), 0, keys, ents, compressed=True)
    k, l, o, ty = ref.db_read(str(tmp_path / "c"))
    d = db.DB(str(tmp_path / "c"))
    assert [d.key(i) for i in range(len(d))] == list(k) and [d.data(i) for i in range(len(d))] == o
    assert [d.entry_len(i) for i in range(len(d))] == list(l)
    d.close()


@pytest.mark.gpu
def test_align_module_over_db_files(gold, ctx, submat, tmp_path):
    """query DB + target DB + prefilter DB (ASCII sequences, text records) -> alignment DB: the three output files equal the ones the
    reference's Matcher + DBWriter produce for the same lists (`align -a --threads 1`)"""
    ex = np.load(os.path.join(ROOT, "tests", "golden", "examples_v1.npz"))
    b = np.load(os.path.join(ROOT, "tests", "golden", "blosum62.npz"))
    letters = b["alphabet"]
    nq, nt = len(ex["qoff"]) - 1, len(ex["toff"]) - 1

    def ascii_entries(data, off, n):
        return [letters[data[int(off[i]):int(off[i + 1])]].tobytes() + b"\n" for i in range(n)]

    tkeys = gold["target_keys"]
    qkeys = 5000 + np.arange(nq)
    db.write_db(str(tmp_path / "target"), db.DBTYPE_AMINO_ACIDS, tkeys, ascii_entries(ex["tdata"], ex["toff"], nt))
    db.write_db(str(tmp_path / "query"), db.DBTYPE_AMINO_ACIDS, qkeys, ascii_entries(ex["qdata"], ex["qoff"], nq))
    ho = gold["hit_off"]
    pref = []
    for qi in range(nq):
        hits = np.zeros(int(ho[qi + 1] - ho[qi]), al.PREF_HIT_DTYPE)
        ids = gold["hit_targets"][int(ho[qi]):int(ho[qi + 1])]
        hits["seq_id"], hits["pref_score"], hits["diagonal"] = tkeys[ids], ex["ungapped"][qi][ids], 0
        pref.append(al.prefilter_hits_to_buffer(hits))
    db.write_db(str(tmp_path / "pref"), db.DBTYPE_PREFILTER_RES, qkeys, pref)
    n_aln, n_rec = db.align_db(ctx, submat, bytes(letters), str(tmp_path / "query"), str(tmp_path / "target"), str(tmp_path / "pref"),
                               str(tmp_path / "aln"), al.AlignParams(sw_mode=al.SCORE_COV_SEQID, eval_thr=1e-3), bucket_queries=16)
    for suf, name in (("", "data"), (".index", "index"), (".dbtype", "dbtype")):
        assert open(str(tmp_path / "aln") + suf, "rb").read() == gold["alndb_file_" + name].tobytes(), name
    assert n_aln == int(gold["cfg_default_a_naligned"].sum()) and n_rec == sum(bytes(t).count(b"\n") for t in gold["cfg_default_a_text"])


@pytest.mark.gpu
def test_prefilter_module_over_db_files_and_search(gold, ctx, submat, tmp_path):
    """`ungappedprefilter` on DB files: the prefilter DB equals the one built from the reference's own scores; then `align` on that DB
    runs end to end (search --prefilter-mode 1 without a reference process in the loop)"""
    ex = np.load(os.path.join(ROOT, "tests", "golden", "examples_v1.npz"))
    b = np.load(os.path.join(ROOT, "tests", "golden", "blosum62.npz"))
    letters = b["alphabet"]
    nq, nt = len(ex["qoff"]) - 1, len(ex["toff"]) - 1

    def ascii_entries(data, off, n):
        return [letters[data[int(off[i]):int(off[i + 1])]].tobytes() + b"\n" for i in range(n)]

    db.write_db(str(tmp_path / "target"), db.DBTYPE_AMINO_ACIDS, gold["target_keys"], ascii_entries(ex["tdata"], ex["toff"], nt))
    db.write_db(str(tmp_path / "query"), db.DBTYPE_AMINO_ACIDS, 5000 + np.arange(nq), ascii_entries(ex["qdata"], ex["qoff"], nq))
    n_hits = db.prefilter_db(ctx, submat, bytes(letters), str(tmp_path / "query"), str(tmp_path / "target"), str(tmp_path / "pref"),
                             bucket_queries=7)
    for suf, name in (("", "data"), (".index", "index"), (".dbtype", "dbtype")):
        assert open(str(tmp_path / "pref") + suf, "rb").read() == gold["prefdb_file_" + name].tobytes(), name
    assert n_hits == gold["prefdb_file_data"].tobytes().count(b"\n")
    n_aln, n_rec = db.align_db(ctx, submat, bytes(letters), str(tmp_path / "query"), str(tmp_path / "target"), str(tmp_path / "pref"),
                               str(tmp_path / "aln"), al.AlignParams(sw_mode=al.SCORE_COV_SEQID, eval_thr=1e-3))
    res = db.DB(str(tmp_path / "aln"))
    assert len(res) == nq and res.dbtype == db.DBTYPE_ALIGNMENT_RES and n_aln == n_hits
    assert sum(res.data(i).count(b"\n") for i in range(nq)) == n_rec > 100
    res.close()
