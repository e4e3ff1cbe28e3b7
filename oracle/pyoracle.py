"""oracle/pyoracle.py -- TEST INFRASTRUCTURE: ctypes access to the CPU checker libraries.

  Oracle()   -> oracle/liboracle.so          (C restatement, oracle/oracle.c)
  Ref()      -> oracle/_ref/libmmseqs_ref.so (the reference's own sources compiled in place; optional)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libmmseqs_ref.so")

_vp = ctypes.c_void_p


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def build(with_ref=True):
    """Compile the checker(s).  The reference library is only (re)built when /root/reference exists."""
    subprocess.check_call(["make", "-s", "-C", HERE])
    if with_ref and os.path.isdir("/root/reference"):
        subprocess.check_call(["make", "-s", "-j8", "-C", HERE, "ref"])


def pack_targets(seqs):
    """list of uint8 arrays -> (concatenated residues, int64 offsets[n+1]) as SequenceLookup lays them out."""
    off = np.zeros(len(seqs) + 1, np.int64)
    if len(seqs):
        off[1:] = np.cumsum([len(s) for s in seqs])
    data = np.concatenate(seqs).astype(np.uint8) if len(seqs) else np.zeros(0, np.uint8)
    return np.ascontiguousarray(data), off


class Oracle:
    def __init__(self, mat, pback):
        if not os.path.exists(ORACLE_SO):
            build(with_ref=False)
        self.lib = ctypes.CDLL(ORACLE_SO)
        self.mat = np.ascontiguousarray(mat, np.int16)
        self.pback = np.ascontiguousarray(pback, np.float64)
        self.A = int(self.mat.shape[0])
        self.lib.orc_ssw_bias.restype = ctypes.c_int
        self.lib.orc_ungapped_alignment.restype = ctypes.c_int
        self.lib.orc_diag_score.restype = ctypes.c_int

    def comp_bias(self, q, scale=1.0):
        q = np.ascontiguousarray(q, np.uint8)
        out = np.zeros(len(q), np.float32)
        self.lib.orc_comp_bias(_p(self.mat), _p(self.pback), self.A, _p(q), len(q), ctypes.c_float(scale), _p(out))
        return out

    def round_bias_ssw(self, f):
        f = np.ascontiguousarray(f, np.float32)
        out = np.zeros(len(f), np.int8)
        self.lib.orc_round_bias_ssw(_p(f), len(f), _p(out))
        return out

    def round_bias_diag(self, f):
        f = np.ascontiguousarray(f, np.float32)
        out = np.zeros(len(f), np.int8)
        self.lib.orc_round_bias_diag(_p(f), len(f), _p(out))
        return out

    def query_cb(self, q, comp_bias=True):
        """int8 composition bias and profile bias constant exactly as ssw_init derives them."""
        q = np.ascontiguousarray(q, np.uint8)
        cb = self.round_bias_ssw(self.comp_bias(q)) if comp_bias else np.zeros(len(q), np.int8)
        bias = self.lib.orc_ssw_bias(_p(self.mat), self.A, _p(cb), len(q), 1 if comp_bias else 0)
        return cb, int(bias)

    def ungapped(self, q, cb, bias, tdata, toff, nthreads=8, fast=False):
        q = np.ascontiguousarray(q, np.uint8)
        n = len(toff) - 1
        out = np.zeros(n, np.int32)
        (self.lib.orc_ungapped_alignment_batch_fast if fast else self.lib.orc_ungapped_alignment_batch)(_p(self.mat), self.A, _p(q), len(q), _p(cb), bias, _p(tdata), _p(toff),
                                              ctypes.c_int64(n), _p(out), nthreads)
        return out

    def sw_score_endpos(self, q, cb, bias, tdata, toff, go=11, ge=1, nthreads=8):
        q = np.ascontiguousarray(q, np.uint8)
        n = len(toff) - 1
        out = np.zeros((n, 4), np.int32)
        self.lib.orc_sw_score_endpos_batch(_p(self.mat), self.A, _p(q), len(q), _p(cb), bias, _p(tdata), _p(toff),
                                           ctypes.c_int64(n), go, ge, _p(out), nthreads)
        return out

    def sw_align(self, q, cb, bias, tdata, toff, go=11, ge=1, gate=None, nthreads=8):
        q = np.ascontiguousarray(q, np.uint8)
        n = len(toff) - 1
        out = np.zeros((n, 6), np.int32)
        g = None if gate is None else np.ascontiguousarray(gate, np.uint8)
        self.lib.orc_sw_align_batch(_p(self.mat), self.A, _p(q), len(q), _p(cb), bias, _p(tdata), _p(toff),
                                    ctypes.c_int64(n), go, ge, _p(g), _p(out), nthreads)
        return out

    def backtrace(self, q, cb, t, aln, go=11, ge=1):
        """aln = (score, qstart, qend, dbstart, dbend, ...) -> (backtrace string or None on trace-back error, identical)"""
        q = np.ascontiguousarray(q, np.uint8); t = np.ascontiguousarray(t, np.uint8)
        buf = ctypes.create_string_buffer(len(q) + len(t) + 8)
        ids = ctypes.c_int32()
        self.lib.orc_sw_backtrace.restype = ctypes.c_int
        n = self.lib.orc_sw_backtrace(_p(self.mat), self.A, _p(q), _p(cb), _p(t), int(aln[1]), int(aln[2]), int(aln[3]), int(aln[4]),
                                      int(aln[0]), go, ge, buf, len(buf), ctypes.byref(ids))
        return (buf.value.decode() if n >= 0 else None), ids.value

    def rescore_diagonal(self, q_ascii, t_ascii, diagonal_u16, asciimat, mode):
        """DistanceCalculator::computeUngappedAlignment restated (8f row 3 groundwork) -> 6 fields"""
        out = np.zeros(6, np.int64)
        self.lib.orc_rescore_diagonal(q_ascii, len(q_ascii), t_ascii, len(t_ascii), ctypes.c_uint16(diagonal_u16 & 0xffff), _p(asciimat), mode,
                                      _p(out))
        return out

    def diag(self, q, cb4, tdata, toff, hit_ids, hit_diags):
        q = np.ascontiguousarray(q, np.uint8)
        ids = np.ascontiguousarray(hit_ids, np.uint32)
        dg = np.ascontiguousarray(hit_diags, np.uint16)
        counts = np.zeros(len(ids), np.uint8)
        raw = np.zeros(len(ids), np.int32)
        self.lib.orc_diag_score_batch(_p(self.mat), self.A, _p(q), len(q), _p(cb4), _p(tdata), _p(toff), _p(ids),
                                      _p(dg), ctypes.c_int64(len(ids)), _p(counts), _p(raw))
        return counts, raw


NUCL_KMAT = None


def ksw_mat(nmat):
    """5x5 int8 matrix BandedNucleotideAligner hands to ksw2 (BandedNucleotideAligner.cpp:29-34)"""
    return np.ascontiguousarray(nmat, np.int8)


class KswOracle:
    """oracle/oracle_ksw.c"""

    def __init__(self, nucl_mat):
        if not os.path.exists(ORACLE_SO):
            build(with_ref=False)
        self.lib = ctypes.CDLL(ORACLE_SO)
        self.mat = np.ascontiguousarray(nucl_mat, np.int8)

    def extz2(self, q, t, gapo=5, gape=2, w=64, zdrop=40, flag=0x41, cap=None):
        q = np.ascontiguousarray(q, np.uint8); t = np.ascontiguousarray(t, np.uint8)
        ez = np.zeros(10, np.int32)
        cap = cap or (len(q) + len(t) + 4)
        cg = np.zeros(cap, np.uint32)
        self.lib.orc_ksw_extz2(len(q), _p(q), len(t), _p(t), 5, _p(self.mat), gapo, gape, w, zdrop, flag, _p(ez), _p(cg), cap)
        return ez, cg[:ez[9]]

    def align(self, q, t, diagonal, gapo=5, gape=2, zdrop=40):
        q = np.ascontiguousarray(q, np.uint8); t = np.ascontiguousarray(t, np.uint8)
        out = np.zeros(7, np.int32)
        cap = len(q) + len(t) + 8
        cg = np.zeros(cap, np.uint32)
        bt = ctypes.create_string_buffer(cap)
        self.lib.orc_banded_nucl_align(_p(q), len(q), _p(t), len(t), ctypes.c_uint16(int(diagonal) & 0xffff), _p(self.mat), _p(self.mat),
                                       gapo, gape, zdrop, _p(out), _p(cg), cap, bt)
        return out, cg[:out[6]], bt.value.decode()


class Ref:
    """The reference's own hot-path code (oracle/_ref).  available() is False on boxes without the build."""

    @staticmethod
    def available():
        return os.path.exists(REF_SO)

    def __init__(self):
        self.lib = ctypes.CDLL(REF_SO)
        self.lib.ref_init()
        self.lib.ref_evalue.restype = ctypes.c_double

    def matrix(self, nucl=False):
        A = self.lib.ref_alphabet_size(1 if nucl else 0)
        mat = np.zeros((A, A), np.int16)
        pb = np.zeros(A, np.float64)
        n2a = ctypes.create_string_buffer(A)
        self.lib.ref_get_matrix(1 if nucl else 0, _p(mat), _p(pb), n2a)
        return mat, pb, n2a.raw.decode()

    def evalue(self, go, ge, db_residues, score, qlen):
        return float(self.lib.ref_evalue(go, ge, ctypes.c_int64(db_residues), ctypes.c_double(score), ctypes.c_double(qlen), None))

    def evalue_bits(self, go, ge, db_residues, score, qlen):
        """-> (E-value, bit score) of the gapped statistics"""
        b = ctypes.c_double(0)
        e = self.lib.ref_evalue(go, ge, ctypes.c_int64(db_residues), ctypes.c_double(score), ctypes.c_double(qlen), ctypes.byref(b))
        return float(e), float(b.value)

    def evalue_bits_ungapped(self, db_residues, score, qlen):
        """-> (E-value, bit score) of the ungapped statistics rescorediagonal uses (EvalueComputation(dbResCount, subMat))"""
        self.lib.ref_evalue_ungapped.restype = ctypes.c_double
        b = ctypes.c_double(0)
        e = self.lib.ref_evalue_ungapped(ctypes.c_int64(db_residues), ctypes.c_double(score), ctypes.c_double(qlen), ctypes.byref(b))
        return float(e), float(b.value)

    def tantan_matrix(self):
        lr = np.zeros((21, 21), np.float64)
        self.lib.ref_tantan_matrix(_p(lr))
        return lr

    def tantan_probabilities(self, seq):
        s = np.ascontiguousarray(seq, np.uint8)
        out = np.zeros(len(s), np.float32)
        self.lib.ref_tantan_probabilities(_p(s), len(s), _p(out))
        return out

    # ---- `align` module at record level (ref_glue.cpp: ref_align_query) ----
    def align_query(self, q, qkey, tdata, toff, hit_idx, hit_keys, db_residues, comp_bias=True, comp_bias_scale=1.0, go=11, ge=1,
                    sw_mode=2, eval_thr=1e-3, cov_thr=0.0, cov_mode=0, seq_id_thr=0.0, aln_len_thr=0, seq_id_mode=0,
                    max_accept=0x7fffffff, max_reject=0x7fffffff, include_identity=False, add_backtrace=True, compress=True):
        """-> (records text, n getSWResult calls, n accepted)"""
        q = np.ascontiguousarray(q, np.uint8)
        hi = np.ascontiguousarray(hit_idx, np.uint32)
        hk = np.ascontiguousarray(hit_keys, np.uint32)
        to = np.ascontiguousarray(toff, np.int64)
        cap = 4096 + len(hi) * 4096
        out = ctypes.create_string_buffer(cap)
        na = ctypes.c_int64(0); nacc = ctypes.c_int64(0)
        self.lib.ref_align_query.restype = ctypes.c_int64
        n = self.lib.ref_align_query(_p(q), len(q), ctypes.c_uint32(qkey), 1 if comp_bias else 0, ctypes.c_float(comp_bias_scale),
                                     _p(tdata), _p(to), _p(hi), _p(hk), ctypes.c_int64(len(hi)), ctypes.c_int64(db_residues), go, ge,
                                     sw_mode, ctypes.c_double(eval_thr), ctypes.c_float(cov_thr), cov_mode, ctypes.c_float(seq_id_thr),
                                     aln_len_thr, seq_id_mode, ctypes.c_uint32(max_accept), ctypes.c_uint32(max_reject),
                                     1 if include_identity else 0, 1 if add_backtrace else 0, 1 if compress else 0, out,
                                     ctypes.c_int64(cap), ctypes.byref(na), ctypes.byref(nacc))
        if n < 0:
            raise RuntimeError("ref_align_query: buffer too small")
        return out.raw[:n], int(na.value), int(nacc.value)

    def align_query_nucl(self, q, qkey, tdata, toff, hit_idx, hit_keys, hit_diag, hit_rev, db_residues, go=5, ge=2, zdrop=40,
                         eval_thr=1e-3, cov_thr=0.0, cov_mode=0, seq_id_thr=0.0, aln_len_thr=0, seq_id_mode=0, max_accept=0x7fffffff,
                         max_reject=0x7fffffff, include_identity=False, add_backtrace=True, compress=True):
        """nucleotide `align` entry of one read -> (records text, n getSWResult calls, n accepted)"""
        q = np.ascontiguousarray(q, np.uint8)
        hi = np.ascontiguousarray(hit_idx, np.uint32); hk = np.ascontiguousarray(hit_keys, np.uint32)
        hd = np.ascontiguousarray(hit_diag, np.int16)
        hr = None if hit_rev is None else np.ascontiguousarray(hit_rev, np.uint8)
        to = np.ascontiguousarray(toff, np.int64)
        cap = 4096 + len(hi) * 4096
        out = ctypes.create_string_buffer(cap)
        na = ctypes.c_int64(0); nacc = ctypes.c_int64(0)
        self.lib.ref_align_query_nucl.restype = ctypes.c_int64
        n = self.lib.ref_align_query_nucl(_p(q), len(q), ctypes.c_uint32(qkey), _p(tdata), _p(to), _p(hi), _p(hk), _p(hd), _p(hr),
                                          ctypes.c_int64(len(hi)), ctypes.c_int64(db_residues), go, ge, zdrop, ctypes.c_double(eval_thr),
                                          ctypes.c_float(cov_thr), cov_mode, ctypes.c_float(seq_id_thr), aln_len_thr, seq_id_mode,
                                          ctypes.c_uint32(max_accept), ctypes.c_uint32(max_reject), 1 if include_identity else 0,
                                          1 if add_backtrace else 0, 1 if compress else 0, out, ctypes.c_int64(cap), ctypes.byref(na),
                                          ctypes.byref(nacc))
        if n < 0:
            raise RuntimeError("ref_align_query_nucl: buffer too small")
        return out.raw[:n], int(na.value), int(nacc.value)

    # ---- DB triple through the reference's DBWriter / DBReader (ref_glue.cpp) ----
    def db_write(self, path, dbtype, keys, entries, compressed=False):
        keys = np.ascontiguousarray(keys, np.uint32)
        off = np.zeros(len(entries) + 1, np.int64)
        off[1:] = np.cumsum([len(e) for e in entries])
        blob = b"".join(entries) + b"\0"
        self.lib.ref_db_write_mode(path.encode(), int(dbtype), _p(keys), blob, _p(off), ctypes.c_int64(len(entries)),
                                   ctypes.c_int(1 if compressed else 0))

    def db_read(self, path, max_entries=1 << 16, cap=1 << 24):
        keys = np.zeros(max_entries, np.uint32); lens = np.zeros(max_entries, np.int64)
        data = ctypes.create_string_buffer(cap)
        used = ctypes.c_int64(0); ty = ctypes.c_int(0)
        self.lib.ref_db_read.restype = ctypes.c_int64
        n = self.lib.ref_db_read(path.encode(), _p(keys), _p(lens), data, ctypes.c_int64(cap), ctypes.byref(used), ctypes.byref(ty),
                                 ctypes.c_int64(max_entries))
        out, u = [], 0
        raw = ctypes.string_at(data, int(used.value))
        for i in range(n):
            out.append(raw[u:u + int(lens[i]) - 1]); u += int(lens[i]) - 1
        return keys[:n].copy(), lens[:n].copy(), out, int(ty.value)

    def gpuserver_query(self, shm_name, q, profile, cap=4096):
        """one request through the reference's GPUSharedMemory client side (ref_glue.cpp: ref_gpuserver_query) -> (ids, scores)"""
        q = np.ascontiguousarray(q, np.uint8); prof = np.ascontiguousarray(profile, np.int8)
        ids = np.zeros(cap, np.uint32); sc = np.zeros(cap, np.int32)
        self.lib.ref_gpuserver_query.restype = ctypes.c_int64
        n = self.lib.ref_gpuserver_query(shm_name.encode(), _p(q), len(q), _p(prof), prof.shape[0], _p(ids), _p(sc), ctypes.c_int64(cap))
        if n < 0:
            raise RuntimeError("server exited")
        return ids[:n].copy(), sc[:n].copy()

    def ascii_matrix(self):
        m = np.zeros((123, 123), np.int8)
        self.lib.ref_rescore_diagonal(None, 0, None, 0, ctypes.c_uint16(0), 0, None, _p(m))
        return m

    def rescore_diagonal(self, q_ascii, t_ascii, diagonal_u16, mode):
        out = np.zeros(6, np.int64)
        self.lib.ref_rescore_diagonal(q_ascii, len(q_ascii), t_ascii, len(t_ascii), ctypes.c_uint16(diagonal_u16 & 0xffff), mode, _p(out), None)
        return out

    def result_to_buffer(self, db_key, score, seq_id, evalue, qs, qe, ql, ds, de, dl, backtrace=b"", add_backtrace=False, compress=True):
        out = ctypes.create_string_buffer(1024 + 2 * len(backtrace))
        self.lib.ref_result_to_buffer.restype = ctypes.c_int64
        n = self.lib.ref_result_to_buffer(ctypes.c_uint32(db_key), score, ctypes.c_float(seq_id), ctypes.c_double(evalue), qs, qe, ql, ds, de,
                                          dl, backtrace, 1 if add_backtrace else 0, 1 if compress else 0, out)
        return out.raw[:n]

    def prefilter_roundtrip(self, entry):
        cap = entry.count(b"\n") + 4
        ids = np.zeros(cap, np.uint32); sc = np.zeros(cap, np.int32); dg = np.zeros(cap, np.uint16)
        out = ctypes.create_string_buffer(64 * cap)
        self.lib.ref_prefilter_roundtrip.restype = ctypes.c_int64
        n = self.lib.ref_prefilter_roundtrip(entry + b"\0", _p(ids), _p(sc), _p(dg), ctypes.c_int64(cap), out)
        return ids[:n], sc[:n], dg[:n], out.value

    # ---- profile (PSSM) queries (ref_glue.cpp: ref_profile_align / ref_profile_diag) ----
    def profile_align(self, pssm, consensus, tdata, toff, mode=1, go=11, ge=1, eval_thr=1e9, cov_mode=0, cov_thr=0.0, db_residues=None,
                      want_bt=False):
        """pssm: int8 [20][L] (Sequence::getAlignmentProfile layout).  mode -1: ungapped scores only.  -> (out[n][10], evalues, bts)"""
        pssm = np.ascontiguousarray(pssm, np.int8)
        cons = np.ascontiguousarray(consensus, np.uint8)
        to = np.ascontiguousarray(toff, np.int64)
        n = len(to) - 1
        out = np.zeros((n, 10), np.int32)
        ev = np.zeros(n, np.float64)
        stride = int(np.diff(to).max()) + pssm.shape[1] + 8 if want_bt else 0
        bt = ctypes.create_string_buffer(max(1, stride * n)) if want_bt else None
        self.lib.ref_profile_align(_p(pssm), _p(cons), pssm.shape[1], _p(tdata), _p(to), ctypes.c_int64(n), go, ge, mode,
                                   ctypes.c_double(eval_thr), cov_mode, ctypes.c_float(cov_thr),
                                   ctypes.c_int64(int(to[-1]) if db_residues is None else db_residues), _p(out), _p(ev), bt,
                                   ctypes.c_int64(stride))
        bts = [bt.raw[i * stride:(i + 1) * stride].split(b"\0", 1)[0] for i in range(n)] if want_bt else None
        return out, ev, bts

    def profile_diag(self, pssm, consensus, tdata, toff, ids, diags):
        pssm = np.ascontiguousarray(pssm, np.int8)
        cons = np.ascontiguousarray(consensus, np.uint8)
        to = np.ascontiguousarray(toff, np.int64)
        ids = np.ascontiguousarray(ids, np.uint32); dg = np.ascontiguousarray(diags, np.uint16)
        counts = np.zeros(len(ids), np.uint8); raw = np.zeros(len(ids), np.int32)
        self.lib.ref_profile_diag(_p(pssm), _p(cons), pssm.shape[1], _p(tdata), _p(to), ctypes.c_int64(len(to) - 1), _p(ids), _p(dg),
                                  ctypes.c_int64(len(ids)), _p(counts), _p(raw))
        return counts, raw

    def bit_score(self, go, ge, db_residues, score):
        b = ctypes.c_double(0)
        self.lib.ref_evalue(go, ge, ctypes.c_int64(db_residues), ctypes.c_double(score), ctypes.c_double(100.0), ctypes.byref(b))
        return float(b.value)

    def aa2num(self, nucl=False):
        t = np.zeros(256, np.uint8)
        self.lib.ref_aa2num(1 if nucl else 0, _p(t))
        return t

    def comp_bias(self, q, scale=1.0):
        q = np.ascontiguousarray(q, np.uint8)
        out = np.zeros(len(q), np.float32)
        self.lib.ref_comp_bias(_p(q), len(q), ctypes.c_float(scale), _p(out))
        return out

    def ungapped(self, q, comp_bias, tdata, toff, nthreads=8):
        q = np.ascontiguousarray(q, np.uint8)
        n = len(toff) - 1
        out = np.zeros(n, np.int32)
        self.lib.ref_ungapped_alignment(_p(q), len(q), 1 if comp_bias else 0, _p(tdata), _p(toff), ctypes.c_int64(n),
                                        _p(out), nthreads)
        return out

    def scan_team(self, max_len, comp_bias=True, nthreads=8):
        """persistent thread team + per-thread SmithWaterman objects (ref_scan_init); use with scan_batch / scan_free"""
        self.lib.ref_scan_init.restype = ctypes.c_void_p
        return ctypes.c_void_p(self.lib.ref_scan_init(ctypes.c_int64(int(max_len)), 1 if comp_bias else 0, int(nthreads)))

    def scan_batch(self, team, queries, tdata, toff, out=None):
        """ungapped_alignment of every query against every target on the team; -> u8 [nq][n]"""
        qd, qo = pack_targets([np.ascontiguousarray(q, np.uint8) for q in queries])
        n = len(toff) - 1
        if out is None:
            out = np.empty((len(queries), n), np.uint8)
        self.lib.ref_scan_batch(team, _p(qd), _p(qo), ctypes.c_int64(len(queries)), _p(tdata), _p(toff), ctypes.c_int64(n), _p(out))
        return out

    def scan_free(self, team):
        self.lib.ref_scan_free(team)

    def sw_score_endpos(self, q, comp_bias, tdata, toff, go=11, ge=1, nthreads=8):
        q = np.ascontiguousarray(q, np.uint8)
        n = len(toff) - 1
        out = np.zeros((n, 4), np.int32)
        self.lib.ref_sw_score_endpos(_p(q), len(q), 1 if comp_bias else 0, _p(tdata), _p(toff), ctypes.c_int64(n),
                                     go, ge, _p(out), nthreads)
        return out

    def sw_score_endpos_multi(self, queries, comp_bias, tdata, toff, pairs, go=11, ge=1, nthreads=8):
        """pairs: uint32 [n][2] grouped by query; one OpenMP region over queries (the shape of Alignment::run)"""
        qd, qo = pack_targets(queries)
        pq = np.ascontiguousarray(pairs[:, 0], np.uint32)
        pt = np.ascontiguousarray(pairs[:, 1], np.uint32)
        out = np.zeros((len(pq), 4), np.int32)
        to = np.ascontiguousarray(toff, np.int64)
        self.lib.ref_sw_score_endpos_multi(_p(qd), _p(qo), ctypes.c_int64(len(queries)), 1 if comp_bias else 0, _p(tdata), _p(to),
                                           _p(pq), _p(pt), ctypes.c_int64(len(pq)), go, ge, _p(out), nthreads)
        return out

    def ssw_align(self, q, comp_bias, tdata, toff, go=11, ge=1, mode=1, eval_thr=1e300, cov_mode=0, cov_thr=0.0,
                  db_residues=10**9, want_bt=False, nthreads=8):
        q = np.ascontiguousarray(q, np.uint8)
        n = len(toff) - 1
        out = np.zeros((n, 10), np.int32)
        ev = np.zeros(n, np.float64)
        stride = 0
        bt = None
        if want_bt:
            stride = int(len(q) + np.max(np.diff(toff)) + 8) if n else 8
            bt = np.zeros(n * stride, np.uint8)
        self.lib.ref_ssw_align(_p(q), len(q), 1 if comp_bias else 0, _p(tdata), _p(toff), ctypes.c_int64(n), go, ge,
                               mode, ctypes.c_double(eval_thr), cov_mode, ctypes.c_float(cov_thr),
                               ctypes.c_int64(db_residues), _p(out), _p(ev), _p(bt), ctypes.c_int64(stride), nthreads)
        bts = None
        if want_bt:
            bts = [bytes(bt[i * stride:(i + 1) * stride]).split(b"\0", 1)[0].decode() for i in range(n)]
        return out, ev, bts

    def ksw_extz2(self, q, t, mat5, gapo=5, gape=2, w=64, zdrop=40, flag=0x41):
        q = np.ascontiguousarray(q, np.uint8); t = np.ascontiguousarray(t, np.uint8)
        m = np.ascontiguousarray(mat5, np.int8)
        out = np.zeros(11, np.int32)
        cap = len(q) + len(t) + 4
        cg = np.zeros(cap, np.uint32)
        self.lib.ref_ksw_extz2(_p(q), len(q), _p(t), len(t), _p(m), gapo, gape, w, zdrop, flag, _p(out), _p(cg), cap)
        return out, cg[:out[10]]

    def nucl_align(self, q, t, diagonal, gapo=5, gape=2, zdrop=40):
        q = np.ascontiguousarray(q, np.uint8); t = np.ascontiguousarray(t, np.uint8)
        out = np.zeros(7, np.int32)
        cap = len(q) + len(t) + 8
        cg = np.zeros(cap, np.uint32)
        bt = ctypes.create_string_buffer(cap)
        self.lib.ref_banded_nucl_align(_p(q), len(q), _p(t), len(t), int(diagonal), gapo, gape, zdrop, _p(out), _p(cg), cap, bt, cap)
        return out, cg[:out[6]], bt.value.decode()

    def nucl_align_batch(self, reads, tdata, toff, tasks, gapo=5, gape=2, zdrop=40, nthreads=8):
        qd, qo = pack_targets(reads)
        tq = np.ascontiguousarray(tasks[:, 0], np.uint32); tt = np.ascontiguousarray(tasks[:, 1], np.uint32)
        dg = np.ascontiguousarray(tasks[:, 2], np.int64)
        dg = np.where(dg >= 32768, dg - 65536, dg).astype(np.int32)
        out = np.zeros((len(tq), 7), np.int32)
        to = np.ascontiguousarray(toff, np.int64)
        self.lib.ref_banded_nucl_align_batch(_p(qd), _p(qo), _p(tdata), _p(to), _p(tq), _p(tt), _p(dg), ctypes.c_int64(len(tq)), gapo, gape,
                                             zdrop, _p(out), nthreads)
        return out

    def diag(self, q, bias_f32, tdata, toff, hit_ids, hit_diags):
        q = np.ascontiguousarray(q, np.uint8)
        ids = np.ascontiguousarray(hit_ids, np.uint32)
        dg = np.ascontiguousarray(hit_diags, np.uint16)
        counts = np.zeros(len(ids), np.uint8)
        raw = np.zeros(len(ids), np.int32)
        b = None if bias_f32 is None else np.ascontiguousarray(bias_f32, np.float32)
        self.lib.ref_diag_align(_p(q), len(q), _p(b), _p(tdata), _p(toff), ctypes.c_int64(len(toff) - 1), _p(ids),
                                _p(dg), ctypes.c_int64(len(ids)), _p(counts), _p(raw))
        return counts, raw
