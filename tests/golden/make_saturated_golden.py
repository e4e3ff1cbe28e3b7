"""tests/golden/make_saturated_golden.py -- word-mode saturation fixtures from the REFERENCE's own code (oracle/_ref).

sw_sse2_word (StripedSmithWaterman.cpp:301-476) adds profile scores with adds_epi16, so every cell saturates at 32767.  A pair
whose exact local score passes 32767 reports 32767, ends at the first column in which a cell reaches 32767 (smallest row in it),
takes its start from a reverse pass that stops at the first column whose maximum is 32767, and backtraces inside that rectangle.
The cases: long sequence queries (5 900 - 17 000 residues, one of more than 16 384) against themselves, mutated copies with and
without indels, pieces, flanked copies, random prefixes and half-length prefixes; pairs whose exact score lies just below 32767;
pairs on both sides of the device's int16 routing bound; two sharp PSSM queries; and `align` records of hit lists that mix
saturated pairs with ordinary hits from examples_v1.npz.  Every pair also carries its exact (unsaturated int32) score and end,
so the fixture shows where saturation moves the answer.

Build container only:  python tests/golden/make_saturated_golden.py  ->  tests/golden/saturated_v1.npz"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.pyoracle import Oracle, Ref, pack_targets  # noqa: E402
from mmseqs2_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

# `mmseqs align` parameter sets of the record cases (Ref.align_query keywords)
ALIGN_CONFIGS = {
    "sat_mode2": dict(sw_mode=2, eval_thr=1e-3),
    "sat_mode1_cov": dict(sw_mode=1, eval_thr=1e-3, cov_thr=0.8, cov_mode=0, add_backtrace=False),
    "sat_identity": dict(sw_mode=1, eval_thr=1e-3, include_identity=True, add_backtrace=False),
}


def exact_endpos(prof, t, go, ge):
    """exact int32 affine local DP (no saturation) with the reference's end rule: first column where the running maximum
    strictly increases, smallest row in it.  prof: int32 [A][qL] (mat[a][q[j]] + cb[j]); needs go >= ge (the F chain is then
    a prefix maximum over the rows).  -> (score, qEnd, dbEnd)"""
    qL = prof.shape[1]
    rows = np.arange(qL, dtype=np.int64)
    H = np.zeros(qL, np.int64)
    E = np.zeros(qL, np.int64)
    best, bq, bt = 0, -1, -1
    for i, r in enumerate(t):
        diag = np.concatenate(([0], H[:-1]))
        h0 = np.maximum(np.maximum(diag + prof[r], E), 0)
        a = np.maximum.accumulate(h0 - go + (rows + 1) * ge)
        f = np.concatenate(([0], a[:-1] - rows[1:] * ge))
        H = np.maximum(h0, f)
        E = np.maximum(E - ge, H - go)
        m = int(H.max())
        if m > best:
            best, bq, bt = m, int(np.argmax(H)), i
    return best, bq, bt


def seq(rng, bg, n):
    return synth.random_seqs(rng, 1, bg, mean=n, sigma=0, lo=n, hi=n, normal=True)[0]


def prefix_for_score(diag_scores, lo, hi):
    """shortest prefix length whose summed self score lies in [lo, hi]"""
    c = np.cumsum(diag_scores)
    k = np.nonzero((c >= lo) & (c <= hi))[0]
    assert len(k), (lo, hi)
    return int(k[0]) + 1


def make_pssm(rng, mat, q, sharp):
    """sharp position-specific table around a seed sequence: int8 [20][L]"""
    base = mat[:20, :][:, q].astype(np.float64)
    p = np.rint(base * sharp + rng.normal(0, 1.5, base.shape))
    return np.clip(p, -60, 127).astype(np.int8)


def main():
    ref = Ref()
    mat, pb, _ = ref.matrix()
    orc = Oracle(mat, pb)
    ex = np.load(os.path.join(HERE, "examples_v1.npz"))
    rng = np.random.default_rng(20261017)
    bg = synth.background(pb)

    pool = []

    def add(t):
        pool.append(np.ascontiguousarray(t, np.uint8))
        return len(pool) - 1

    def flank(q, a, b):
        return np.concatenate([seq(rng, bg, a), q, seq(rng, bg, b)])

    def insert(q, at, n):
        return np.concatenate([q[:at], seq(rng, bg, n), q[at:]])

    queries, groups = [], []       # groups: (query index, comp bias, go, ge, [pool indices])
    Q = {}
    for name, L in (("q7000", 7000), ("q6500", 6500), ("q9000", 9000), ("q12000", 12000), ("q17000", 17000)):
        Q[name] = len(queries)
        queries.append(seq(rng, bg, L))
    q = queries[Q["q7000"]]
    m = lambda s, i=0.0: synth.mutate(rng, q, bg, s, i)     # noqa: E731
    groups.append((Q["q7000"], 1, 11, 1, [add(q), add(m(0.03)), add(m(0.05)), add(m(0.05, 0.01)), add(q[300:6700]), add(insert(q, 3500, 50)),
                                           add(flank(q, 400, 600)), add(np.concatenate([seq(rng, bg, 700), q[100:]])), add(q[:3500])]))
    g0 = groups[0][4]
    piece_lo, piece_hi = add(q[100:3009]), add(q[100:3010])        # smax 11 (cb off): 2909 * 11 < 32000 <= 2910 * 11
    groups.append((Q["q7000"], 0, 11, 1, [g0[0], g0[2], g0[7], g0[6], piece_lo, piece_hi, add(m(0.10, 0.02))]))
    q = queries[Q["q6500"]]
    groups.append((Q["q6500"], 0, 11, 1, [add(q), add(synth.mutate(rng, q, bg, 0.03, 0.0)),
                                           add(flank(synth.mutate(rng, q, bg, 0.03, 0.01), 3000, 10000))]))   # target >> query
    q = queries[Q["q9000"]]
    m = lambda s, i=0.0: synth.mutate(rng, q, bg, s, i)     # noqa: E731
    groups.append((Q["q9000"], 1, 5, 2, [add(q), add(m(0.10, 0.02)), add(m(0.15)), add(q[500:8000]), add(flank(q, 1000, 300)), add(q[:4500])]))
    g3 = groups[-1][4]
    groups.append((Q["q9000"], 0, 20, 1, [g3[0], add(m(0.10, 0.03)), add(m(0.15, 0.01)), add(np.concatenate([seq(rng, bg, 900), q[200:]])),
                                          g3[5]]))
    q = queries[Q["q12000"]]
    m = lambda s, i=0.0: synth.mutate(rng, q, bg, s, i)     # noqa: E731
    groups.append((Q["q12000"], 0, 5, 2, [add(q), add(m(0.10)), add(m(0.15, 0.03)), add(flank(q, 250, 250)), add(q[2000:10000])]))
    q = queries[Q["q17000"]]
    m = lambda s, i=0.0: synth.mutate(rng, q, bg, s, i)     # noqa: E731
    groups.append((Q["q17000"], 1, 11, 1, [add(q), add(m(0.05, 0.01)), add(m(0.15, 0.02)), add(q[5000:12000]),           # query >> target
                                           add(np.concatenate([seq(rng, bg, 700), q[100:]]))]))
    # just below saturation (cb off: a sequence profile's row maxima are the matrix diagonal, so qsum == self score)
    for lo, hi in ((31000, 31990), (32600, 32766)):
        src = seq(rng, bg, 7000)
        L = prefix_for_score(mat[src, src].astype(np.int64), lo, hi)
        q = src[:L]
        Q["below%d" % lo] = len(queries)
        queries.append(q)
        dsc = mat[q, q].astype(np.int64)
        tg = [add(q), add(synth.mutate(rng, q, bg, 0.03, 0.0)), add(flank(q, 200, 200))]
        for a, b in ((31000, 31400), (32000, 32300), (32600, 32766)):
            if dsc.sum() >= a:
                tg.append(add(q[:prefix_for_score(dsc, a, b)]))
        groups.append((len(queries) - 1, 0, 11, 1, tg))
    groups.append((Q["below32600"], 1, 11, 1, groups[-1][4][:3]))

    # ordinary real-protein targets for the mixed `align` hit lists
    ex_q = [ex["qdata"][int(ex["qoff"][i]):int(ex["qoff"][i + 1])] for i in (2, 3)]
    ex_hits = [ex["hit_ids"][int(ex["hit_off"][i]):int(ex["hit_off"][i + 1])] for i in (2, 3)]
    ex_pick = sorted(set(range(40)) | set(int(t) for h in ex_hits for t in h))
    ex_ids = {t: add(ex["tdata"][int(ex["toff"][t]):int(ex["toff"][t + 1])]) for t in ex_pick}

    # two sharp PSSM queries against their consensus and mutated copies
    pssms, pssm_targets = [], []
    for L, sharp in ((2500, 3.0), (4000, 2.0)):
        p = make_pssm(rng, mat, seq(rng, bg, L), sharp)
        c = p.argmax(0).astype(np.uint8)
        pssms.append(p)
        pssm_targets.append([add(c), add(synth.mutate(rng, c, bg, 0.05, 0.0)), add(synth.mutate(rng, c, bg, 0.10, 0.01)),
                             add(c[L // 5:L - L // 5]), add(flank(c, 300, 300))])

    td, to = pack_targets(pool)
    qd, qo = pack_targets(queries)
    out = {"tdata": td, "toff": to, "qdata": qd, "qoff": qo}
    gq = np.array([g[0] for g in groups], np.int32)
    gcb = np.array([g[1] for g in groups], np.int32)
    ggo = np.array([g[2] for g in groups], np.int32)
    gge = np.array([g[3] for g in groups], np.int32)
    goff = np.zeros(len(groups) + 1, np.int64)
    goff[1:] = np.cumsum([len(g[4]) for g in groups])
    out.update(grp_query=gq, grp_cb=gcb, grp_go=ggo, grp_ge=gge, grp_off=goff,
               grp_targets=np.concatenate([np.array(g[4], np.int32) for g in groups]))

    endpos, align, ident, bts, exact = [], [], [], [], []
    for qi, cbf, go, ge, tg in groups:
        q = queries[qi]
        sd, so = pack_targets([pool[t] for t in tg])
        e = ref.sw_score_endpos(q, bool(cbf), sd, so, go, ge)
        a1, _, _ = ref.ssw_align(q, bool(cbf), sd, so, go, ge, mode=1)
        a2, _, bt = ref.ssw_align(q, bool(cbf), sd, so, go, ge, mode=2, want_bt=True)
        assert np.array_equal(a1[:, :6], a2[:, :6]) and np.array_equal(a1[:, [0, 2, 4, 5]], e)
        cb, _ = orc.query_cb(q, bool(cbf))
        prof = mat[:, q].astype(np.int64) + cb.astype(np.int64)
        for k, t in enumerate(tg):
            if e[k, 0] == 32767:
                exact.append(exact_endpos(prof, pool[t], go, ge))
            else:
                exact.append((int(e[k, 0]), int(e[k, 1]), int(e[k, 2])))
                if k == 0 and len(q) < 8000:       # the exact DP agrees with the reference wherever nothing saturates
                    assert exact_endpos(prof, pool[t], go, ge) == exact[-1]
        endpos.append(e); align.append(a1[:, :6]); ident.append(a2[:, 6]); bts += bt
        print("group q%d L%d cb%d %d/%d:" % (qi, len(q), cbf, go, ge), [tuple(r) for r in e[:, :3]])
    out["endpos"], out["align"], out["ident"] = np.concatenate(endpos), np.concatenate(align), np.concatenate(ident)
    out["bt"] = np.array(bts)
    out["exact"] = np.array(exact, np.int32)
    sat = out["endpos"][:, 0] == 32767
    moved = sat & ((out["exact"][:, 1] != out["endpos"][:, 1]) | (out["exact"][:, 2] != out["endpos"][:, 2]))
    below = (out["endpos"][:, 0] >= 31000) & (out["endpos"][:, 0] < 32767)
    print("pairs %d, saturated %d, exact argmax elsewhere %d, exact score in [31000, 32767) %d"
          % (len(sat), int(sat.sum()), int(moved.sum()), int(below.sum())))
    assert sat.sum() >= 20 and moved.sum() >= 20 and below.sum() >= 4
    assert (out["exact"][sat, 0] > 32767).all()

    for k, (p, tg) in enumerate(zip(pssms, pssm_targets)):
        c = p.argmax(0).astype(np.uint8)
        sd, so = pack_targets([pool[t] for t in tg])
        a1, _, _ = ref.profile_align(p, c, sd, so, mode=1)
        a2, _, pbt = ref.profile_align(p, c, sd, so, mode=2, want_bt=True)
        assert np.array_equal(a1[:, :6], a2[:, :6])
        out["pssm%d" % k], out["pssm%d_targets" % k] = p, np.array(tg, np.int32)
        out["pssm%d_align" % k], out["pssm%d_ident" % k], out["pssm%d_bt" % k] = a1[:, :6], a2[:, 6], np.array(pbt)
        print("pssm", k, "L", p.shape[1], [tuple(r) for r in a1[:, :5]])
        assert (a1[:, 0] == 32767).sum() >= 2

    # `align` records: saturated hits and ordinary hits of two long queries, plus an ordinary query, in one batch
    tkeys = (1000 + 3 * np.arange(len(pool))).astype(np.uint32)
    aq = [queries[Q["q7000"]], queries[Q["q9000"]]] + ex_q
    rnd = [ex_ids[t] for t in range(40)]
    hits = [np.array(groups[0][4] + rnd[:15] + [piece_lo, piece_hi], np.uint32),
            np.array(rnd[15:30] + groups[3][4], np.uint32),
            np.array([ex_ids[int(t)] for t in ex_hits[0]] + rnd[30:] + [groups[0][4][0]], np.uint32),
            np.array(rnd[:10] + [ex_ids[int(t)] for t in ex_hits[1]], np.uint32)]
    out["aln_hit_off"] = np.concatenate([[0], np.cumsum([len(h) for h in hits])]).astype(np.int64)
    out["aln_hits"] = np.concatenate(hits)
    qd2, qo2 = pack_targets(aq)
    out["aln_qdata"], out["aln_qoff"] = qd2, qo2
    out["target_keys"] = tkeys
    for name, kw in ALIGN_CONFIGS.items():
        texts = []
        for qi, (q, h) in enumerate(zip(aq, hits)):
            txt, _, nacc = ref.align_query(q, 7000 + qi, td, to, h, tkeys[h], int(to[-1]), **kw)
            texts.append(txt)
        out["cfg_%s_text" % name] = np.array(texts)
        print(name, [t.count(b"\n") for t in texts], "records")
    np.savez_compressed(os.path.join(HERE, "saturated_v1.npz"), **out)
    print("wrote saturated_v1.npz", os.path.getsize(os.path.join(HERE, "saturated_v1.npz")))


if __name__ == "__main__":
    main()
