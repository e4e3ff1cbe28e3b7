/* oracle/oracle.c -- TEST INFRASTRUCTURE.  CPU restatement of MMseqs2's alignment hot path.
 *
 * This file is the checker, never the product: only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load liboracle.so.  Nothing under
 * mmseqs2_b200/ links, imports or executes it.
 *
 * Parity status: PINNED.  Every function below is checked against the reference's own code
 * compiled in place from /root/reference (oracle/_ref/libmmseqs_ref.so, see oracle/Makefile and
 * oracle/ref_glue.cpp) by tests/test_oracle_vs_ref.py, and against the committed fixtures in
 * tests/golden/ (generated from that library by tests/golden/make_golden.py).
 * Exception (SURVEY.md T7): word-mode start positions in the *official* binary come from the Rust
 * block-aligner, which cannot be built here; they are pinned against the reference's own
 * fallback path (StripedSmithWaterman.cpp:879-882) only.
 *
 * Conventions: residues are numeric codes 0..A-1; `mat` is the A*A int16 substitution matrix
 * (row-major, mat[a*A+b] = BaseMatrix::subMatrix[a][b]); `cb` is the int8 composition bias per
 * query position (all zero when the correction is off).  Plain scalar C, textbook recurrences:
 * SURVEY.md T1-T5 establish (and tests/test_oracle_vs_ref.py re-checks) that SIMD width and
 * striping do not leak into any output.
 */
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_MAX(a, b) ((a) > (b) ? (a) : (b))
#define ORC_MIN(a, b) ((a) < (b) ? (a) : (b))

/* ------------------------------------------------------------------------------------------
 * Composition bias, float.  Follows SubstitutionMatrix::calcLocalAaBiasCorrection,
 * src/commons/SubstitutionMatrix.cpp:79-109 -- the float/double mixing is part of the contract.
 * ------------------------------------------------------------------------------------------ */
void orc_comp_bias(const int16_t *mat, const double *pback, int A, const uint8_t *seq, int N, float scale,
                   float *out) {
    const int windowSize = 40;
    for (int i = 0; i < N; i++) {
        const int minPos = ORC_MAX(0, i - windowSize / 2);
        const int maxPos = ORC_MIN(N, i + windowSize / 2);
        const int windowLength = maxPos - minPos;
        int sumSubScores = 0;
        const int16_t *row = mat + (size_t) seq[i] * A;
        for (int j = minPos; j < maxPos; j++) sumSubScores += row[seq[j]];
        sumSubScores -= row[seq[i]];
        float deltaS_i = (float) sumSubScores;
        deltaS_i = (float) ((double) deltaS_i / (-1.0 * (double) (float) windowLength));
        for (int a = 0; a < A; a++) deltaS_i = (float) ((double) deltaS_i + pback[a] * (double) (float) row[a]);
        out[i] = scale * deltaS_i;
    }
}

/* int8 rounding used by the gapped/ungapped-scan profile: StripedSmithWaterman.cpp:1379
 * ((int8_t) binds to the comparison, the float is then converted on assignment). */
void orc_round_bias_ssw(const float *in, int N, int8_t *out) {
    for (int i = 0; i < N; i++) {
        double v = (in[i] < 0.0) ? (in[i] - 0.5) : (in[i] + 0.5); /* float -/+ double literal: double */
        out[i] = (int8_t) v;
    }
}

/* int8 rounding used by the per-diagonal scorer (note the /4): UngappedAlignment.cpp:395-400 */
void orc_round_bias_diag(const float *in, int N, int8_t *out) {
    for (int i = 0; i < N; i++) {
        float v = in[i];
        v = (v < 0.0) ? (float) (v / 4 - 0.5) : (float) (v / 4 + 0.5);
        out[i] = (int8_t) (char) v;
    }
}

/* Profile bias constant: StripedSmithWaterman.cpp:1375-1406.  cbEnabled = aaBiasCorrection flag. */
int orc_ssw_bias(const int16_t *mat, int A, const int8_t *cb, int qL, int cbEnabled) {
    int bias = 0;
    for (int i = 0; i < A * A; i++) {
        int8_t m = (int8_t) mat[i];
        if (m < bias) bias = m;
    }
    int compositionBias = 0;
    if (cbEnabled) {
        for (int i = 0; i < qL; i++) compositionBias = (compositionBias < cb[i]) ? compositionBias : cb[i];
        compositionBias = ORC_MIN(compositionBias, 0);
    }
    return abs(bias) + abs(compositionBias);
}

/* score of query position j against target residue t: mat[t][q[j]] + cb[j]
 * (createQueryProfile, StripedSmithWaterman.cpp:753-786: row index is the TARGET residue). */
static inline int orc_s(const int16_t *mat, int A, const uint8_t *q, const int8_t *cb, int j, int t) {
    return mat[(size_t) t * A + q[j]] + cb[j];
}

/* ------------------------------------------------------------------------------------------
 * A2: SmithWaterman::ungapped_alignment, StripedSmithWaterman.cpp:1817-1876.
 * Saturating u8: S(j,i) = subs_u8(adds_u8(S(j-1,i-1), s+bias), bias).
 * ------------------------------------------------------------------------------------------ */
int orc_ungapped_alignment(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias,
                           const uint8_t *t, int tL) {
    int *prev = (int *) calloc((size_t) qL + 1, sizeof(int));
    int *cur = (int *) calloc((size_t) qL + 1, sizeof(int));
    int best = 0;
    for (int i = 0; i < tL; i++) {
        for (int j = 0; j < qL; j++) {
            int diag = (j == 0) ? 0 : prev[j - 1];
            int p = (uint8_t) (int8_t) (orc_s(mat, A, q, cb, j, t[i]) + bias); /* profile byte as stored */
            int v = diag + p;
            if (v > 255) v = 255;
            v -= bias;
            if (v < 0) v = 0;
            cur[j] = v;
            if (v > best) best = v;
        }
        int *tmp = prev; prev = cur; cur = tmp;
    }
    free(prev); free(cur);
    return best;
}

/* ------------------------------------------------------------------------------------------
 * A3/A4: one direction of the affine local DP with the reference's reporting rules.
 * sw_sse2_byte StripedSmithWaterman.cpp:98-299, sw_sse2_word :301-476 (H,E,F recurrences and
 * the "first column where the running max strictly increases" end rule :233-247 / :414-424,
 * smallest query index in the saved column :263-271 / :441-449).
 *
 * qs/ts with strides let the same routine run forward (stride +1) or on reversed prefixes
 * (stride -1), which is how alignStartPosBacktrace (:1129-1183) reuses the kernels.
 * terminate < 0: scan everything.  terminate >= 0: stop at the first column whose max equals it.
 * Returns max; *endCol = column (scan order) of the saved column or -1; *endRow = smallest row
 * with H == max in the saved column (rows >= 0), or defaultRow when nothing was saved.
 * ------------------------------------------------------------------------------------------ */
static int orc_gotoh(const int16_t *mat, int A, const uint8_t *q, const int8_t *cb, int qL, int qStride,
                     const uint8_t *t, int tL, int tStride, int go, int ge, int terminate, int *endCol,
                     int *endRow) {
    int *H = (int *) calloc((size_t) qL + 1, sizeof(int));   /* H[j+1] = H(prev col, row j) */
    int *E = (int *) calloc((size_t) qL + 1, sizeof(int));
    int *saved = (int *) calloc((size_t) qL + 1, sizeof(int));
    int max = 0, ec = -1;
    for (int i = 0; i < tL; i++) {
        int tr = t[(ptrdiff_t) i * tStride];
        int diag = 0, F = 0, colmax = 0;
        for (int j = 0; j < qL; j++) {
            int s = mat[(size_t) tr * A + q[(ptrdiff_t) j * qStride]] + cb[(ptrdiff_t) j * qStride];
            int h = diag + s;
            if (h > 32767) h = 32767;   /* adds_epi16 (word mode) saturates the diagonal move; E and F follow from it */
            int e = E[j + 1];
            if (h < e) h = e;
            if (h < F) h = F;
            if (h < 0) h = 0;
            diag = H[j + 1];
            H[j + 1] = h;
            if (h > colmax) colmax = h;
            int hg = h - go; if (hg < 0) hg = 0;
            e -= ge; if (e < 0) e = 0;
            E[j + 1] = ORC_MAX(e, hg);
            F -= ge; if (F < 0) F = 0;
            F = ORC_MAX(F, hg);
        }
        if (colmax > max) {
            max = colmax;
            ec = i;
            memcpy(saved, H, ((size_t) qL + 1) * sizeof(int));
        }
        if (terminate >= 0 && colmax == terminate) break;
    }
    int er = -1;
    if (ec >= 0) {
        for (int j = 0; j < qL; j++) if (saved[j + 1] == max) { er = j; break; }
    }
    *endCol = ec;
    *endRow = er;
    free(H); free(E); free(saved);
    return max;
}

/* alignScoreEndPos<SEQ_SEQ>, StripedSmithWaterman.cpp:892-941: byte pass, word pass iff byte
 * reports 255 (i.e. some column had max + bias >= 255, :238-242,:275).  out = score, qEnd, dbEnd, word */
void orc_sw_score_endpos(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias,
                         const uint8_t *t, int tL, int go, int ge, int32_t *out) {
    int ec, er;
    int max = orc_gotoh(mat, A, q, cb, qL, 1, t, tL, 1, go, ge, -1, &ec, &er);
    if (max + bias >= 255) {            /* word mode: every cell saturates at INT16_MAX (orc_gotoh), so a pair whose exact score
                                           passes 32767 reports 32767 and ends at the first cell that reached it */
        out[0] = max; out[1] = (er < 0) ? qL - 1 : er; out[2] = (ec < 0) ? 0 : ec; out[3] = 1;
    } else if (max == 0) {              /* byte mode, nothing aligned: end_db = -1; pvHmax is all zero so the
                                           trace loop (:263-271) matches index 0 first */
        out[0] = 0; out[1] = 0; out[2] = -1; out[3] = 0;
    } else {
        out[0] = max; out[1] = er; out[2] = ec; out[3] = 0;
    }
}

/* ssw_align up to start positions (alignment modes 0/1; the E-value / coverage gate is applied by the
 * caller: gate != 0 means "continue to start positions").  StripedSmithWaterman.cpp:831-890, :1129-1212.
 * out = score, qStart, qEnd, dbStart, dbEnd, word */
void orc_sw_align(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias, const uint8_t *t,
                  int tL, int go, int ge, int gate, int32_t *out) {
    int32_t r[4];
    orc_sw_score_endpos(mat, A, q, qL, cb, bias, t, tL, go, ge, r);
    out[0] = r[0]; out[1] = -1; out[2] = r[1]; out[3] = -1; out[4] = r[2]; out[5] = r[3];
    if (r[2] == -1 || !gate) return;
    const int qEnd = r[1], dbEnd = r[2];
    int ec, er;
    int max = orc_gotoh(mat, A, q + qEnd, cb + qEnd, qEnd + 1, -1, t + dbEnd, dbEnd + 1, -1, go, ge, r[0], &ec, &er);
    (void) max;
    out[3] = dbEnd - ec;
    out[1] = qEnd - er;
}

/* ------------------------------------------------------------------------------------------
 * A1: per-diagonal scorer.  UngappedAlignment::createProfile :388-421 (profile[pos*21+a] =
 * subMatrix[q[pos]][a] + cb4[pos], stored as char), scalarDiagonalScoring :45-57,
 * computeSingelSequenceScores :423-437; count = min(255, score) (:283, T2).
 * diagonal is the u16 as stored in CounterResult; lengths < 32768 only (T6).
 * ------------------------------------------------------------------------------------------ */
int orc_diag_score(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb4, const uint8_t *t, int tL,
                   uint16_t diagonal) {
    int d = (int16_t) diagonal;
    unsigned short dist1 = (unsigned short) (0 - diagonal), dist2 = diagonal;
    int minDist = ORC_MIN(dist1, dist2);
    int qOff, tOff, len;
    if (d >= 0 && minDist < qL) {
        qOff = minDist; tOff = 0; len = ORC_MIN(tL, qL - minDist);
    } else if (d < 0 && minDist < tL) {
        qOff = 0; tOff = minDist; len = ORC_MIN(tL - minDist, qL);
    } else {
        return 0;
    }
    int max = 0, score = 0;
    for (int pos = 0; pos < len; pos++) {
        int curr = (int8_t) (mat[(size_t) q[qOff + pos] * A + t[tOff + pos]] + cb4[qOff + pos]);
        score += curr;
        if (score < 0) score = 0;
        if (score > max) max = score;
    }
    return max;
}

/* ------------------------------------------------------------------------------------------
 * Batch drivers (OpenMP) -- one query against n targets laid out as SequenceLookup does
 * (concatenated residues + offsets[n+1], SequenceLookup.cpp:42-46).
 * ------------------------------------------------------------------------------------------ */
void orc_ungapped_alignment_batch(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias,
                                  const uint8_t *tdata, const int64_t *toff, int64_t n, int32_t *out, int nthreads) {
#pragma omp parallel for schedule(dynamic, 16) num_threads(nthreads)
    for (int64_t i = 0; i < n; i++)
        out[i] = orc_ungapped_alignment(mat, A, q, qL, cb, bias, tdata + toff[i], (int) (toff[i + 1] - toff[i]));
}

/* The same scores, organised for throughput (at-scale parity checks on >= 200 k-sequence DBs and the "port" CPU baseline): the
 * biased profile bytes are precomputed once per query as int16 rows P[a][j], and one target column updates a whole row of cells,
 * cur[j+1] = max(0, min(prev[j] + P[t_i][j], 255) - bias), a loop without cross-iteration dependency that the compiler vectorises.
 * tests/test_oracle_golden.py checks it cell for cell against orc_ungapped_alignment above. */
void orc_ungapped_alignment_batch_fast(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias,
                                       const uint8_t *tdata, const int64_t *toff, int64_t n, int32_t *out, int nthreads) {
    int16_t *P = (int16_t *) malloc((size_t) A * qL * sizeof(int16_t));
    for (int a = 0; a < A; a++)
        for (int j = 0; j < qL; j++) P[(size_t) a * qL + j] = (int16_t) (uint8_t) (int8_t) (orc_s(mat, A, q, cb, j, a) + bias);
#pragma omp parallel num_threads(nthreads)
    {
        int16_t *prev = (int16_t *) malloc(((size_t) qL + 1) * sizeof(int16_t));
        int16_t *cur = (int16_t *) malloc(((size_t) qL + 1) * sizeof(int16_t));
#pragma omp for schedule(dynamic, 64)
        for (int64_t k = 0; k < n; k++) {
            const uint8_t *t = tdata + toff[k];
            const int tL = (int) (toff[k + 1] - toff[k]);
            memset(prev, 0, ((size_t) qL + 1) * sizeof(int16_t));
            cur[0] = 0;
            int16_t best = 0;
            for (int i = 0; i < tL; i++) {
                const int16_t *row = P + (size_t) t[i] * qL;
                int16_t colbest = 0;
                for (int j = 0; j < qL; j++) {
                    int16_t v = (int16_t) (prev[j] + row[j]);
                    v = v > 255 ? 255 : v;
                    v = (int16_t) (v - bias);
                    v = v < 0 ? 0 : v;
                    cur[j + 1] = v;
                    colbest = v > colbest ? v : colbest;
                }
                best = colbest > best ? colbest : best;
                int16_t *tmp = prev; prev = cur; cur = tmp;
                cur[0] = 0;
            }
            out[k] = best;
        }
        free(prev); free(cur);
    }
    free(P);
}

void orc_sw_score_endpos_batch(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias,
                               const uint8_t *tdata, const int64_t *toff, int64_t n, int go, int ge, int32_t *out,
                               int nthreads) {
#pragma omp parallel for schedule(dynamic, 4) num_threads(nthreads)
    for (int64_t i = 0; i < n; i++)
        orc_sw_score_endpos(mat, A, q, qL, cb, bias, tdata + toff[i], (int) (toff[i + 1] - toff[i]), go, ge, out + i * 4);
}

void orc_sw_align_batch(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb, int bias,
                        const uint8_t *tdata, const int64_t *toff, int64_t n, int go, int ge, const uint8_t *gate,
                        int32_t *out, int nthreads) {
#pragma omp parallel for schedule(dynamic, 4) num_threads(nthreads)
    for (int64_t i = 0; i < n; i++)
        orc_sw_align(mat, A, q, qL, cb, bias, tdata + toff[i], (int) (toff[i + 1] - toff[i]), go, ge,
                     gate ? gate[i] : 1, out + i * 6);
}

void orc_diag_score_batch(const int16_t *mat, int A, const uint8_t *q, int qL, const int8_t *cb4, const uint8_t *tdata,
                          const int64_t *toff, const uint32_t *hitIds, const uint16_t *hitDiags, int64_t nHits,
                          uint8_t *counts, int32_t *raw) {
    for (int64_t i = 0; i < nHits; i++) {
        uint32_t id = hitIds[i];
        int s = orc_diag_score(mat, A, q, qL, cb4, tdata + toff[id], (int) (toff[id + 1] - toff[id]), hitDiags[i]);
        if (raw) raw[i] = s;
        counts[i] = (uint8_t) ORC_MIN(255, s);
    }
}

/* ------------------------------------------------------------------------------------------
 * A6: CIGAR of an alignment whose score and end points are known.
 * SmithWaterman::banded_sw, StripedSmithWaterman.cpp:1478-1693 (band |dbLen-qLen|+1, doubled until the banded score
 * reaches the known score; three direction bytes per cell; trace back from the bottom-right corner) and
 * computerBacktrace :1280-1308 (expansion to an M/I/D string, identity count).
 * The h/e rows and the direction bytes persist across band doublings exactly as the reference's realloc'ed buffers do.
 * bt receives the backtrace string (NUL-terminated, cap bytes); returns its length, -1 on "trace back error".
 * ------------------------------------------------------------------------------------------ */
typedef struct { int band; } orc_band;
static inline int band_u(int band, int i, int j) { int x = i - band; x = x > 0 ? x : 0; return j - x + 1; }
static inline int64_t band_d(int band, int i, int j, int p) { int x = i - band; x = x > 0 ? x : 0; return (int64_t) (j - x) * 3 + p; }

int orc_sw_backtrace(const int16_t *mat, int A, const uint8_t *q, const int8_t *cb, const uint8_t *t, int qStart, int qEnd,
                     int dbStart, int dbEnd, int score, int go, int ge, char *bt, int cap, int32_t *identical) {
    const uint8_t *qs = q + qStart, *ts = t + dbStart;
    const int8_t *cbs = cb + qStart;
    const int q_len = qEnd - qStart + 1, db_len = dbEnd - dbStart + 1;
    int band = abs(db_len - q_len) + 1;
    /* generous fixed buffers: the band at most doubles past max(q_len, db_len) */
    int max_band = band;
    while (max_band < q_len + db_len) max_band *= 2;
    max_band *= 2;
    const size_t rowcap = (size_t) max_band * 2 + 8;
    int32_t *hb = (int32_t *) calloc(rowcap, sizeof(int32_t)), *eb = (int32_t *) calloc(rowcap, sizeof(int32_t)),
            *hc = (int32_t *) calloc(rowcap, sizeof(int32_t));
    size_t dcap = 0;
    int8_t *direction = NULL, *dl = NULL;
    int64_t width = 0, width_d = 0;
    int max = 0;
    do {
        width = (int64_t) band * 2 + 3; width_d = (int64_t) band * 2 + 1;
        const size_t need = (size_t) (width_d * q_len * 3) + 16;
        if (need > dcap) {
            int8_t *nd = (int8_t *) calloc(need, 1);
            if (direction) { memcpy(nd, direction, dcap); free(direction); }
            direction = nd; dcap = need;
        }
        for (int64_t j = 1; j < width - 1; j++) hb[j] = 0;
        for (int i = 0; i < q_len; i++) {
            int beg = i - band; if (beg < 0) beg = 0;
            int end = i + band; if (end > db_len - 1) end = db_len - 1;
            const int64_t edge = end + 1 < width - 1 ? end + 1 : width - 1;
            int f = 0, u = 0;
            hb[0] = eb[0] = hb[edge] = eb[edge] = hc[0] = 0;
            dl = direction + width_d * i * 3;
            for (int j = beg; j <= end; j++) {
                u = band_u(band, i, j);
                const int e_ = band_u(band, i - 1, j), b = band_u(band, i, j - 1), d = band_u(band, i - 1, j - 1);
                const int64_t de = band_d(band, i, j, 0), df = band_d(band, i, j, 1), dh = band_d(band, i, j, 2);
                int t1 = (i == 0) ? -go : hb[e_] - go;
                int t2 = (i == 0) ? -ge : eb[e_] - ge;
                eb[u] = t1 > t2 ? t1 : t2;
                dl[de] = t1 > t2 ? 3 : 2;
                t1 = hc[b] - go; t2 = f - ge;
                f = t1 > t2 ? t1 : t2;
                dl[df] = t1 > t2 ? 5 : 4;
                const int f1 = f > 0 ? f : 0, e1 = eb[u] > 0 ? eb[u] : 0;
                t1 = e1 > f1 ? e1 : f1;
                t2 = hb[d] + mat[(size_t) qs[i] * A + ts[j]] + cbs[i];
                hc[u] = t1 > t2 ? t1 : t2;
                if (hc[u] > max) max = hc[u];
                if (t1 <= t2) dl[dh] = 1; else dl[dh] = e1 > f1 ? dl[de] : dl[df];
            }
            for (int j = 1; j <= u; j++) hb[j] = hc[j];
        }
        band *= 2;
    } while (max < score);
    band /= 2;
    /* trace back */
    int i = q_len - 1, j = db_len - 1, e = 0, n = 0, state = 2, ok = 1;
    char op = 'M', prev_op = 'M';
    uint32_t *c = (uint32_t *) malloc(((size_t) q_len + db_len + 4) * sizeof(uint32_t));
    while (i > 0 || j > 0) {
        const int64_t idx = band_d(band, i, j, state);
        switch (dl[idx]) {
            case 1: --i; --j; state = 2; dl -= width_d * 3; op = 'M'; break;
            case 2: --i; state = 0; dl -= width_d * 3; op = 'I'; break;
            case 3: --i; state = 2; dl -= width_d * 3; op = 'I'; break;
            case 4: --j; state = 1; op = 'D'; break;
            case 5: --j; state = 2; op = 'D'; break;
            default: ok = 0; break;
        }
        if (!ok) break;
        if (op == prev_op) ++e;
        else { c[n++] = (uint32_t) e << 4 | (prev_op == 'M' ? 0u : prev_op == 'I' ? 1u : 2u); prev_op = op; e = 1; }
    }
    int len = -1;
    if (ok) {
        if (op == 'M') c[n++] = (uint32_t) (e + 1) << 4;
        else { c[n++] = (uint32_t) e << 4 | (op == 'I' ? 1u : 2u); c[n++] = 1u << 4; }
        /* the list was built end -> start: read it backwards (computerBacktrace) */
        int ids = 0, tp = dbStart, qp = qStart;
        len = 0;
        for (int k = n - 1; k >= 0; k--) {
            const uint32_t L = c[k] >> 4, o = c[k] & 0xf;
            for (uint32_t r = 0; r < L; r++) {
                if (o == 0) { ids += t[tp] == q[qp]; ++tp; ++qp; }
                else if (o == 1) ++qp;
                else ++tp;
                if (len < cap - 1) bt[len] = "MID"[o];
                len++;
            }
        }
        if (len < cap) bt[len] = 0; else bt[cap - 1] = 0;
        *identical = ids;
    } else { bt[0] = 0; *identical = 0; }
    free(c); free(direction); free(hb); free(eb); free(hc);
    return len;
}

/* ---- SURVEY 8f row 3 groundwork: DistanceCalculator::computeUngappedAlignment on ASCII sequences -------------------
 * (src/alignment/DistanceCalculator.h:93-174, the per-mode scorers :15-37,177-271, DistanceCalculator.cpp:5-25), as
 * rescorediagonal (src/alignment/rescorediagonal.cpp:231-236) and BandedNucleotideAligner (:104-107) call it.
 * asciimat: [123][123] scores indexed by the two characters (SubstitutionMatrix::createAsciiSubMat).
 * out = {score, startPos, endPos, diagonalLen, distToDiagonal, diagonal}.  No device counterpart yet (next round). */
static void orc_rescore_one(const char *q, unsigned qL, const char *t, unsigned tL, int diagonal, const int8_t *m, int mode, int64_t out[6]) {
    const unsigned dist = (unsigned) (diagonal < 0 ? -diagonal : diagonal);
    out[0] = 0; out[1] = -1; out[2] = -1; out[3] = 0; out[4] = dist; out[5] = diagonal;
    const char *a, *b;
    unsigned len;
    if (diagonal >= 0 && dist < qL) { len = tL < qL - dist ? tL : qL - dist; a = q + dist; b = t; }
    else if (diagonal < 0 && dist < tL) { len = tL - dist < qL ? tL - dist : qL; a = q; b = t + dist; }
    else return;
    out[3] = len;
#define SC(i) ((int) m[(size_t) (unsigned char) a[i] * 123 + (unsigned char) b[i]])
    if (mode == 0) {                       /* HAMMING: number of equal characters */
        unsigned same = 0;
        for (unsigned i = 0; i < len; i++) same += a[i] == b[i];
        out[0] = same;
    } else if (mode == 1) {                /* SUBSTITUTION: best 0-reset running sum */
        int best = 0, s = 0;
        for (unsigned i = 0; i < len; i++) { s += SC(i); if (s < 0) s = 0; if (s > best) best = s; }
        out[0] = best;
    } else if (mode == 2) {                /* ALIGNMENT: the same with the segment that attains it (first maximum) */
        int best = 0, s = 0, minPos = -1, st = 0, en = 0;
        for (unsigned i = 0; i < len; i++) {
            s += SC(i);
            if (s <= 0) { s = 0; minPos = (int) i; }
            if (s > best) { best = s; en = (int) i; st = minPos + 1; }
        }
        out[0] = best; out[1] = st; out[2] = en;
    } else if (mode == 3) {                /* END_TO_END: whole diagonal, '*' at either end skipped, floor 0 */
        unsigned first = (a[0] == '*' || b[0] == '*') ? 1 : 0, last = len - 1;
        if (last > 0 && (a[len - 1] == '*' || b[len - 1] == '*')) last--;
        int64_t s = 0;
        for (unsigned i = first; i <= last; i++) s += SC(i);
        out[0] = s > 0 ? s : 0; out[1] = first; out[2] = last;
    } else {                               /* WINDOW_QUALITY: longest stretch with <= 5 mismatches in any window of 20 */
        const unsigned W = 20, E = 5;
        uint64_t window = 0;
        const uint64_t mask = (uint64_t) 1 << (W - 1);
        unsigned errs = 0, maxLen = 0, curLen = 0, maxEnd = 0, maxStart = 0;
        unsigned first = (a[0] == '*' || b[0] == '*') ? 1 : 0, last = len - 1;
        if (last > 0 && (a[len - 1] == '*' || b[len - 1] == '*')) last--;
        unsigned start = first;
        for (unsigned i = first; i <= last; i++) {
            const int match = a[i] == b[i];
            if (window & mask) errs -= 1;
            window <<= 1;
            if (!match) { window |= 1; errs += 1; }
            curLen += 1;
            if (i >= W - 1 && errs > E) { start = i - W + 2; curLen = W - 1; }
            if (curLen > maxLen) { maxStart = start; maxEnd = i; maxLen = curLen; }
        }
        int s = 0;
        for (unsigned i = maxStart; i < maxEnd; i++) s += SC(i);
        out[0] = (unsigned) s; out[1] = maxStart; out[2] = maxEnd;
    }
#undef SC
}

void orc_rescore_diagonal(const char *q, int qL, const char *t, int tL, uint16_t diagonal, const int8_t *asciimat, int mode, int64_t out[6]) {
    int64_t best[6] = {0, -1, -1, 0, 0, 0}, cur[6];
    /* the unsigned short diagonal stands for every real diagonal congruent to it mod 65536 that meets the rectangle (:98-112) */
    for (unsigned d = 1; d <= 1 + (unsigned) tL / 32768; d++) {
        orc_rescore_one(q, (unsigned) qL, t, (unsigned) tL, -(int) (d * 65536) + (int) diagonal, asciimat, mode, cur);
        if ((uint32_t) cur[0] > (uint32_t) best[0]) for (int k = 0; k < 6; k++) best[k] = cur[k];
    }
    for (unsigned d = 0; d <= (unsigned) qL / 65536; d++) {
        orc_rescore_one(q, (unsigned) qL, t, (unsigned) tL, (int) (d * 65536) + (int) diagonal, asciimat, mode, cur);
        if ((uint32_t) cur[0] > (uint32_t) best[0]) for (int k = 0; k < 6; k++) best[k] = cur[k];
    }
    for (int k = 0; k < 6; k++) out[k] = best[k];
}
