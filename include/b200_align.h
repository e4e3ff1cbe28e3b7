/* include/b200_align.h -- C ABI of libb200align.so: MMseqs2's alignment hot path on one B200 (sm_100a).
 *
 * Plain C, opaque handles, int status codes, caller-allocated outputs, no exceptions (the MMseqs2 host is
 * built -fno-exceptions, src/CMakeLists.txt:97-100).  One b200_ctx owns one GPU, one stream and the
 * resident target DB; calls on one ctx are serialised by an internal mutex, so the per-OpenMP-thread
 * operator objects of the reference (QueryMatcher.cpp:73, Alignment.cpp:295) can share it.
 *
 * Each entry point names the reference interface it replaces (paths relative to the MMseqs2 tree):
 *
 *   b200_db_load            Marv::loadDb/setDb (lib/libmarv/src/marv.h:20-24) and SequenceLookup
 *                           (src/prefiltering/SequenceLookup.cpp:42-46): concatenated numeric residues + offsets.
 *   b200_ungapped_scan      SmithWaterman::ungapped_alignment (src/alignment/StripedSmithWaterman.cpp:1817-1876)
 *                           over every target + the filter/sort/truncate of runFilterOnCpu
 *                           (src/prefiltering/ungappedprefilter.cpp:418-478); same role as Marv::scan (marv.h:47).
 *   b200_diag_score         UngappedAlignment::align / scoreSingelSequenceByCounterResult
 *                           (src/prefiltering/UngappedAlignment.cpp:36-42, 440-460).
 *   b200_sw_score           the score of alignScoreEndPos (ALIGNMENT_MODE_SCORE_ONLY use, Matcher.cpp:62-144).
 *   b200_sw_score_endpos    SmithWaterman::alignScoreEndPos (StripedSmithWaterman.cpp:892-941).
 *   b200_sw_startpos        the reverse pass of SmithWaterman::alignStartPosBacktrace (:1129-1212).
 *   b200_sw_backtrace       SmithWaterman::banded_sw + computerBacktrace (:1478-1693, :1280-1308).
 *   b200_nucl_align         BandedNucleotideAligner::align + ksw_extz2_sse (src/alignment/BandedNucleotideAligner.cpp:73-263,
 *                           lib/ksw2/ksw2_extz2_sse.cpp:44-285).
 *   b200_sw_align           ssw_align alignment modes 0/1 (:831-890) with the E-value/coverage gate supplied
 *                           by the caller (host double math stays in the reference: EvalueComputation.h:18-40).
 *
 * Query profiles are int8, layout [A][qlen] (profile[a*qlen + j] = score of query position j against residue a,
 * composition bias already folded in, NO bias offset added) -- the layout Marv::scan takes
 * (ungappedprefilter.cpp:195-203) and SmithWaterman::profile_word_linear holds (StripedSmithWaterman.cpp:1434-1439).
 */
#ifndef B200_ALIGN_H
#define B200_ALIGN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200_ctx b200_ctx;
typedef struct b200_job b200_job;

enum {
    B200_OK = 0,
    B200_ERR_CUDA = -1,   /* a CUDA runtime call failed; see b200_last_error */
    B200_ERR_ARG = -2,    /* bad argument (NULL, negative length, id out of range, ...) */
    B200_ERR_NODB = -3,   /* no target DB loaded */
    B200_ERR_RANGE = -4,  /* input outside the supported domain (e.g. sequence >= 32768 for the diagonal scorer, T6) */
    B200_ERR_NOMEM = -5
};

typedef struct {
    const int8_t *profile; /* [A][qlen], host memory */
    int32_t qlen;
    int32_t bias;          /* SSW profile bias = |min(mat)| + |min(0, min cb)| (StripedSmithWaterman.cpp:1397-1406);
                              drives the u8 saturation of the scan (T1) and the byte->word rule (T5) */
} b200_query;

typedef struct { uint32_t id; int32_t score; } b200_hit;                 /* ordered: score desc, id asc */
typedef struct { uint32_t query; uint32_t target; } b200_pair;           /* query = index into queries[], target = DB id */
typedef struct { int32_t score, qend, dbend, word; } b200_sw_end;        /* s_align score1,qEndPos1,dbEndPos1,word */
typedef struct { int32_t score, qstart, qend, dbstart, dbend, word; } b200_sw_aln;

/* ---- context -------------------------------------------------------------------------------- */
int b200_device_count(void);                       /* Marv::getDeviceIds (marv.h:19) */
int b200_create(int device, b200_ctx **ctx);
void b200_destroy(b200_ctx *ctx);
const char *b200_last_error(const b200_ctx *ctx);
int b200_device_info(const b200_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, uint64_t *hbm_bytes);
/* kernels launched by this ctx since creation (bench.py reports the delta as gpu_launches) */
uint64_t b200_launch_count(const b200_ctx *ctx);
/* CUDA events on the ctx stream, for device-side timing of resident-input runs */
int b200_event_record(b200_ctx *ctx, int slot /*0..15*/);
int b200_event_elapsed_ms(b200_ctx *ctx, int slot_a, int slot_b, float *ms); /* synchronises on slot_b */
int b200_sync(b200_ctx *ctx);
/* device time (CUDA events on the ctx stream) of the kernels launched by the last b200_nucl_align / b200_sw_backtrace call */
float b200_last_kernel_ms(const b200_ctx *ctx);

/* ---- target DB ------------------------------------------------------------------------------- */
/* residues: numeric codes 0..alphabet-1, sequence i = residues[offsets[i] .. offsets[i+1]).  Copied to HBM. */
int b200_db_load(b200_ctx *ctx, const uint8_t *residues, const uint64_t *offsets, uint64_t n_seq, int alphabet);
/* The same from the padded GPU DB of `makepaddedseqdb` as Marv::loadDb takes it (lib/libmarv/src/marv.h:20; layout
 * src/util/makepaddedseqdb.cpp:66-98; offsets/lengths as src/prefiltering/ungappedprefilter.cpp:127-139 builds them): sequence i =
 * data[offsets[i] .. offsets[i] + lengths[i]), numeric codes with +32 marking soft-masked residues, which become X = alphabet-1 as
 * in the CPU scorer (ungappedprefilter.cpp:401-404). */
int b200_db_load_padded(b200_ctx *ctx, const uint8_t *data, const size_t *offsets, const int32_t *lengths, uint64_t n_seq, int alphabet);
/* The same layout with the mask bit stripped instead (code - 32): the residues Sequence::mapSequence yields for a padded DB read back
 * through DBReader::getUnpadded (src/commons/DBReader.cpp:349-371: masked letters come back lower-case and map to the same codes) -- what
 * the `align` module scores against. */
int b200_db_load_padded_unmasked(b200_ctx *ctx, const uint8_t *data, const size_t *offsets, const int32_t *lengths, uint64_t n_seq, int alphabet);
uint64_t b200_db_num_seqs(const b200_ctx *ctx);
uint64_t b200_db_num_residues(const b200_ctx *ctx);

/* ---- A2: all-diagonals ungapped scan ---------------------------------------------------------- */
/* For each query: score every DB sequence; keep score > min_score_excl; order by (score desc, id asc);
 * truncate to max_hits.  hits: [n_queries][max_hits]; n_hits: [n_queries].
 * dense (optional, may be NULL): [n_queries][n_seq] raw scores as u8 (0..255). */
int b200_ungapped_scan(b200_ctx *ctx, const b200_query *queries, int n_queries, int min_score_excl,
                       uint32_t max_hits, b200_hit *hits, uint32_t *n_hits, uint8_t *dense);

/* ---- A1: per-diagonal scorer ------------------------------------------------------------------ */
/* One query; hit i = (ids[i], diagonals[i]).  counts in/out: entries that are non-zero on input are skipped
 * (UngappedAlignment.cpp:327-329); others receive min(255, score).  raw (optional): unclamped score for
 * every hit (scoreSingleSequence).  The profile here is the diagonal scorer's own (bias/4 rounding,
 * UngappedAlignment.cpp:395-400); q->bias is ignored. */
int b200_diag_score(b200_ctx *ctx, const b200_query *q, const uint32_t *ids, const uint16_t *diagonals, uint64_t n,
                    uint8_t *counts, int32_t *raw);

/* The same for many queries at once: queries[i] (each with its own diagonal-scorer profile) owns hits
 * [hit_offsets[i], hit_offsets[i+1]) of ids / diagonals / counts / raw.  One upload, one launch, one download: the shape in which
 * the k-mer prefilter's per-thread UngappedAlignment objects (QueryMatcher.cpp:73,131) can share a GPU without a round trip and a
 * stream synchronisation per query. */
int b200_diag_score_batch(b200_ctx *ctx, const b200_query *queries, int n_queries, const uint64_t *hit_offsets, const uint32_t *ids,
                          const uint16_t *diagonals, uint8_t *counts, int32_t *raw);

/* ---- rescorediagonal: DistanceCalculator::computeUngappedAlignment on ASCII sequences (SURVEY 8f row 3) -------- */
/* A resident ASCII copy of a sequence DB (entries as DBReader::getData returns them, without the trailing newline): sequence i =
 * data[offsets[i] .. offsets[i+1]).  Independent of the numeric DB of b200_db_load: both can be resident. */
int b200_db_load_ascii(b200_ctx *ctx, const char *data, const uint64_t *offsets, uint64_t n_seq);
/* DistanceCalculator::LocalAlignment (src/alignment/DistanceCalculator.h:75-91) + the identical-residue count rescorediagonal.cpp:296-301
 * derives from it (case-insensitive; modes 2-4 only, 0 otherwise) */
typedef struct { int32_t score, start_pos, end_pos, diagonal_len, dist_to_diagonal, diagonal, identical; } b200_rescore;
/* For every hit (ids[i], diagonals[i]) of every query: computeUngappedAlignment(query, qLen, target, tLen, diagonal, matrix, mode)
 * (src/alignment/DistanceCalculator.h:93-174) as rescorediagonal.cpp:231-236 calls it.  queries: ASCII, concatenated, query i =
 * query_data[query_offsets[i] .. query_offsets[i+1]) owning hits [hit_offsets[i], hit_offsets[i+1]).  ascii_matrix: [123][123] int8,
 * SubstitutionMatrix::createAsciiSubMat (FastMatrix).  mode: Parameters::RESCORE_MODE_* 0 HAMMING, 1 SUBSTITUTION, 2 ALIGNMENT,
 * 3 END_TO_END_ALIGNMENT, 4 WINDOW_QUALITY_ALIGNMENT.  The unsigned short diagonal aliases every real diagonal congruent to it
 * mod 65536 (:98-112), handled as the reference does. */
int b200_rescore_diagonal(b200_ctx *ctx, const char *query_data, const uint64_t *query_offsets, int n_queries, const uint64_t *hit_offsets,
                          const uint32_t *ids, const uint16_t *diagonals, const int8_t *ascii_matrix, int mode, b200_rescore *out);

/* ---- A3-A5: affine-gap local alignment --------------------------------------------------------- */
/* score only (s_align.score1 as alignScoreEndPos reports it: exact below 32767; a pair whose exact score would pass it reports 32767,
 * as the reference's saturating word-mode kernel does, and its end and start positions follow that rule too).  This is the fast path
 * (two targets per warp in int16x2); Matcher-level callers run it on every prefilter hit, apply the reference's
 * E-value gate on the host, and ask for positions (below) only for the survivors. */
int b200_sw_score(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n,
                  int gap_open, int gap_extend, int32_t *scores);
int b200_sw_score_endpos(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n,
                         int gap_open, int gap_extend, b200_sw_end *out);
/* End positions for known scores (scores[i] = the pair's alignment score as b200_sw_score returns it; pairs with score 0 come back
 * as "no residue aligned", dbend -1).  For hosts that gate on the score between the two steps, e.g. by E-value (b200_align_batch). */
int b200_sw_endpos(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n, int gap_open,
                   int gap_extend, const int32_t *scores, b200_sw_end *out);
/* ends[i] is the result of b200_sw_score_endpos for pairs[i]; pairs with ends[i].dbend == -1 are passed through */
int b200_sw_startpos(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n,
                     int gap_open, int gap_extend, const b200_sw_end *ends, b200_sw_aln *out);
/* score + end for every pair, start positions for pairs with gate[i] != 0 (gate == NULL: all) */
int b200_sw_align(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n,
                  int gap_open, int gap_extend, const uint8_t *gate, b200_sw_aln *out);

/* ---- A6: CIGAR / backtrace of protein alignments (alignment modes 2 and 3) ------------------------------- */
/* banded_sw + computerBacktrace (src/alignment/StripedSmithWaterman.cpp:1478-1693, 1280-1308) for alignments whose score,
 * start and end are known (alns[i] from b200_sw_align / b200_sw_startpos; entries with dbend < 0 or qstart < 0 are skipped).
 * query_seqs[q]: numeric residues of query q (for the identity count).  The substitution scores are read from the same
 * [A][qlen] profile as everywhere else, i.e. mat[target][query]; banded_sw reads mat[query][target] -- identical for the
 * symmetric matrices MMseqs2 ships.  cigars: task i owns cigars[cigar_offsets[i] .. cigar_offsets[i+1]), at least
 * (qend-qstart+1) + (dbend-dbstart+1) + 2 entries; ops are len << 4 | op (0 = M, 1 = I query only, 2 = D target only) in
 * alignment order; the reference's backtrace string is their expansion.  ok == 0 reproduces the reference's
 * "Trace back error" outcome (no CIGAR).  Word-mode alignments: the official binary uses the Rust block-aligner here
 * (SURVEY.md T7); this reproduces the reference's own fallback path (:879-882). */
typedef struct { int32_t n_cigar, identical, bt_len, ok; } b200_sw_bt;
int b200_sw_backtrace(b200_ctx *ctx, const b200_query *queries, const uint8_t *const *query_seqs, int n_queries,
                      const b200_pair *pairs, uint64_t n, int gap_open, int gap_extend, const b200_sw_aln *alns, b200_sw_bt *out,
                      uint32_t *cigars, const uint64_t *cigar_offsets);

/* ---- A7: nucleotide gapped aligner ------------------------------------------------------------------ */
/* BandedNucleotideAligner::initQuery + align (src/alignment/BandedNucleotideAligner.cpp:51-263; forward strand,
 * wrappedScoring = false): ungapped seed on the prefilter diagonal, leftward ksw_extz2 (score only), rightward ksw_extz2
 * with CIGAR, band 64.  The DB must have been loaded with alphabet 5 (A,C,T,G,X = 0..4, src/commons/NucleotideMatrix.cpp);
 * scores are nucleotide.out at bit factor 1 (+2/-3; X scores 0 inside ksw2, -3 in the seed).  Sequences 1..32767 long.
 * The reference reads one byte past each sequence when it reverses them (seq_reverse called with L,
 * BandedNucleotideAligner.cpp:60,88); that byte is history-dependent there and is defined as X here.
 * cigars: caller buffer; task i owns cigars[cigar_offsets[i] .. cigar_offsets[i+1]), at least 2*qlen + 72 entries,
 * filled with out[i].n_cigar ops (len << 4 | op, op 0 = M, 1 = I (query only), 2 = D (target only)) in alignment order. */
typedef struct { uint32_t query; uint32_t target; uint16_t diagonal; uint16_t reserved; } b200_nucl_task;
typedef struct { int32_t score, qstart, qend, dbstart, dbend, identical, n_cigar; } b200_nucl_aln;
int b200_nucl_align(b200_ctx *ctx, const uint8_t *query_residues, const uint64_t *query_offsets, uint32_t n_queries,
                    const b200_nucl_task *tasks, uint64_t n, int gap_open, int gap_extend, int zdrop, b200_nucl_aln *out,
                    uint32_t *cigars, const uint64_t *cigar_offsets);

/* ---- resident-input jobs (inputs staged in HBM once, run many times; used for kernel-only timing) ----- */
int b200_scan_job_create(b200_ctx *ctx, const b200_query *queries, int n_queries, int min_score_excl,
                         uint32_t max_hits, b200_job **job);
int b200_sw_job_create(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n,
                       int gap_open, int gap_extend, b200_job **job);
int b200_sw_score_job_create(b200_ctx *ctx, const b200_query *queries, int n_queries, const b200_pair *pairs, uint64_t n,
                             int gap_open, int gap_extend, b200_job **job);
int b200_job_run(b200_job *job);                       /* enqueue on the ctx stream; does not synchronise */
int b200_scan_job_fetch(b200_job *job, b200_hit *hits, uint32_t *n_hits, uint8_t *dense);
int b200_sw_job_fetch(b200_job *job, b200_sw_end *out);
int b200_sw_score_job_fetch(b200_job *job, int32_t *scores);
uint64_t b200_job_cells(const b200_job *job);          /* sum over work items of qlen*tlen (GCUPS numerator) */
void b200_job_destroy(b200_job *job);

#ifdef __cplusplus
}
#endif
#endif /* B200_ALIGN_H */
