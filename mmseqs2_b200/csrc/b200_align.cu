// mmseqs2_b200/csrc/b200_align.cu -- libb200align.so: MMseqs2's alignment hot path, hand-written for sm_100a.
//
// Kernels (see DESIGN.md for layouts and rooflines):
//   ungapped_scan_kernel<G,K>  A2  all-diagonals ungapped scan, int16x2 DPX (__viaddmin_s16x2_relu), profile in smem
//                              (quads of G = 8 queries: half of the profile words from tensor memory, tcgen05.ld)
//   topk_select_kernel         A2  per-query histogram cut-off + ordered compaction of the u8 score vector
//   diag_score_kernel          A1  per-(target,diagonal) max-prefix score as a parallel max-subarray reduction
//   pad_profile_kernel             [A][qlen] int8 -> padded forward / reversed device profiles
//   sw32_kernel<DIR>           A3-A5 affine-gap local DP, one warp per pair, int32 DPX (__viaddmax_s32), wavefront over
//                              lanes, score + end position in one pass; DIR=-1 is the reverse (start position) pass
//
// Semantics follow the reference (cited per function); nothing here is derived from lib/libmarv.
#include "b200_internal.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

struct QueryDesc {     // device-side description of one query profile
    uint64_t raw_off;  // byte offset of the raw [A][qlen] int8 profile in d_raw
    uint64_t pad_off;  // byte offset of the padded [(A+1)][Lp] profile in d_pad (forward; reversed copy follows at +rev_off)
    uint64_t rev_off;
    uint64_t p16_off;  // forward copy for the packed kernel: rows of the last (partial) tile at a lane stride rounded up to 4
    int32_t qlen;
    int32_t Lp;
    int32_t bias;
    int32_t k16;       // rows per lane of the packed kernel's last tile (even, 2..16)
};

struct PairDesc {  // one (query,target) work unit of the gapped kernel, device side
    uint32_t target;
    int32_t qend;   // reverse pass only
    int32_t dbend;  // reverse pass only
    int32_t score;  // reverse pass only: terminate value
};

struct WorkItem {  // one CTA's share: pairs [p0,p1) of one query
    uint32_t query;
    uint32_t p0;
    uint32_t p1;
    uint32_t pad_;
};


// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack16(int lo, int hi) {
    return (uint32_t) (lo & 0xffff) | ((uint32_t) (hi & 0xffff) << 16);
}

// 1-D bulk (TMA) copy global -> shared, completion on an mbarrier.  bytes % 16 == 0, both pointers 16-byte aligned.
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    unsigned a = (unsigned) __cvta_generic_to_shared(bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    unsigned a = (unsigned) __cvta_generic_to_shared(bar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, unsigned bytes, uint64_t *bar) {
    unsigned d = (unsigned) __cvta_generic_to_shared(smem_dst);
    unsigned b = (unsigned) __cvta_generic_to_shared(bar);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d),
                 "l"(gsrc), "r"(bytes), "r"(b)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    unsigned a = (unsigned) __cvta_generic_to_shared(bar);
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// A2: all-diagonals ungapped scan.
// Reference semantics: SmithWaterman::ungapped_alignment, StripedSmithWaterman.cpp:1817-1876 --
//   S(j,i) = subs_u8(adds_u8(S(j-1,i-1), s(j,i)+bias), bias)  ==  max(0, min(S(j-1,i-1) + s(j,i), 255-bias))
// i.e. exactly one __viaddmin_s16x2_relu per two cells.
//
// A group of G lanes owns one target; a lane keeps K packed registers = 2K query rows.  Only the (i-1,j-1)
// dependency exists, so all lanes sit on the SAME target column (no wavefront skew).  To avoid a per-register
// shift for the diagonal move, columns alternate between two row packings:
//   V-form  reg r = rows (b+2r,   b+2r+1)     W-form  reg r = rows (b+2r-1, b+2r)        (b = first row of the lane)
//   V(i+1)[r] = f(W(i)[r]   + P [a][r])        same register, no data movement
//   W(i+2)[r] = f(V(i+1)[r-1] + P'[a][r])      shift by one whole register (descending in-place), one shuffle per lane
// P / P' are the two packings of the int16 query profile, staged in shared memory, laid out [a][c][g] as uint4 so
// that a group's LDS.128 is conflict-free.
// ------------------------------------------------------------------------------------------------
#ifndef B200_SCAN_MINB
#define B200_SCAN_MINB 3
#endif
#ifndef B200_SCAN_K3
#define B200_SCAN_K3 24      // classes up to this K are compiled for B200_SCAN_MINB CTAs per SM
#endif

// Quad variant (QUAD, G = 8 only): a warp scans ONE target for four queries, group q = lane/8 holding query q of the quad.  The
// residue of a column is then warp-uniform, which is what tcgen05.ld needs: the first R registers of every V-form column come from
// tensor memory instead of shared memory, halving the shared-memory bytes per cell (the scan's binding resource; DESIGN §3.1).
// TMEM lane 32*(warp%4) + 8q + g, column a*R + r holds query q's V-form register r of lane g for residue a (each lane quadrant has
// its own copy).  One 512-thread CTA per SM owns all 512 columns.
constexpr int kScanQuadThreads = 512;
constexpr int kScanTmemCols = 512;
constexpr int kScanQuadMinSmem = 116 * 1024;   // > half of an SM's shared memory: no two quad CTAs (any K) share an SM's TMEM
__host__ __device__ constexpr int scan_quad_R(int K) { return K <= 22 ? K : 20; }   // 22 residue rows x R <= 512 columns

__device__ __forceinline__ void tmem_fence_sync() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// tcgen05.ld / st of N (16, 8, 4 or 2) consecutive 32-bit columns per lane, shape 32x32b
template <int N> __device__ __forceinline__ void tmem_ld(uint32_t t, uint32_t *v);
template <> __device__ __forceinline__ void tmem_ld<16>(uint32_t t, uint32_t *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(t));
}
template <> __device__ __forceinline__ void tmem_ld<8>(uint32_t t, uint32_t *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(t));
}
template <> __device__ __forceinline__ void tmem_ld<4>(uint32_t t, uint32_t *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(t));
}
template <> __device__ __forceinline__ void tmem_ld<2>(uint32_t t, uint32_t *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(t));
}
template <int N> __device__ __forceinline__ void tmem_st(uint32_t t, const uint32_t *v);
template <> __device__ __forceinline__ void tmem_st<16>(uint32_t t, const uint32_t *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(t),
                 "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
                 "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
template <> __device__ __forceinline__ void tmem_st<8>(uint32_t t, const uint32_t *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(t), "r"(v[0]), "r"(v[1]), "r"(v[2]),
                 "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
template <> __device__ __forceinline__ void tmem_st<4>(uint32_t t, const uint32_t *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(t), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
}
template <> __device__ __forceinline__ void tmem_st<2>(uint32_t t, const uint32_t *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(t), "r"(v[0]), "r"(v[1]) : "memory");
}
// R consecutive columns (R even, < 32) as x16 / x8 / x4 / x2 pieces
template <int R> __device__ __forceinline__ void tmem_ld_cols(uint32_t t, uint32_t *v) {
    if (R & 16) tmem_ld<16>(t, v);
    if (R & 8) tmem_ld<8>(t + (R & 16), v + (R & 16));
    if (R & 4) tmem_ld<4>(t + (R & 24), v + (R & 24));
    if (R & 2) tmem_ld<2>(t + (R & 28), v + (R & 28));
}
template <int R> __device__ __forceinline__ void tmem_st_cols(uint32_t t, const uint32_t *v) {
    if (R & 16) tmem_st<16>(t, v);
    if (R & 8) tmem_st<8>(t + (R & 16), v + (R & 16));
    if (R & 4) tmem_st<4>(t + (R & 24), v + (R & 24));
    if (R & 2) tmem_st<2>(t + (R & 28), v + (R & 28));
}
// wait::ld, then tie the loaded registers to it so that no use of them is scheduled above the wait
template <int R> __device__ __forceinline__ void tmem_wait_ld(uint32_t *v) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < R; i++) asm volatile("" : "+r"(v[i]));
}

template <int G, int K, bool TILED, bool QUAD>
__global__ void __launch_bounds__(QUAD ? kScanQuadThreads : 256, QUAD || TILED ? 1 : (K <= 12 ? 5 : (K <= B200_SCAN_K3 ? B200_SCAN_MINB : 1)))
ungapped_scan_kernel(const int8_t *__restrict__ raw, const QueryDesc *__restrict__ qd, const uint8_t *__restrict__ db,
                     const uint64_t *__restrict__ off, const int32_t *__restrict__ len,
                     const uint32_t *__restrict__ order, uint32_t n_seq, int A, uint8_t *__restrict__ out, uint32_t n_queries,
                     uint32_t units_per_query, uint32_t unit_targets, unsigned *__restrict__ unit_counter,
                     uint32_t *__restrict__ tile_bnd, uint32_t bnd_slot_words) {
    static_assert(K % 2 == 0, "K must be even");
    static_assert(!TILED || G == 32, "the tiled (long-query) variant runs one target per warp");
    static_assert(!QUAD || (G == 8 && !TILED), "quads are four groups of 8 lanes on one target");
    constexpr int C = K / 4;           // full uint4 chunks of a lane's K registers ...
    constexpr int T = (K % 4) / 2;     // ... plus one uint2 tail chunk when K = 4C + 2
    // V-form registers [0, R) come from tensor memory (QUAD), the rest from shared memory; R % 4 == 0 whenever R < K
    constexpr int R = QUAD ? scan_quad_R(K) : 0;
    constexpr int C_V = R / 4;         // first uint4 chunk of the V table read from shared memory
    constexpr bool T_V = T && R < K;   // the V tail chunk is read from shared memory
    // 32-bit words per residue row and query: [c][g] uint4, then [g] uint2.  With G = 8 a half-warp (the unit of an LDS.64) holds
    // two groups.  Without quads they read two residue rows, and their 64-byte tail chunks would land on the same 16 banks whenever the
    // rows differ by an even number (r01 ncu: 3-4 % of all wavefronts of <8,22>/<8,26> were such conflicts): a second copy of the tail
    // 16 words further on, read by the odd groups, puts the two on disjoint bank halves; the row stride becomes 32(C+1) words.
    // With quads the two groups read one residue row of two queries, ROW_W = 8K = 32C + 16 words apart: disjoint halves already.
    constexpr int TAIL2 = (G == 8 && T == 1 && !QUAD) ? 16 : 0;
    constexpr int ROW_W = G * K + TAIL2;
    constexpr int NQ = QUAD ? 4 : 1;   // queries per residue row of the tables, laid out [a][q][c][g]
    extern __shared__ uint4 smem_u4[];
    uint32_t *P = reinterpret_cast<uint32_t *>(smem_u4);
    uint32_t *Pp = P + (size_t) (A + 1) * NQ * ROW_W;

    __shared__ unsigned cur_unit;
    __shared__ uint32_t tmem_slot;
    const int lane = threadIdx.x & 31;
    const int g = lane % G;
    constexpr int TARGETS_PER_WARP = QUAD ? 1 : 32 / G;
    const uint32_t warps_per_cta = blockDim.x >> 5;
    const uint32_t warp_in_cta = threadIdx.x >> 5;
    const uint32_t padword = (uint32_t) A * 0x01010101u;
    const int q_off = QUAD ? (lane >> 3) * ROW_W : 0;   // this group's query within a residue row of the tables
    const int tail_off = q_off + 4 * C * G + (TAIL2 ? ((lane >> 3) & 1) * TAIL2 : 0);   // which copy of the tail chunk this group reads
    int cur_q = -1;
    uint32_t cst = 0;
    uint32_t tmem = 0;                 // QUAD: this warp's lane quadrant of the CTA's 512 columns
    if (QUAD) {
        if (warp_in_cta == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t) __cvta_generic_to_shared(&tmem_slot)),
                         "r"(kScanTmemCols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tmem_fence_sync();
        tmem = tmem_slot + ((uint32_t) (32 * (warp_in_cta & 3)) << 16);
    }

  // persistent CTA: work units = (query or quad, chunk of the length-sorted target order), handed out query-major / longest
  // targets first by a global counter; the profile tables are rebuilt only when the query changes
  while (true) {
    if (QUAD) tmem_fence_sync(); else __syncthreads();
    if (threadIdx.x == 0) cur_unit = atomicAdd(unit_counter, 1u);
    __syncthreads();
    const uint32_t unit = cur_unit;
    if (unit >= n_queries * units_per_query) break;
    const int qu = (int) (unit / units_per_query);          // query, or quad
    const int qi = QUAD ? 4 * qu + (lane >> 3) : qu;        // this group's query
    const uint32_t chunk = unit % units_per_query;
    // Query rows are processed in tiles of ROWS = 2*G*K (one tile unless TILED).  Tile p covers rows [p*ROWS, (p+1)*ROWS);
    // in W-form columns it also recomputes row p*ROWS-1 from the boundary words the previous tile left in tile_bnd.
    constexpr int ROWS = 2 * G * K;
    const QueryDesc q = qd[qi];
    const int n_tiles = TILED ? (q.qlen + ROWS) / ROWS : 1;   // the last tile needs room for qlen+1 rows
    uint8_t *outq = out + (size_t) qi * n_seq;
    const uint32_t unit_end = min(n_seq, (chunk + 1) * unit_targets);
    uint32_t *cta_bnd = TILED ? tile_bnd + (size_t) blockIdx.x * unit_targets * bnd_slot_words : nullptr;
  for (int tile = 0; tile < n_tiles; tile++) {
    const int row_base = tile * ROWS;
    if (TILED || qu != cur_q) {
        if (TILED) __syncthreads();          // every warp is done with the previous tile's tables (and boundary words)
        const int words = G * K;
        for (int idx = threadIdx.x; idx < (A + 1) * NQ * words; idx += blockDim.x) {
            const int a = idx / (NQ * words), qq = idx / words % NQ, w = idx % words;
            const int gg = w / K, r = w % K;
            const QueryDesc &dq = QUAD ? qd[4 * qu + qq] : q;
            const int8_t *prof = raw + dq.raw_off;
            const int qlen = dq.qlen;
            const int r0 = row_base + 2 * w;
            int s0 = 0, s1 = 0, sm1 = 0;  // rows r0, r0+1, r0-1
            if (a < A) {
                const int8_t *pa = prof + (size_t) a * qlen;
                if (r0 < qlen) s0 = pa[r0];
                if (r0 + 1 < qlen) s1 = pa[r0 + 1];
                if (r0 - 1 >= 0 && r0 - 1 < qlen) sm1 = pa[r0 - 1];
            }
            const int dst = (a * NQ + qq) * ROW_W + (r < 4 * C ? ((r >> 2) * G + gg) * 4 + (r & 3) : 4 * C * G + gg * 2 + (r - 4 * C));
            if (r >= R) P[dst] = pack16(s0, s1);
            Pp[dst] = pack16(sm1, s0);
            if (TAIL2 && r >= 4 * C) { P[dst + TAIL2] = pack16(s0, s1); Pp[dst + TAIL2] = pack16(sm1, s0); }
        }
        if (QUAD && warp_in_cta < 4) {   // one warp per lane quadrant writes that quadrant's copy of V-form registers [0, R)
            const int8_t *prof = raw + q.raw_off;
            for (int a = 0; a <= A; a++) {
                uint32_t v[R > 0 ? R : 1];
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int r0 = 2 * (g * K + r);
                    int s0 = 0, s1 = 0;
                    if (a < A) {
                        if (r0 < q.qlen) s0 = prof[(size_t) a * q.qlen + r0];
                        if (r0 + 1 < q.qlen) s1 = prof[(size_t) a * q.qlen + r0 + 1];
                    }
                    v[r] = pack16(s0, s1);
                }
                tmem_st_cols<R>(tmem + a * R, v);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        cst = (uint32_t) (255 - q.bias) * 0x00010001u;
        cur_q = qu;
        if (QUAD) tmem_fence_sync(); else __syncthreads();
    }
    const bool first_tile = tile == 0, last_tile = tile + 1 == n_tiles;

    for (uint32_t base = chunk * unit_targets + warp_in_cta * TARGETS_PER_WARP; base < unit_end; base += warps_per_cta * TARGETS_PER_WARP) {
        const uint32_t it = base + (QUAD ? 0 : lane / G);
        uint32_t tid = 0;
        int tl = 0;
        if (it < unit_end) { tid = order[it]; tl = len[tid]; }
        const uint4 *tp = reinterpret_cast<const uint4 *>(db + off[tid]);
        int maxl = tl;
        if (!QUAD) {
#pragma unroll
            for (int o = 16; o >= G; o >>= 1) maxl = max(maxl, __shfl_xor_sync(0xffffffffu, maxl, o));
        }

        uint32_t S[K];
#pragma unroll
        for (int r = 0; r < K; r++) S[r] = 0;
        uint32_t best = 0;

        uint32_t *tb = TILED ? cta_bnd + (size_t) (it - chunk * unit_targets) * bnd_slot_words : nullptr;
        for (int i0 = 0; i0 < maxl; i0 += 16) {
            uint4 ch = make_uint4(padword, padword, padword, padword);
            if (i0 < tl) ch = __ldg(tp + (i0 >> 4));
            const uint32_t cw[4] = {ch.x, ch.y, ch.z, ch.w};
            uint32_t bin[8], bout[8];            // boundary words of the 8 V-form columns of this chunk (TILED only)
            if (TILED) {
#pragma unroll
                for (int k = 0; k < 8; k++) { bin[k] = 0; bout[k] = 0; }
                if (!first_tile && g == 0) {
                    const uint4 b0 = *reinterpret_cast<const uint4 *>(tb + (i0 >> 1)), b1 = *reinterpret_cast<const uint4 *>(tb + (i0 >> 1) + 4);
                    bin[0] = b0.x; bin[1] = b0.y; bin[2] = b0.z; bin[3] = b0.w; bin[4] = b1.x; bin[5] = b1.y; bin[6] = b1.z; bin[7] = b1.w;
                }
            }
            // QUAD: the V column's tensor-memory words, loaded one column pair ahead (the residue is warp-uniform)
            uint32_t tv[R > 0 ? R : 1];
            if (QUAD) tmem_ld_cols<R>(tmem + (cw[0] & 0xffu) * R, tv);
#pragma unroll
            for (int u = 0; u < 16; u += 2) {
                // the columns beyond the longest target of the warp are pad residues (neutral row): the second half of the last
                // 16-column chunk is skipped when nothing real is in it (8-column granularity of the loop end, ~1 % fewer cells)
                const bool last_half = !TILED && i0 + 8 >= maxl;
                if (u == 8 && last_half) break;
                const uint32_t wv = cw[u >> 2];
                const uint32_t a0 = (wv >> (8 * (u & 3))) & 0xffu;
                const uint32_t a1 = (wv >> (8 * ((u + 1) & 3))) & 0xffu;
                {   // even column: V from W, same registers
                    if (QUAD) {
                        tmem_wait_ld<R>(tv);
#pragma unroll
                        for (int r = 0; r < R; r++) S[r] = __viaddmin_s16x2_relu(S[r], tv[r], cst);
                        if (u + 2 < 16 && !(u + 2 == 8 && last_half))
                            tmem_ld_cols<R>(tmem + ((cw[(u + 2) >> 2] >> (8 * ((u + 2) & 3))) & 0xffu) * R, tv);
                    }
                    const uint32_t *prow = P + a0 * NQ * ROW_W;
                    const uint4 *p = reinterpret_cast<const uint4 *>(prow + q_off) + g;
#pragma unroll
                    for (int c = C_V; c < C; c++) {
                        const uint4 x = p[c * G];
                        S[4 * c + 0] = __viaddmin_s16x2_relu(S[4 * c + 0], x.x, cst);
                        S[4 * c + 1] = __viaddmin_s16x2_relu(S[4 * c + 1], x.y, cst);
                        S[4 * c + 2] = __viaddmin_s16x2_relu(S[4 * c + 2], x.z, cst);
                        S[4 * c + 3] = __viaddmin_s16x2_relu(S[4 * c + 3], x.w, cst);
                    }
                    if (T_V) {
                        const uint2 x = reinterpret_cast<const uint2 *>(prow + tail_off)[g];
                        S[4 * C + 0] = __viaddmin_s16x2_relu(S[4 * C + 0], x.x, cst);
                        S[4 * C + 1] = __viaddmin_s16x2_relu(S[4 * C + 1], x.y, cst);
                    }
#pragma unroll
                    for (int r = 0; r < K; r += 2) best = __vimax3_s16x2(best, S[r], S[r + 1]);
                    if (TILED) bout[u >> 1] = S[K - 1];   // rows (row_base+ROWS-2, row_base+ROWS-1) in the last lane
                }
                {   // odd column: W from V, shifted by one register
                    uint32_t carry = __shfl_up_sync(0xffffffffu, S[K - 1], 1, G);
                    if (g == 0) carry = TILED ? bin[u >> 1] : 0u;
                    const uint32_t *prow = Pp + a1 * NQ * ROW_W;
                    const uint4 *p = reinterpret_cast<const uint4 *>(prow + q_off) + g;
#ifndef B200_SCAN_NO_PRELOAD
                    uint4 x[C > 0 ? C : 1];
#pragma unroll
                    for (int c = 0; c < C; c++) x[c] = p[c * G];
#endif
                    if (T) {
                        const uint2 xt = reinterpret_cast<const uint2 *>(prow + tail_off)[g];
                        S[4 * C + 1] = __viaddmin_s16x2_relu(S[4 * C + 0], xt.y, cst);
                        S[4 * C + 0] = __viaddmin_s16x2_relu(C > 0 ? S[4 * C - 1] : carry, xt.x, cst);
                    }
#pragma unroll
                    for (int c = C - 1; c >= 0; c--) {
#ifdef B200_SCAN_NO_PRELOAD
                        const uint4 xc = p[c * G];
#else
                        const uint4 xc = x[c];
#endif
                        S[4 * c + 3] = __viaddmin_s16x2_relu(S[4 * c + 2], xc.w, cst);
                        S[4 * c + 2] = __viaddmin_s16x2_relu(S[4 * c + 1], xc.z, cst);
                        S[4 * c + 1] = __viaddmin_s16x2_relu(S[4 * c + 0], xc.y, cst);
                        S[4 * c + 0] = __viaddmin_s16x2_relu(c > 0 ? S[4 * c - 1] : carry, xc.x, cst);
                    }
#pragma unroll
                    for (int r = 0; r < K; r += 2) best = __vimax3_s16x2(best, S[r], S[r + 1]);
                }
            }
            if (TILED && !last_tile && g == G - 1 && i0 < tl) {
                *reinterpret_cast<uint4 *>(tb + (i0 >> 1)) = make_uint4(bout[0], bout[1], bout[2], bout[3]);
                *reinterpret_cast<uint4 *>(tb + (i0 >> 1) + 4) = make_uint4(bout[4], bout[5], bout[6], bout[7]);
            }
        }
        int m = max((int) (best & 0xffffu), (int) (best >> 16));
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (g == 0 && it < unit_end) {
            if (TILED && !first_tile) m = max(m, (int) outq[tid]);
            outq[tid] = (uint8_t) m;
        }
    }
  }  // tiles
  }
  if (QUAD) {   // every warp's tensor-memory loads have completed (waited) before the columns go back
      tmem_fence_sync();
      if (warp_in_cta == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_slot), "r"(kScanTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// A2 epilogue: per query keep score > thr, order (score desc, id asc), truncate to k.
// (runFilterOnCpu: ungappedprefilter.cpp:450-478; comparator compareHitsByScoreAndId.)
// One CTA per query: 256-bin histogram -> cut-off score -> ordered (by id) compaction.  The final sort of the
// <= k survivors happens on the host.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
topk_select_kernel(const uint8_t *__restrict__ dense, uint32_t n_seq, int thr, uint32_t k, b200_hit *__restrict__ hits,
                   uint32_t *__restrict__ n_hits) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t warp_sums[32][2];
    __shared__ int s_cut;
    __shared__ uint32_t s_need, s_total, s_base_hi, s_base_tie;
    const uint8_t *sc = dense + (size_t) blockIdx.x * n_seq;
    b200_hit *oh = hits + (size_t) blockIdx.x * k;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n_seq; i += blockDim.x) atomicAdd(&hist[sc[i]], 1u);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t cum = 0;
        int cut = thr;  // keep everything > cut, plus `need` smallest-id entries == cut
        uint32_t need = 0;
        for (int s = 255; s > thr; s--) {
            if (cum + hist[s] > k) { cut = s; need = k - cum; break; }
            cum += hist[s];
        }
        s_cut = cut; s_need = need; s_total = cum + need; s_base_hi = 0; s_base_tie = 0;
    }
    __syncthreads();
    const int cut = s_cut;
    const uint32_t need = s_need;
    const bool take_ties = need > 0;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t i0 = 0; i0 < n_seq; i0 += blockDim.x) {
        const uint32_t i = i0 + threadIdx.x;
        int s = (i < n_seq) ? (int) sc[i] : -0x7fffffff;
        const bool hi = s > cut;
        const bool tie = take_ties && s == cut;
        const unsigned bh = __ballot_sync(0xffffffffu, hi), bt = __ballot_sync(0xffffffffu, tie);
        if (lane == 0) { warp_sums[wid][0] = __popc(bh); warp_sums[wid][1] = __popc(bt); }
        __syncthreads();
        uint32_t pre_h = 0, pre_t = 0;
        for (int w = 0; w < wid; w++) { pre_h += warp_sums[w][0]; pre_t += warp_sums[w][1]; }
        const uint32_t lm = (1u << lane) - 1u;
        const uint32_t rh = s_base_hi + pre_h + __popc(bh & lm);
        const uint32_t rt = s_base_tie + pre_t + __popc(bt & lm);
        const uint32_t n_hi_total = s_total - need;  // entries strictly above the cut
        if (hi) { oh[rh].id = i; oh[rh].score = s; }
        if (tie && rt < need) { oh[n_hi_total + rt].id = i; oh[n_hi_total + rt].score = s; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t th = 0, tt = 0;
            for (int w = 0; w < (int) (blockDim.x >> 5); w++) { th += warp_sums[w][0]; tt += warp_sums[w][1]; }
            s_base_hi += th; s_base_tie += tt;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) n_hits[blockIdx.x] = s_total;
}

// The same selection spread over TOPK_PARTS CTAs per query, for callers that scan one query at a time (Marv::scan is called once per
// query, ungappedprefilter.cpp:207): a single CTA walking 1 M scores costs ~1.5 ms, a fifth of the scan itself.
//   topk_hist_kernel     CTA (query, part): 256-bin histogram of its slice of the score vector -> part_hist[q][part][256]
//   topk_compact_kernel  CTA (query, part): cut-off from the summed histograms, the slice's base ranks from the parts before it,
//                        ordered compaction of the slice -- the output is identical to topk_select_kernel's (ids ascending within
//                        "above the cut" and within "ties at the cut").
constexpr int TOPK_PARTS = 64;

__global__ void __launch_bounds__(256)
topk_hist_kernel(const uint8_t *__restrict__ dense, uint32_t n_seq, uint32_t *__restrict__ part_hist) {
    __shared__ uint32_t hist[256];
    const uint32_t q = blockIdx.y, part = blockIdx.x;
    const uint32_t per = ((n_seq + TOPK_PARTS - 1) / TOPK_PARTS + 15) / 16 * 16;
    const uint32_t a = min(n_seq, part * per), b = min(n_seq, a + per);
    const uint8_t *sc = dense + (size_t) q * n_seq;
    hist[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t i = a + threadIdx.x; i < b; i += blockDim.x) atomicAdd(&hist[sc[i]], 1u);
    __syncthreads();
    part_hist[((size_t) q * TOPK_PARTS + part) * 256 + threadIdx.x] = hist[threadIdx.x];
}

__global__ void __launch_bounds__(256)
topk_compact_kernel(const uint8_t *__restrict__ dense, uint32_t n_seq, int thr, uint32_t k, const uint32_t *__restrict__ part_hist,
                    b200_hit *__restrict__ hits, uint32_t *__restrict__ n_hits) {
    __shared__ uint32_t total[256], before[256];
    __shared__ uint32_t warp_sums[8][2];
    __shared__ int s_cut;
    __shared__ uint32_t s_need, s_total, s_base_hi, s_base_tie;
    const uint32_t q = blockIdx.y, part = blockIdx.x;
    const uint32_t per = ((n_seq + TOPK_PARTS - 1) / TOPK_PARTS + 15) / 16 * 16;
    const uint32_t a = min(n_seq, part * per), b = min(n_seq, a + per);
    const uint8_t *sc = dense + (size_t) q * n_seq;
    b200_hit *oh = hits + (size_t) q * k;
    {   // per bin: count over all parts, and over the parts before this one
        uint32_t t = 0, bf = 0;
        const uint32_t *ph = part_hist + (size_t) q * TOPK_PARTS * 256 + threadIdx.x;
        for (uint32_t p2 = 0; p2 < TOPK_PARTS; p2++) { const uint32_t c = ph[(size_t) p2 * 256]; t += c; if (p2 < part) bf += c; }
        total[threadIdx.x] = t; before[threadIdx.x] = bf;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t cum = 0;
        int cut = thr;  // keep everything > cut, plus `need` smallest-id entries == cut
        uint32_t need = 0;
        for (int s = 255; s > thr; s--) {
            if (cum + total[s] > k) { cut = s; need = k - cum; break; }
            cum += total[s];
        }
        uint32_t bh = 0;
        for (int s = 255; s > cut; s--) bh += before[s];
        s_cut = cut; s_need = need; s_total = cum + need; s_base_hi = bh; s_base_tie = (need > 0 && cut >= 0) ? before[cut] : 0;
    }
    __syncthreads();
    const int cut = s_cut;
    const uint32_t need = s_need;
    const bool take_ties = need > 0;
    const uint32_t n_hi_total = s_total - need;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t i0 = a; i0 < b; i0 += blockDim.x) {
        const uint32_t i = i0 + threadIdx.x;
        const int s = (i < b) ? (int) sc[i] : -0x7fffffff;
        const bool hi = s > cut;
        const bool tie = take_ties && s == cut;
        const unsigned bhm = __ballot_sync(0xffffffffu, hi), btm = __ballot_sync(0xffffffffu, tie);
        if (lane == 0) { warp_sums[wid][0] = __popc(bhm); warp_sums[wid][1] = __popc(btm); }
        __syncthreads();
        uint32_t pre_h = 0, pre_t = 0;
        for (int w = 0; w < wid; w++) { pre_h += warp_sums[w][0]; pre_t += warp_sums[w][1]; }
        const uint32_t lm = (1u << lane) - 1u;
        const uint32_t rh = s_base_hi + pre_h + __popc(bhm & lm);
        const uint32_t rt = s_base_tie + pre_t + __popc(btm & lm);
        if (hi) { oh[rh].id = i; oh[rh].score = s; }
        if (tie && rt < need) { oh[n_hi_total + rt].id = i; oh[n_hi_total + rt].score = s; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t th = 0, tt = 0;
            for (int w = 0; w < (int) (blockDim.x >> 5); w++) { th += warp_sums[w][0]; tt += warp_sums[w][1]; }
            s_base_hi += th; s_base_tie += tt;
        }
        __syncthreads();
    }
    if (part == 0 && threadIdx.x == 0) n_hits[q] = s_total;
}

// ------------------------------------------------------------------------------------------------
// A1: per-diagonal scorer.  UngappedAlignment.cpp:45-57 (scalarDiagonalScoring), :423-437 (segment selection),
// :283 (min(255,.)).  max over prefixes of the 0-reset running sum == maximum-subarray sum, which is associative:
// each lane scans a contiguous chunk into (sum, best prefix, best suffix, best), then an ordered tree combine.
// ------------------------------------------------------------------------------------------------
struct Seg { int sum, pre, suf, best; };
__device__ __forceinline__ Seg seg_combine(const Seg &L, const Seg &R) {
    Seg o;
    o.sum = L.sum + R.sum;
    o.pre = max(L.pre, L.sum + R.pre);
    o.suf = max(R.suf, R.sum + L.suf);
    o.best = max(max(L.best, R.best), L.suf + R.pre);
    return o;
}

struct DiagQuery { uint64_t prof_off; uint64_t hit_begin; int32_t qlen; int32_t pad_; };   // one query of a batched call

__global__ void __launch_bounds__(256)
diag_score_kernel(const int8_t *__restrict__ prof_base, const DiagQuery *__restrict__ dq, int nq, const uint8_t *__restrict__ db,
                  const uint64_t *__restrict__ off, const int32_t *__restrict__ len, const uint32_t *__restrict__ ids,
                  const uint16_t *__restrict__ diags, uint64_t n, uint8_t *__restrict__ counts,
                  int32_t *__restrict__ raw) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps_total = (uint64_t) gridDim.x * (blockDim.x >> 5);
    for (uint64_t h = (uint64_t) blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); h < n; h += warps_total) {
        const bool skip_count = counts[h] != 0;
        if (skip_count && raw == nullptr) continue;
        // the query this hit belongs to: last descriptor whose hit_begin <= h (hit lists are concatenated in query order)
        int lo = 0, hi = nq - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (dq[mid].hit_begin <= h) lo = mid; else hi = mid - 1; }
        const int8_t *prof = prof_base + dq[lo].prof_off;
        const int qlen = dq[lo].qlen;
        const uint32_t id = ids[h];
        const uint16_t dg = diags[h];
        const int d = (int) (int16_t) dg;
        const int dist1 = (uint16_t) (0 - dg), dist2 = dg;
        const int mind = min(dist1, dist2);
        const int tl = len[id];
        int qoff = 0, toff = 0, cells = 0;
        if (d >= 0 && mind < qlen) { qoff = mind; cells = min(tl, qlen - mind); }
        else if (d < 0 && mind < tl) { toff = mind; cells = min(tl - mind, qlen); }
        const uint8_t *t = db + off[id] + toff;
        const int chunk = (cells + 31) >> 5;
        const int s0 = lane * chunk, s1 = min(cells, s0 + chunk);
        Seg sg = {0, 0, 0, 0};
        int cur = 0;
        for (int p = s0; p < s1; p++) {
            const int v = prof[(size_t) t[p] * qlen + qoff + p];
            sg.sum += v;
            sg.pre = max(sg.pre, sg.sum);
            cur = max(0, cur + v);
            sg.best = max(sg.best, cur);
        }
        sg.suf = cur;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            Seg r;
            r.sum = __shfl_down_sync(0xffffffffu, sg.sum, o);
            r.pre = __shfl_down_sync(0xffffffffu, sg.pre, o);
            r.suf = __shfl_down_sync(0xffffffffu, sg.suf, o);
            r.best = __shfl_down_sync(0xffffffffu, sg.best, o);
            if ((lane & (2 * o - 1)) == 0) sg = seg_combine(sg, r);
        }
        if (lane == 0) {
            if (raw) raw[h] = sg.best;
            if (!skip_count) counts[h] = (uint8_t) min(255, sg.best);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// padded device profiles for the gapped kernel: [(A+1)][Lp] int8, rows >= qlen and residue row A = -128.
// The reversed copy (prof_rev[a][r] = prof[a][qlen-1-r]) serves the start-position pass, which the reference runs
// on query_rev_sequence / composition_bias_rev (StripedSmithWaterman.cpp:1150-1175).
// ------------------------------------------------------------------------------------------------
__global__ void pad_profile_kernel(const int8_t *__restrict__ raw, const QueryDesc *__restrict__ qd, int A,
                                   int8_t *__restrict__ padded) {
    const QueryDesc q = qd[blockIdx.x];
    const int8_t *src = raw + q.raw_off;
    int8_t *fwd = padded + q.pad_off;
    int8_t *rev = padded + q.rev_off;
    int8_t *p16 = padded + q.p16_off;
    const int total = (A + 1) * q.Lp;
    // packed-kernel copy: full 512-row tiles as they are; in the last tile lane l owns rows [l*k16, (l+1)*k16) stored at
    // byte l*kp (kp = k16 rounded up to 4), so that its vector load stays aligned for k16 = 2, 6, 10, 14
    const int last_base = (q.qlen - 1) / 512 * 512, kp = (q.k16 + 3) / 4 * 4;
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const int a = idx / q.Lp, j = idx % q.Lp;
        int8_t f = -128, r = -128, s16 = -128;
        if (a < A && j < q.qlen) { f = src[(size_t) a * q.qlen + j]; r = src[(size_t) a * q.qlen + (q.qlen - 1 - j)]; }
        int row = j;
        if (j >= last_base) {
            const int jl = j - last_base, ln = jl / kp, e = jl % kp;
            row = (ln < 32 && e < q.k16) ? last_base + ln * q.k16 + e : q.qlen;
        }
        if (a < A && row < q.qlen) s16 = src[(size_t) a * q.qlen + row];
        fwd[idx] = f;
        rev[idx] = r;
        p16[idx] = s16;
    }
}

// ------------------------------------------------------------------------------------------------
// A3-A5: affine-gap local alignment, one warp per (query,target) pair, exact int32.
// Reference semantics (SURVEY.md T3-T5, re-verified by tests/test_oracle_vs_ref.py): textbook Gotoh
//   H = max(0, Hdiag + s, E, F);  E' = max(E - ge, H - go);  F' = max(F - ge, H - go)
// (sw_sse2_byte StripedSmithWaterman.cpp:98-299, sw_sse2_word :301-476); end column = first column at which the
// running maximum reaches its final value, end row = smallest row holding it in that column (:233-247, :263-271).
// DIR=-1 runs the same recurrence on the reversed prefixes query[qEnd..0] x target[dbEnd..0] and stops at the first
// column whose maximum equals the forward score (alignStartPosBacktrace :1129-1212, `terminate` :259,:435).
// Word mode adds with adds_epi16, so the diagonal move saturates at 32767 and E and F follow from the saturated H: a pair whose
// exact score passes 32767 reports 32767 at the first cell that reaches it, and the reverse pass meets 32767 exactly.
//
// Lane l owns ROWS consecutive query rows of the current 32*ROWS-row tile and trails lane l-1 by one column; H and F
// of the boundary row travel by __shfl_up.  Query tiles beyond the first pick their top boundary up from a per-warp
// scratch row written by the previous tile.  Profile bytes come from shared memory (staged with a 1-D bulk/TMA copy)
// or, for very long queries, straight from global memory.
// ------------------------------------------------------------------------------------------------
constexpr int SW_ROWS = 8;
constexpr int SW_TILE = 32 * SW_ROWS;
constexpr int SW_WARPS = 4;

template <int DIR, bool SMEM>
__global__ void __launch_bounds__(SW_WARPS * 32)
sw32_kernel(const int8_t *__restrict__ padded, const QueryDesc *__restrict__ qd, const WorkItem *__restrict__ items,
            const PairDesc *__restrict__ pairs, const uint8_t *__restrict__ db, const uint64_t *__restrict__ off,
            const int32_t *__restrict__ len, int A, int go, int ge, int2 *__restrict__ bnd, int bnd_stride,
            int smem_profile, unsigned n_items, unsigned *__restrict__ item_counter, int4 *__restrict__ out) {
    extern __shared__ __align__(16) int8_t smem_prof[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ unsigned next_pair;
    __shared__ unsigned cur_item;

    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * SW_WARPS + (threadIdx.x >> 5);
    int2 *bnd0 = bnd + (size_t) warp_global * 2 * bnd_stride;
    int2 *bnd1 = bnd0 + bnd_stride;
    const int neg_ge = -ge;
    unsigned phase = 0;
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }

  // persistent CTA: items (<= kPairsPerItem pairs of one query, heaviest first) are handed out by a global counter
  while (true) {
    __syncthreads();  // everyone is done with the previous item's profile and next_pair
    if (threadIdx.x == 0) cur_item = atomicAdd(item_counter, 1u);
    __syncthreads();
    const unsigned item_idx = cur_item;
    if (item_idx >= n_items) break;
    const WorkItem item = items[item_idx];
    const QueryDesc q = qd[item.query];
    const int8_t *gprof = padded + (DIR > 0 ? q.pad_off : q.rev_off);
    const int Lp = q.Lp;
    if (threadIdx.x == 0) next_pair = item.p0;
    if (SMEM) {
        const unsigned bytes = (unsigned) ((A + 1) * Lp);  // Lp % 16 == 0
        if (threadIdx.x == 0) {
            mbar_expect_tx(&bar, bytes);
            for (unsigned o = 0; o < bytes; o += 32768u) bulk_g2s(smem_prof + o, gprof + o, min(32768u, bytes - o), &bar);
        }
        __syncthreads();
        mbar_wait(&bar, phase);
        phase ^= 1u;
    } else {
        __syncthreads();
    }

    while (true) {
        unsigned p = 0;
        if (lane == 0) p = atomicAdd(&next_pair, 1u);
        p = __shfl_sync(0xffffffffu, p, 0);
        if (p >= item.p1) break;
        const PairDesc pd = pairs[p];
        const int tl = len[pd.target];
        const uint8_t *tbase = db + off[pd.target];
        int nrows, row0, ncols, target_score;
        if (DIR > 0) { nrows = q.qlen; row0 = 0; ncols = tl; target_score = 0; }
        else { nrows = pd.qend + 1; row0 = q.qlen - 1 - pd.qend; ncols = pd.dbend + 1; tbase += pd.dbend; target_score = pd.score; }

        int gbest = 0, gcol = 0x7fffffff, grow = 0x7fffffff;
        int col_limit = ncols;
        const int tiles = (nrows + SW_TILE - 1) / SW_TILE;
        for (int tile = 0; tile < tiles; tile++) {
            const int8_t *pptr = (SMEM ? (const int8_t *) smem_prof : gprof) + row0 + tile * SW_TILE + lane * SW_ROWS;
            int2 *bnd_rd = (tile & 1) ? bnd0 : bnd1;
            int2 *bnd_wr = (tile & 1) ? bnd1 : bnd0;
            const bool write_bnd = tile + 1 < tiles;
            int H[SW_ROWS], Hg[SW_ROWS], E[SW_ROWS];
#pragma unroll
            for (int j = 0; j < SW_ROWS; j++) { H[j] = 0; Hg[j] = -go; E[j] = 0; }
            int lbest = 0, lcol = 0, lrow = 0;
            int hlast = 0, fout = 0, hdiag_in = 0;
            int res = A, tchunk = A;
            int2 bchunk = make_int2(0, 0);
            int stop_at = -1;
            const int nsteps = col_limit + 31;
            for (int step = 0; step < nsteps; step++) {
                if ((step & 31) == 0) {
                    const int c = step + lane;
                    tchunk = (c < col_limit) ? (int) tbase[(ptrdiff_t) c * DIR] : A;
                    if (tile > 0) bchunk = (c < col_limit) ? bnd_rd[c] : make_int2(0, 0);
                }
                const int r0 = __shfl_sync(0xffffffffu, tchunk, step & 31);
                res = __shfl_up_sync(0xffffffffu, res, 1);
                int hin = __shfl_up_sync(0xffffffffu, hlast, 1);
                int fin = __shfl_up_sync(0xffffffffu, fout, 1);
                if (tile > 0) {
                    const int bh = __shfl_sync(0xffffffffu, bchunk.x, step & 31);
                    const int bf = __shfl_sync(0xffffffffu, bchunk.y, step & 31);
                    if (lane == 0) { hin = bh; fin = bf; }
                } else if (lane == 0) { hin = 0; fin = 0; }
                if (lane == 0) res = r0;
                const int col = step - lane;
                if (col >= 0 && col < col_limit) {
                    const int8_t *pp = pptr + (size_t) res * Lp;
                    int diag = hdiag_in, f = fin, cm = 0;
#pragma unroll
                    for (int j = 0; j < SW_ROWS; j++) {
                        const int s = pp[j];
                        const int e = __viaddmax_s32(E[j], neg_ge, Hg[j]);
                        // adds_epi16 of the reference's word mode: the diagonal move saturates at 32767 (E and F follow from H)
                        const int h = __vimax3_s32_relu(__viaddmin_s32(diag, s, 32767), e, f);
                        diag = H[j];
                        H[j] = h;
                        E[j] = e;
                        const int hg = h - go;
                        Hg[j] = hg;
                        f = __viaddmax_s32(f, neg_ge, hg);
                        cm = max(cm, h);
                    }
                    hlast = H[SW_ROWS - 1];
                    fout = f;
                    if (write_bnd && lane == 31) bnd_wr[col] = make_int2(hlast, f);
                    if (cm > lbest) {
                        lbest = cm; lcol = col;
                        int jr = SW_ROWS - 1;
#pragma unroll
                        for (int j = SW_ROWS - 2; j >= 0; j--) if (H[j] == cm) jr = j;
                        lrow = tile * SW_TILE + lane * SW_ROWS + jr;
                    }
                }
                hdiag_in = hin;
                if (DIR < 0) {
                    if (stop_at < 0 && __any_sync(0xffffffffu, lbest == target_score)) stop_at = step + 31;
                    if (stop_at >= 0 && step >= stop_at) break;
                }
            }
            // warp-wide lexicographic reduction: max score, then min column, then min row
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const int ob = __shfl_xor_sync(0xffffffffu, lbest, o);
                const int oc = __shfl_xor_sync(0xffffffffu, lcol, o);
                const int orow = __shfl_xor_sync(0xffffffffu, lrow, o);
                if (ob > lbest || (ob == lbest && (oc < lcol || (oc == lcol && orow < lrow)))) { lbest = ob; lcol = oc; lrow = orow; }
            }
            if (lbest > gbest || (lbest == gbest && lbest > 0 && (lcol < gcol || (lcol == gcol && lrow < grow)))) {
                gbest = lbest; gcol = lcol; grow = lrow;
            }
            if (DIR < 0 && gbest == target_score && gbest > 0) col_limit = min(col_limit, gcol + 1);
            if (write_bnd) __syncwarp();
        }
        if (lane == 0) out[p] = (gbest > 0) ? make_int4(gbest, gcol, grow, 0) : make_int4(0, -1, -1, 0);
    }
  }
}


// ------------------------------------------------------------------------------------------------
// A3/A4 fast path: score-only affine-gap local DP, TWO targets of the same query per warp, packed in the halves of
// int16x2 registers (DPX VIADDMNMX.S16x2 / VIMNMX3.S16x2).  Same recurrence as sw32_kernel; exact as long as no
// cell exceeds int16 (the host routes pairs that could overflow to sw32_kernel).  The two targets sit on different
// residues at any step, so their int8 profile bytes are fetched separately (vector LDS) and merged + sign-extended
// into one packed score by a single PRMT (selector msb = sign replication).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t prmt_b32(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// One query tile (32*K rows starting at row `row_base`) against the two targets of a warp task, all columns.
// FIRST: tile 0 (no boundary row to read).  Returns the running packed maximum.
// FIND (end positions for known scores): target = packed scores of the two targets (0xFFFF = half not wanted); every lane
// records, per half, the first column in which one of its rows equals the score and the smallest such row
// (key = col << 16 | row); the scan stops 31 steps after every wanted half has been seen somewhere in the warp.
// REV (start positions): the two halves read the REVERSED profile copy at their own, arbitrarily aligned row offsets
// (pptr / pptr_b: byte loads instead of vector loads) and walk their targets backwards from dbEnd (pa_t/pb_t point at it).
template <int K, bool FIRST, bool FIND, bool REV = false>
__device__ __forceinline__ uint32_t sw16_tile(const int8_t *pptr, int Lp, const uint8_t *pa_t, const uint8_t *pb_t, int tla,
                                              int tlb, int ncols, int A, uint32_t neg_ge2, uint32_t neg_go2,
                                              const uint2 *bnd_rd, uint2 *bnd_wr, bool write_bnd, uint32_t best,
                                              uint32_t target = 0, int row_base = 0, uint32_t *key_lo = nullptr,
                                              uint32_t *key_hi = nullptr, const int8_t *pptr_b = nullptr, uint32_t rev_shift = 0) {
    static_assert(K % 2 == 0 && K <= 16 && (!REV || K % 4 == 0), "K even, <= 16 (multiple of 4 in the reverse pass)");
    constexpr int KP = (K + 3) / 4 * 4;   // bytes a lane owns in the profile row (K = 2, 6, 10, 14 leave two unused)
    constexpr int W = KP / 4;
    constexpr int TDIR = REV ? -1 : 1;
    const int lane = threadIdx.x & 31;
    const uint32_t padres = (uint32_t) A | ((uint32_t) A << 8);
    // State per row: H (previous column) and Eh = E + go.  F travels down the column as Fh = F + go.
    // With go >= ge (host-checked) the recurrences become, per cell,
    //   Eh' = max(Eh - ge, Hleft)            T = max(Hdiag + s, Eh' - go, 0)
    //   H   = max(T, Fh - go)                Fh' = max(Fh - ge, T)
    // all in place: a descending pass (E, T) then an ascending pass (F chain, one dependent op per row).
    // Lanes that have not reached column 0 yet, or are past the last column, see the pad residue (profile -128):
    // their cells stay 0 / stay below every real cell, so no per-step range predicate is needed.
    uint32_t H[K], Eh[K];
#pragma unroll
    for (int j = 0; j < K; j++) { H[j] = 0; Eh[j] = 0; }
    uint32_t hlast = 0, fout = 0, hdiag_in = 0;
    uint32_t res = padres, tchunk = padres;
    uint2 bchunk = make_uint2(0, 0);
    int nsteps = ncols + 31;
    bool stopping = false;
    uint32_t tgt = target;
    const bool want_lo = FIND && (target & 0xffffu) != 0xffffu, want_hi = FIND && (target >> 16) != 0xffffu;
    uint32_t klo = FIND ? *key_lo : 0u, khi = FIND ? *key_hi : 0u;
    // REV: the rows a half gained by rounding its start down to a word (rev_shift = shift_lo | shift_hi << 8, each 0..3)
    // sit in lane 0 of the first tile and score as pad there, so they stay 0 like the boundary above row 0
    uint32_t rv_and[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, rv_or[3] = {0u, 0u, 0u};
    if (REV && FIRST && lane == 0) {
#pragma unroll
        for (int j = 0; j < 3; j++) {
            if (j < (int) (rev_shift & 0xffu)) { rv_and[j] &= 0xffff0000u; rv_or[j] |= 0x0000ff80u; }
            if (j < (int) (rev_shift >> 8)) { rv_and[j] &= 0x0000ffffu; rv_or[j] |= 0xff800000u; }
        }
    }
    const int row_lo = row_base + lane * K - (int) (rev_shift & 0xffu), row_hi = row_base + lane * K - (int) (rev_shift >> 8);
    for (int step = 0; step < nsteps; step++) {
        if ((step & 31) == 0) {
            const int c = step + lane;
            const uint32_t ra = (c < tla) ? (uint32_t) pa_t[c * TDIR] : (uint32_t) A;
            const uint32_t rb = (c < tlb) ? (uint32_t) pb_t[c * TDIR] : (uint32_t) A;
            tchunk = ra | (rb << 8);
            if (!FIRST) bchunk = (c < ncols) ? bnd_rd[c] : make_uint2(0, 0);
        }
        const uint32_t r0 = __shfl_sync(0xffffffffu, tchunk, step & 31);
        res = __shfl_up_sync(0xffffffffu, res, 1);
        uint32_t hin = __shfl_up_sync(0xffffffffu, hlast, 1);
        uint32_t fin = __shfl_up_sync(0xffffffffu, fout, 1);
        if (!FIRST) {
            const uint32_t bh = __shfl_sync(0xffffffffu, bchunk.x, step & 31);
            const uint32_t bf = __shfl_sync(0xffffffffu, bchunk.y, step & 31);
            if (lane == 0) { hin = bh; fin = bf; }
        } else if (lane == 0) { hin = 0; fin = 0; }
        if (lane == 0) res = r0;
        const int8_t *ppa = pptr + (res & 0xffu) * (uint32_t) Lp;
        const int8_t *ppb = (REV ? pptr_b : pptr) + (res >> 8) * (uint32_t) Lp;
        uint32_t wa[W], wb[W];
        if constexpr (REV) {   // word aligned only (each half starts at its own row offset rounded down to 4)
#pragma unroll
            for (int w = 0; w < W; w++) {
                wa[w] = reinterpret_cast<const uint32_t *>(ppa)[w];
                wb[w] = reinterpret_cast<const uint32_t *>(ppb)[w];
            }
        } else if constexpr (KP == 16) {
            const uint4 va = *reinterpret_cast<const uint4 *>(ppa), vb = *reinterpret_cast<const uint4 *>(ppb);
            wa[0] = va.x; wa[1] = va.y; wa[2] = va.z; wa[3] = va.w;
            wb[0] = vb.x; wb[1] = vb.y; wb[2] = vb.z; wb[3] = vb.w;
        } else if constexpr (KP == 8) {
            const uint2 va = *reinterpret_cast<const uint2 *>(ppa), vb = *reinterpret_cast<const uint2 *>(ppb);
            wa[0] = va.x; wa[1] = va.y; wb[0] = vb.x; wb[1] = vb.y;
        } else {
#pragma unroll
            for (int w = 0; w < W; w++) {
                wa[w] = reinterpret_cast<const uint32_t *>(ppa)[w];
                wb[w] = reinterpret_cast<const uint32_t *>(ppb)[w];
            }
        }
        constexpr uint32_t SEL[4] = {0xC480u, 0xD591u, 0xE6A2u, 0xF7B3u};
#pragma unroll
        for (int j = K - 1; j >= 0; j--) {
            uint32_t sc = prmt_b32(wa[j >> 2], wb[j >> 2], SEL[j & 3]);
            if (REV && FIRST && j < 3) sc = (sc & rv_and[j]) | rv_or[j];
            Eh[j] = __viaddmax_s16x2(Eh[j], neg_ge2, H[j]);
            const uint32_t e = __vadd2(Eh[j], neg_go2);
            H[j] = __viaddmax_s16x2_relu(j > 0 ? H[j - 1] : hdiag_in, sc, e);
        }
        uint32_t f = fin;
#pragma unroll
        for (int j = 0; j < K; j++) {
            const uint32_t fn = __viaddmax_s16x2(f, neg_ge2, H[j]);
            H[j] = __viaddmax_s16x2(f, neg_go2, H[j]);
            f = fn;
        }
        if (!FIND) {
#pragma unroll
            for (int j = 0; j < K; j += 2) best = __vimax3_s16x2(best, H[j], H[j + 1]);
        } else {
            uint32_t cm = 0;
#pragma unroll
            for (int j = 0; j < K; j += 2) cm = __vimax3_s16x2(cm, H[j], H[j + 1]);
            const uint32_t dx = cm ^ tgt;
            if ((dx & 0xffffu) == 0 || dx < 0x10000u) {          // rare: a lane reaches the final score of a half
                const int col = step - lane;
                if ((dx & 0xffffu) == 0) {
                    int jr = K - 1;
#pragma unroll
                    for (int j = K - 2; j >= 0; j--) if ((H[j] & 0xffffu) == (target & 0xffffu)) jr = j;
                    klo = ((uint32_t) col << 16) | (uint32_t) (row_lo + jr);
                    tgt |= 0xffffu;                               // recorded: this half cannot match again
                }
                if (dx < 0x10000u) {
                    int jr = K - 1;
#pragma unroll
                    for (int j = K - 2; j >= 0; j--) if ((H[j] >> 16) == (target >> 16)) jr = j;
                    khi = ((uint32_t) col << 16) | (uint32_t) (row_hi + jr);
                    tgt |= 0xffff0000u;
                }
            }
            // a late look only delays the stop: by then every lane has passed the recorded column anyway
            if ((step & 7) == 7 && !stopping) {
                const bool seen_lo = !want_lo || __any_sync(0xffffffffu, klo != 0xffffffffu);
                const bool seen_hi = !want_hi || __any_sync(0xffffffffu, khi != 0xffffffffu);
                if (seen_lo && seen_hi) { stopping = true; nsteps = min(nsteps, step + 32); }
            }
        }
        hlast = H[K - 1];
        fout = f;
        if (write_bnd && lane == 31 && step >= 31) bnd_wr[step - 31] = make_uint2(hlast, f);
        hdiag_in = hin;
    }
    if (write_bnd) __syncwarp();
    if (FIND) { *key_lo = klo; *key_hi = khi; }
    return best;
}

template <int K, bool FIND, bool REV>
__device__ __forceinline__ uint32_t sw16_tile_any(bool first, const int8_t *pptr, int Lp, const uint8_t *pa_t, const uint8_t *pb_t,
                                                  int tla, int tlb, int ncols, int A, uint32_t neg_ge2, uint32_t neg_go2,
                                                  const uint2 *bnd_rd, uint2 *bnd_wr, bool write_bnd, uint32_t best,
                                                  uint32_t target = 0, int row_base = 0, uint32_t *key_lo = nullptr,
                                                  uint32_t *key_hi = nullptr, const int8_t *pptr_b = nullptr, uint32_t rev_shift = 0) {
    if (first) return sw16_tile<K, true, FIND, REV>(pptr, Lp, pa_t, pb_t, tla, tlb, ncols, A, neg_ge2, neg_go2, bnd_rd, bnd_wr, write_bnd,
                                                    best, target, row_base, key_lo, key_hi, pptr_b, rev_shift);
    return sw16_tile<K, false, FIND, REV>(pptr, Lp, pa_t, pb_t, tla, tlb, ncols, A, neg_ge2, neg_go2, bnd_rd, bnd_wr, write_bnd, best,
                                          target, row_base, key_lo, key_hi, pptr_b, rev_shift);
}

// All pairs of one work item.  The query is cut into full 512-row tiles (16 rows per lane) plus one last tile whose
// rows-per-lane flavour (4/8/12/16, item.pad_) is the smallest that covers the remainder.
// MODE 0: score.  MODE 1: end positions for known scores (forward).  MODE 2: start positions -- the same search on the
// reversed prefixes query[qEnd..0] x target[dbEnd..0] (alignStartPosBacktrace, StripedSmithWaterman.cpp:1129-1212).
template <bool SMEM, int MODE>
__device__ __forceinline__ void sw16_item(const int8_t *prof_base, const QueryDesc &q, const WorkItem &item,
                                          const PairDesc *__restrict__ pairs, const uint8_t *__restrict__ db,
                                          const uint64_t *__restrict__ off, const int32_t *__restrict__ len, int A, int go,
                                          int ge, uint2 *bnd0, uint2 *bnd1, unsigned *next_pair_ptr, int32_t *__restrict__ out,
                                          const int32_t *__restrict__ dv_score, const int32_t *__restrict__ dv_pos) {
    constexpr bool FIND = MODE != 0, REV = MODE == 2;
    const int lane = threadIdx.x & 31;
    const int Lp = q.Lp;
    const uint32_t neg_ge2 = pack16(-ge, -ge), neg_go2 = pack16(-go, -go);
    while (true) {
        unsigned p = 0;
        if (lane == 0) p = atomicAdd(next_pair_ptr, 2u);
        p = __shfl_sync(0xffffffffu, p, 0);
        if (p >= item.p1) break;
        const bool has_b = p + 1 < item.p1;
        const PairDesc pda = pairs[p], pdb = has_b ? pairs[p + 1] : pairs[p];
        const uint32_t ta = pda.target, tb = pdb.target;
        int tla, tlb, nrows, offa = 0, offb = 0;
        uint32_t rev_shift = 0;
        const uint8_t *pa_t = db + off[ta], *pb_t = db + off[tb];
        // chained launches (dv_score != nullptr): scores / end positions come from the previous kernel's output in plan
        // order, PairDesc.qend carries the caller's gate; a half with nothing to find runs with zero columns
        int sca = pda.score, scb = pdb.score, qea = pda.qend, qeb = pdb.qend, dea = pda.dbend, deb = pdb.dbend;
        bool wa = true, wb = has_b;
        if (FIND && dv_score != nullptr) {
            sca = dv_score[p]; scb = has_b ? dv_score[p + 1] : 0;
            wa = sca > 0; wb = has_b && scb > 0;
            if (REV) {
                wa = wa && pda.qend != 0; wb = wb && pdb.qend != 0;
                dea = wa ? dv_pos[2 * p] : 0; qea = wa ? dv_pos[2 * p + 1] : 0;
                deb = wb ? dv_pos[2 * (p + 1)] : 0; qeb = wb ? dv_pos[2 * (p + 1) + 1] : 0;
            }
            if (!wa && !wb) {
                if (lane == 0) {
                    out[2 * p] = 65535; out[2 * p + 1] = 65535;
                    if (has_b) { out[2 * (p + 1)] = 65535; out[2 * (p + 1) + 1] = 65535; }
                }
                continue;
            }
        }
        if (REV) {
            tla = wa ? dea + 1 : 0; tlb = wb ? deb + 1 : 0;
            pa_t += dea; pb_t += deb;
            offa = q.qlen - 1 - qea; offb = q.qlen - 1 - qeb;
            rev_shift = (uint32_t) (offa & 3) | ((uint32_t) (offb & 3) << 8);   // word-align each half's first profile row
            offa &= ~3; offb &= ~3;
            nrows = max(wa ? qea + 1 + (int) (rev_shift & 0xffu) : 0, wb ? qeb + 1 + (int) (rev_shift >> 8) : 0);
        } else {
            tla = wa ? len[ta] : 0; tlb = wb ? len[tb] : 0;
            nrows = q.qlen;
        }
        const int n_full = (nrows - 1) / 512;                  // tiles of 512 rows before the last tile
        const int rem = nrows - n_full * 512;                  // 1..512 rows in the last tile
        const int k_last = REV ? min(16, ((rem + 31) / 32 + 3) / 4 * 4) : (int) item.pad_;
        int ncols = max(tla, tlb);
        uint32_t best = 0;
        uint32_t target = 0, key_lo = 0xffffffffu, key_hi = 0xffffffffu, gkey_lo = 0xffffffffu, gkey_hi = 0xffffffffu;
        if (FIND) target = (wa ? (uint32_t) sca & 0xffffu : 0xffffu) | ((wb ? (uint32_t) scb & 0xffffu : 0xffffu) << 16);
        for (int tile = 0; tile <= n_full; tile++) {
            const uint2 *bnd_rd = (tile & 1) ? bnd0 : bnd1;
            uint2 *bnd_wr = (tile & 1) ? bnd1 : bnd0;
            const bool last = tile == n_full;
            const int kk = last ? k_last : 16;
            // REV: a half whose rectangle has fewer rows than its partner's keeps reading, so clamp into the pad columns
            // at the end of the profile row (everything beyond the half's own rows must read as pad anyway)
            const int kp = (kk + 3) & ~3;
            const int8_t *pl = prof_base + min(offa + tile * 512 + lane * kp, Lp - 16);
            const int8_t *plb = prof_base + min(offb + tile * 512 + lane * kp, Lp - 16);
#define B200_SW16_TILE(KK) best = sw16_tile_any<KK, FIND, REV>(tile == 0, pl, Lp, pa_t, pb_t, tla, tlb, ncols, A, neg_ge2, neg_go2, bnd_rd, \
                                                              bnd_wr, !last, best, target, tile * 512, &key_lo, &key_hi, plb, rev_shift)
            if (REV || (kk & 3) == 0) {
                switch (kk) {
                    case 4: B200_SW16_TILE(4); break;
                    case 8: B200_SW16_TILE(8); break;
                    case 12: B200_SW16_TILE(12); break;
                    default: B200_SW16_TILE(16); break;
                }
            } else if constexpr (!REV) {
                switch (kk) {
                    case 2: B200_SW16_TILE(2); break;
                    case 6: B200_SW16_TILE(6); break;
                    case 10: B200_SW16_TILE(10); break;
                    default: B200_SW16_TILE(14); break;
                }
            }
#undef B200_SW16_TILE
            if (FIND) {   // earliest (column, row) so far per half; later tiles only need the columns up to it
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    key_lo = min(key_lo, __shfl_xor_sync(0xffffffffu, key_lo, o));
                    key_hi = min(key_hi, __shfl_xor_sync(0xffffffffu, key_hi, o));
                }
                gkey_lo = min(gkey_lo, key_lo); gkey_hi = min(gkey_hi, key_hi);
                key_lo = 0xffffffffu; key_hi = 0xffffffffu;   // every lane may record again in the next tile
                const int lim_lo = (target & 0xffffu) == 0xffffu ? 0 : (gkey_lo == 0xffffffffu ? tla : (int) (gkey_lo >> 16) + 1);
                const int lim_hi = (target >> 16) == 0xffffu ? 0 : (gkey_hi == 0xffffffffu ? tlb : (int) (gkey_hi >> 16) + 1);
                ncols = min(ncols, max(lim_lo, lim_hi));
            }
        }
        if (!FIND) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(0xffffffffu, best, o));
            if (lane == 0) {
                out[p] = (int) (best & 0xffffu);
                if (has_b) out[p + 1] = (int) (best >> 16);
            }
        } else if (lane == 0) {
            out[2 * p] = (int) (gkey_lo >> 16); out[2 * p + 1] = (int) (gkey_lo & 0xffffu);
            if (has_b) { out[2 * (p + 1)] = (int) (gkey_hi >> 16); out[2 * (p + 1) + 1] = (int) (gkey_hi & 0xffffu); }
        }
    }
}

// One launch covers every query length: items carry the rows-per-lane flavour (4/8/12/16) chosen for their query.
template <bool SMEM, int WARPS, int MODE>
__global__ void __launch_bounds__(WARPS * 32, 24 / WARPS)
sw16_kernel(const int8_t *__restrict__ padded, const QueryDesc *__restrict__ qd, const WorkItem *__restrict__ items,
            const PairDesc *__restrict__ pairs, const uint8_t *__restrict__ db, const uint64_t *__restrict__ off,
            const int32_t *__restrict__ len, int A, int go, int ge, uint2 *__restrict__ bnd, int bnd_stride,
            unsigned n_items, unsigned *__restrict__ item_counter, int32_t *__restrict__ out,
            const int32_t *__restrict__ dv_score, const int32_t *__restrict__ dv_pos) {
    extern __shared__ __align__(16) int8_t smem_prof[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ unsigned next_pair;
    __shared__ unsigned cur_item;

    const int warp_global = blockIdx.x * WARPS + (threadIdx.x >> 5);
    uint2 *bnd0 = bnd + (size_t) warp_global * 2 * bnd_stride;
    uint2 *bnd1 = bnd0 + bnd_stride;
    unsigned phase = 0;
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) cur_item = atomicAdd(item_counter, 1u);
        __syncthreads();
        const unsigned item_idx = cur_item;
        if (item_idx >= n_items) break;
        const WorkItem item = items[item_idx];
        const QueryDesc q = qd[item.query];
        const int8_t *gprof = padded + (MODE == 2 ? q.rev_off : q.p16_off);
        if (threadIdx.x == 0) next_pair = item.p0;
        if (SMEM) {
            const unsigned bytes = (unsigned) ((A + 1) * q.Lp);
            if (threadIdx.x == 0) {
                mbar_expect_tx(&bar, bytes);
                for (unsigned o = 0; o < bytes; o += 32768u) bulk_g2s(smem_prof + o, gprof + o, min(32768u, bytes - o), &bar);
            }
            __syncthreads();
            mbar_wait(&bar, phase);
            phase ^= 1u;
        } else {
            __syncthreads();
        }
        const int8_t *pb = SMEM ? (const int8_t *) smem_prof : gprof;
        sw16_item<SMEM, MODE>(pb, q, item, pairs, db, off, len, A, go, ge, bnd0, bnd1, &next_pair, out, dv_score, dv_pos);
    }
}

// ================================================================================================
// host side
// ================================================================================================
namespace {

int set_err(b200_ctx *ctx, int code, const char *msg) { return b200_set_err(ctx, code, msg); }

// int16 safety of the packed gapped kernels.  No local alignment (and no intermediate H/E/F value, each the score of some partial
// path) can exceed either  min(qlen, tlen) * (largest profile entry)  or  the sum over query rows of the row's best entry (every
// aligned row contributes at most that, unaligned rows nothing).  The second bound is what keeps ordinary long pairs on the packed
// path: a sequence profile's row maxima average ~11 (its self score), half its largest entry.
void profile_bounds(const int8_t *pr, int A, int qlen, int &smax, int64_t &qsum) {
    int m = 1;
    int64_t sum = 0;
    for (int j = 0; j < qlen; j++) {
        int rowmax = 0;
        for (int a = 0; a < A; a++) rowmax = std::max(rowmax, (int) pr[(size_t) a * qlen + j]);
        m = std::max(m, rowmax);
        sum += rowmax;
    }
    smax = m; qsum = sum;
}
inline bool int16_safe(int smax, int64_t qsum, int qlen, int tlen) {
    return std::min((int64_t) std::min(qlen, tlen) * smax, qsum) < 32000;
}

struct ScanCfg { int G, K; };
// capacity 2*G*K rows, ascending: 32-row steps up to 512 (G=8), 64-row steps up to 1024 (G=16), 128-row steps up to 2048 (G=32)
#define B200_SCAN_CFGS(X) \
    X(0, 8, 4) X(1, 8, 6) X(2, 8, 8) X(3, 8, 10) X(4, 8, 12) X(5, 8, 14) \
    X(6, 8, 16) X(7, 8, 18) X(8, 8, 20) X(9, 8, 22) X(10, 8, 24) X(11, 8, 26) \
    X(12, 8, 28) X(13, 8, 30) X(14, 8, 32) X(15, 16, 18) X(16, 16, 20) X(17, 16, 22) \
    X(18, 16, 24) X(19, 16, 26) X(20, 16, 28) X(21, 16, 30) X(22, 16, 32) X(23, 32, 18) \
    X(24, 32, 20) X(25, 32, 22) X(26, 32, 24) X(27, 32, 26) X(28, 32, 28) X(29, 32, 30) \
    X(30, 32, 32)
#define B200_SCAN_ENTRY(n, g, k) {g, k},
const ScanCfg kScanCfgs[] = {B200_SCAN_CFGS(B200_SCAN_ENTRY)};
#undef B200_SCAN_ENTRY

constexpr int kScanCounters = 64;   // one work-unit counter per launch of a batch (launches of one batch may run concurrently)

// nq counts queries, or quads when QUAD (qd then holds 4 * nq descriptors, quad by quad)
template <int G, int K, bool TILED, bool QUAD>
cudaError_t launch_scan_cfg(b200_ctx *ctx, const int8_t *raw, const QueryDesc *qd, int nq, uint8_t *dense, cudaStream_t stream, int counter_slot) {
    const int threads = QUAD ? kScanQuadThreads : 256;
    size_t smem = (size_t) 2 * (ctx->alphabet + 1) * (QUAD ? 4 : 1) * (K * G + ((G == 8 && K % 4 == 2 && !QUAD) ? 16 : 0)) * sizeof(uint32_t);
    if (QUAD) smem = std::max<size_t>(smem, kScanQuadMinSmem);
    cudaError_t e = cudaFuncSetAttribute(ungapped_scan_kernel<G, K, TILED, QUAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ungapped_scan_kernel<G, K, TILED, QUAD>, threads, smem);
    if (e != cudaSuccess) return e;
    // a quad CTA allocates all of an SM's tensor memory: a second one on the SM would block in tcgen05.alloc
    if (QUAD && per_sm != 1) return cudaErrorInvalidConfiguration;
    per_sm = std::max(per_sm, 1);
    const uint64_t resident = (uint64_t) ctx->sm_count * per_sm;
    const uint32_t groups_per_cta = QUAD ? threads / 32 : 256 / G;   // targets per CTA-wide pass
    // ~16 work units per resident CTA over the whole launch, each a multiple of one CTA-wide pass over the sorted targets
    uint64_t unit_targets = ((uint64_t) ctx->n_seq * nq + resident * 16 - 1) / (resident * 16);
    unit_targets = std::max<uint64_t>(groups_per_cta, (unit_targets + groups_per_cta - 1) / groups_per_cta * groups_per_cta);
    if (TILED) unit_targets = std::min<uint64_t>(unit_targets, 4 * groups_per_cta);   // bounds the tile-boundary scratch
    const uint32_t units_per_query = (uint32_t) ((ctx->n_seq + unit_targets - 1) / unit_targets);
    const uint64_t ctas = std::max<uint64_t>(1, std::min<uint64_t>(resident, (uint64_t) units_per_query * nq));
    e = ctx->counter.reserve(sizeof(unsigned) * kScanCounters);
    unsigned *counter = ctx->counter.as<unsigned>() + counter_slot;
    if (e == cudaSuccess) e = cudaMemsetAsync(counter, 0, sizeof(unsigned), stream);
    uint32_t slot_words = 0;
    if (TILED && e == cudaSuccess) {
        slot_words = (uint32_t) (round_up((uint64_t) ctx->max_len, 16) / 2 + 8);
        e = ctx->bnd.reserve(sizeof(uint32_t) * (size_t) slot_words * unit_targets * ctas);
    }
    if (e != cudaSuccess) return e;
    ungapped_scan_kernel<G, K, TILED, QUAD><<<(unsigned) ctas, threads, smem, stream>>>(
        raw, qd, ctx->d_res, ctx->d_off, ctx->d_len, ctx->d_order, (uint32_t) ctx->n_seq, ctx->alphabet, dense, (uint32_t) nq, units_per_query,
        (uint32_t) unit_targets, counter, TILED ? ctx->bnd.as<uint32_t>() : nullptr, slot_words);
    ctx->launches++;
    return cudaGetLastError();
}

template <int G, int K>
cudaError_t launch_scan_quads(b200_ctx *ctx, const int8_t *raw, const QueryDesc *qd, int nq, uint8_t *dense, cudaStream_t stream, int counter_slot) {
    if constexpr (G == 8) return launch_scan_cfg<8, K, false, true>(ctx, raw, qd, nq, dense, stream, counter_slot);
    return cudaErrorInvalidValue;
}

// queries of one launch must share a (G,K) configuration; the caller groups them by capacity class (quad: nq quads of 4 queries)
cudaError_t launch_scan(b200_ctx *ctx, int cfg, bool quad, const int8_t *raw, const QueryDesc *qd, int nq, uint8_t *dense, cudaStream_t stream,
                        int counter_slot) {
    switch (cfg) {
#define B200_SCAN_CASE(n, g, k) \
    case n: return quad ? launch_scan_quads<g, k>(ctx, raw, qd, nq, dense, stream, counter_slot) \
                        : launch_scan_cfg<g, k, false, false>(ctx, raw, qd, nq, dense, stream, counter_slot);
        B200_SCAN_CFGS(B200_SCAN_CASE)
#undef B200_SCAN_CASE
        default: return launch_scan_cfg<32, 32, true, false>(ctx, raw, qd, nq, dense, stream, counter_slot);   // queries longer than 2047: row tiles of 2048
    }
}

// quads need the R tensor-memory columns of every residue row (pad row included) to fit the SM's 512; R is largest at K = 22
bool scan_quads_fit(int alphabet) { return (alphabet + 1) * scan_quad_R(22) <= kScanTmemCols; }

int scan_cfg_for(int qlen) {
    const int n = (int) (sizeof(kScanCfgs) / sizeof(kScanCfgs[0]));
    static const bool coarse = getenv("B200_SCAN_COARSE") != nullptr;   // experiments: the round-0 class list only
    for (int i = 0; i < n; i++) {
        if (coarse && kScanCfgs[i].K % 4 != 0) continue;     // 64/128/256-row steps only
        if (2 * kScanCfgs[i].G * kScanCfgs[i].K >= qlen + 1) return i;
    }
    return n;  // tiled long-query variant
}

// rows per lane (2,4,...,16) of the LAST tile of the packed kernel for a query length; every earlier tile is 512 rows
int sw16_k_for(int qlen) {
    const int rem = qlen - (qlen - 1) / 512 * 512;  // 1..512 rows left for the last tile
    return std::min(16, (rem + 63) / 64 * 2);
}

// stage raw profiles + descriptors for a set of queries; fills h_qd (pad offsets only when with_pad)
int stage_queries(b200_ctx *ctx, const b200_query *queries, int nq, bool with_pad, std::vector<QueryDesc> &h_qd) {
    const int A = ctx->alphabet;
    h_qd.resize(nq);
    uint64_t raw_bytes = 0, pad_bytes = 0;
    for (int i = 0; i < nq; i++) {
        if (queries[i].profile == nullptr || queries[i].qlen <= 0) return set_err(ctx, B200_ERR_ARG, "query without profile or qlen <= 0");
        QueryDesc &d = h_qd[i];
        d.qlen = queries[i].qlen;
        d.bias = queries[i].bias;
        d.raw_off = raw_bytes;
        raw_bytes += round_up((uint64_t) A * d.qlen, 16);
        d.Lp = (int) round_up((uint64_t) d.qlen, 128) + 512;
        d.pad_off = pad_bytes;
        d.rev_off = pad_bytes + (uint64_t) (A + 1) * d.Lp;
        d.p16_off = pad_bytes + 2 * (uint64_t) (A + 1) * d.Lp;
        pad_bytes += 3 * (uint64_t) (A + 1) * d.Lp;
        d.k16 = sw16_k_for(d.qlen);
    }
    std::vector<int8_t> h_raw(raw_bytes, 0);
    for (int i = 0; i < nq; i++) memcpy(h_raw.data() + h_qd[i].raw_off, queries[i].profile, (size_t) A * h_qd[i].qlen);
    CU_TRY(ctx, ctx->raw.reserve(raw_bytes));
    CU_TRY(ctx, ctx->qdesc.reserve(sizeof(QueryDesc) * nq));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->raw.p, h_raw.data(), raw_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->qdesc.p, h_qd.data(), sizeof(QueryDesc) * nq, cudaMemcpyHostToDevice, ctx->stream));
    if (with_pad) {
        CU_TRY(ctx, ctx->pad.reserve(pad_bytes));
        pad_profile_kernel<<<nq, 256, 0, ctx->stream>>>(ctx->raw.as<int8_t>(), ctx->qdesc.as<QueryDesc>(), A, ctx->pad.as<int8_t>());
        ctx->launches++;
        CU_TRY(ctx, cudaGetLastError());
    }
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // h_raw goes out of scope
    return B200_OK;
}

}  // namespace

// ---- jobs ------------------------------------------------------------------------------------------
struct b200_job {
    b200_ctx *ctx = nullptr;
    int kind = 0;  // 1 scan, 2 sw forward
    uint64_t cells = 0;
    // scan
    int nq = 0, thr = 0;
    uint32_t k = 0;
    struct ScanGroup { int cfg; bool quad; std::vector<int> queries; };   // one configuration's launch; quad: 4 queries per quad
    std::vector<ScanGroup> scan_groups;
    DevBuf raw, qdesc, qdesc_grouped, dense, hits, nhits, pad, part_hist;
    std::vector<int> grouped_order;  // position -> original query index
    // sw
    uint64_t n_pairs = 0;
    int go = 0, ge = 0;
    DevBuf pairs, items, out4, bnd;
    uint32_t n_items = 0;
    int bnd_stride = 0;
    int smem_bytes = 0, smem_profile = 0;
    std::vector<uint32_t> perm;        // sorted position -> caller index
    std::vector<b200_pair> h_pairs;    // caller order
    std::vector<int32_t> h_qlen, h_bias;
    // kind 3 (score-only): one part per kernel flavour (packed K in {4,8,12,16}, or 0 = int32 fallback)
    struct Part {
        int K = 0;
        std::vector<uint32_t> perm;
        DevBuf pairs, items, out;
        uint32_t n_items = 0, n_pairs = 0;
        int max_Lp = 0;
    };
    std::vector<Part *> parts;
    cudaEvent_t done = nullptr;   // recorded on the ctx stream behind the job's last kernel
    bool ran = false;
    void free_all() {
        if (done) { cudaEventDestroy(done); done = nullptr; }
        for (Part *pt : parts) { pt->pairs.release(); pt->items.release(); pt->out.release(); delete pt; }
        parts.clear();
        raw.release(); qdesc.release(); qdesc_grouped.release(); dense.release(); hits.release(); nhits.release(); part_hist.release();
        pad.release(); pairs.release(); items.release(); out4.release(); bnd.release();
    }
};

// All b200_* functions below are declared extern "C" in include/b200_align.h and keep that linkage here.

int b200_create(int device, b200_ctx **out) {
    if (out == nullptr) return B200_ERR_ARG;
    *out = nullptr;
    b200_ctx *ctx = new b200_ctx();
    ctx->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 3 && e == cudaSuccess; i++) e = cudaStreamCreateWithFlags(&ctx->side[i], cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete ctx; return B200_ERR_CUDA; }
    for (int i = 0; i < 16; i++) cudaEventCreate(&ctx->ev[i]);
    cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
    for (int i = 0; i < 3; i++) cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major; ctx->cc_minor = prop.minor;
    ctx->hbm = prop.totalGlobalMem;
    ctx->max_smem_optin = (int) prop.sharedMemPerBlockOptin;
    *out = ctx;
    return B200_OK;
}

static void db_free(b200_ctx *ctx) {
    if (ctx->d_res) cudaFree(ctx->d_res);
    if (ctx->d_off) cudaFree(ctx->d_off);
    if (ctx->d_len) cudaFree(ctx->d_len);
    if (ctx->d_order) cudaFree(ctx->d_order);
    ctx->d_res = nullptr; ctx->d_off = nullptr; ctx->d_len = nullptr; ctx->d_order = nullptr;
    ctx->n_seq = 0; ctx->n_res = 0;
}

void b200_destroy(b200_ctx *ctx) {
    if (ctx == nullptr) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    db_free(ctx);
    b200_ascii_db_free(ctx);
    DevBuf *bufs[] = {&ctx->raw, &ctx->pad, &ctx->qdesc, &ctx->dense, &ctx->hits, &ctx->nhits, &ctx->pairs, &ctx->items,
                      &ctx->out4, &ctx->bnd, &ctx->ids, &ctx->diags, &ctx->counts, &ctx->rawout, &ctx->counter};
    for (DevBuf *b : bufs) b->release();
    for (int i = 0; i < 16; i++) cudaEventDestroy(ctx->ev[i]);
    cudaEventDestroy(ctx->ev_fork);
    for (int i = 0; i < 3; i++) { cudaEventDestroy(ctx->ev_join[i]); cudaStreamDestroy(ctx->side[i]); }
    cudaStreamDestroy(ctx->copy_stream);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *b200_last_error(const b200_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

int b200_device_info(const b200_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, uint64_t *hbm_bytes) {
    if (ctx == nullptr) return B200_ERR_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (hbm_bytes) *hbm_bytes = ctx->hbm;
    return B200_OK;
}

uint64_t b200_launch_count(const b200_ctx *ctx) { return ctx ? ctx->launches : 0; }
float b200_last_kernel_ms(const b200_ctx *ctx) { return ctx ? ctx->last_kernel_ms : 0.f; }

int b200_event_record(b200_ctx *ctx, int slot) {
    if (ctx == nullptr || slot < 0 || slot >= 16) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaEventRecord(ctx->ev[slot], ctx->stream));
    return B200_OK;
}

int b200_event_elapsed_ms(b200_ctx *ctx, int a, int b, float *ms) {
    if (ctx == nullptr || ms == nullptr || a < 0 || a >= 16 || b < 0 || b >= 16) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaEventSynchronize(ctx->ev[b]));
    CU_TRY(ctx, cudaEventElapsedTime(ms, ctx->ev[a], ctx->ev[b]));
    return B200_OK;
}

int b200_sync(b200_ctx *ctx) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return B200_OK;
}

// ---- DB -------------------------------------------------------------------------------------------
// Common body of b200_db_load / b200_db_load_padded.  src(i) = first residue of sequence i, len[i] its length; bytes >= mask_from
// (the +32 soft-mask bit of the padded GPU DB, makepaddedseqdb.cpp:77-86) become X = alphabet-1, as runFilterOnCpu treats masked
// residues (ungappedprefilter.cpp:401-404); mask_from = 256 disables that.  The re-layout (16-byte aligned, padded with code
// `alphabet`) runs on all host threads: at 20 M sequences this is 7.5 GB of bytes.
int b200_db_load_impl(b200_ctx *ctx, const uint8_t *base, const uint64_t *starts, const int32_t *lens, uint64_t n_seq, int alphabet,
                      int mask_from, uint64_t n_res, bool strip_mask) {
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    db_free(ctx);
    std::vector<uint64_t> h_off(n_seq);
    ctx->h_len.assign(lens, lens + n_seq);
    uint64_t total = 0;
    int max_len = 0;
    for (uint64_t i = 0; i < n_seq; i++) {
        h_off[i] = total;
        max_len = std::max(max_len, (int) lens[i]);
        total += round_up((uint64_t) lens[i], 16);
    }
    total += 32;
    uint8_t *h_res = nullptr;
    CU_TRY(ctx, cudaMallocHost(&h_res, total));
    const unsigned nt = std::max(1u, std::min(64u, std::thread::hardware_concurrency()));
    std::vector<int> bad(nt, 0);
    {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; t++)
            th.emplace_back([&, t]() {
                const uint64_t i0 = n_seq * t / nt, i1 = n_seq * (t + 1) / nt;
                const uint64_t b0 = i0 < n_seq ? h_off[i0] : total - 32, b1 = i1 < n_seq ? h_off[i1] : total;
                memset(h_res + b0, alphabet, b1 - b0);
                for (uint64_t i = i0; i < i1; i++) {
                    const uint8_t *src = base + starts[i];
                    uint8_t *dst = h_res + h_off[i];
                    for (int32_t j = 0; j < lens[i]; j++) {
                        uint8_t c = src[j];
                        if (c >= mask_from) c = strip_mask ? (uint8_t) (c - 32) : (uint8_t) (alphabet - 1);
                        if (c >= alphabet) bad[t] = 1;
                        dst[j] = c;
                    }
                }
            });
        for (auto &x : th) x.join();
    }
    for (unsigned t = 0; t < nt; t++)
        if (bad[t]) { cudaFreeHost(h_res); return set_err(ctx, B200_ERR_ARG, "b200_db_load: residue code >= alphabet (strip the +32 mask bit first)"); }
    std::vector<uint32_t> order(n_seq);
    std::iota(order.begin(), order.end(), 0u);
    const int32_t *hl = ctx->h_len.data();
    std::stable_sort(order.begin(), order.end(), [hl](uint32_t a, uint32_t b) { return hl[a] > hl[b]; });
    cudaError_t e = cudaMalloc(&ctx->d_res, total);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_off, n_seq * sizeof(uint64_t));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_len, n_seq * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_order, n_seq * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_res, h_res, total, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_off, h_off.data(), n_seq * sizeof(uint64_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_len, ctx->h_len.data(), n_seq * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_order, order.data(), n_seq * sizeof(uint32_t), cudaMemcpyHostToDevice);
    cudaFreeHost(h_res);
    if (e != cudaSuccess) {
        ctx->err = std::string("b200_db_load: ") + cudaGetErrorString(e);
        db_free(ctx);
        return e == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA;
    }
    ctx->n_seq = n_seq;
    ctx->n_res = n_res;
    ctx->alphabet = alphabet;
    ctx->max_len = max_len;
    return B200_OK;
}

int b200_db_load(b200_ctx *ctx, const uint8_t *residues, const uint64_t *offsets, uint64_t n_seq, int alphabet) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (residues == nullptr || offsets == nullptr || n_seq == 0 || alphabet <= 0 || alphabet > 31)
        return set_err(ctx, B200_ERR_ARG, "b200_db_load: bad arguments");
    if (n_seq >= 0xffffffffull) return set_err(ctx, B200_ERR_RANGE, "b200_db_load: more than 2^32-1 sequences");
    std::vector<int32_t> lens(n_seq);
    for (uint64_t i = 0; i < n_seq; i++) {
        if (offsets[i + 1] < offsets[i]) return set_err(ctx, B200_ERR_ARG, "b200_db_load: offsets not monotone");
        const uint64_t l = offsets[i + 1] - offsets[i];
        if (l > 65535) return set_err(ctx, B200_ERR_RANGE, "b200_db_load: sequence longer than 65535 (maxSeqLen)");
        lens[i] = (int32_t) l;
    }
    return b200_db_load_impl(ctx, residues, offsets, lens.data(), n_seq, alphabet, 256, offsets[n_seq] - offsets[0], false);
}

static int db_load_padded_common(b200_ctx *ctx, const uint8_t *data, const size_t *offsets, const int32_t *lengths, uint64_t n_seq, int alphabet,
                                 bool strip_mask) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (data == nullptr || offsets == nullptr || lengths == nullptr || n_seq == 0 || alphabet <= 0 || alphabet > 31)
        return set_err(ctx, B200_ERR_ARG, "b200_db_load_padded: bad arguments");
    if (n_seq >= 0xffffffffull) return set_err(ctx, B200_ERR_RANGE, "b200_db_load_padded: more than 2^32-1 sequences");
    std::vector<uint64_t> starts(n_seq);
    uint64_t n_res = 0;
    for (uint64_t i = 0; i < n_seq; i++) {
        if (lengths[i] < 0 || lengths[i] > 65535) return set_err(ctx, B200_ERR_RANGE, "b200_db_load_padded: sequence length outside [0,65535]");
        starts[i] = offsets[i];
        n_res += (uint64_t) lengths[i];
    }
    return b200_db_load_impl(ctx, data, starts.data(), lengths, n_seq, alphabet, 32, n_res, strip_mask);
}

int b200_db_load_padded(b200_ctx *ctx, const uint8_t *data, const size_t *offsets, const int32_t *lengths, uint64_t n_seq, int alphabet) {
    return db_load_padded_common(ctx, data, offsets, lengths, n_seq, alphabet, false);
}

int b200_db_load_padded_unmasked(b200_ctx *ctx, const uint8_t *data, const size_t *offsets, const int32_t *lengths, uint64_t n_seq, int alphabet) {
    return db_load_padded_common(ctx, data, offsets, lengths, n_seq, alphabet, true);
}

int b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

uint64_t b200_db_num_seqs(const b200_ctx *ctx) { return ctx ? ctx->n_seq : 0; }
uint64_t b200_db_num_residues(const b200_ctx *ctx) { return ctx ? ctx->n_res : 0; }

// ---- A2 ---------------------------------------------------------------------------------------------
int b200_scan_job_create(b200_ctx *ctx, const b200_query *queries, int nq, int min_score_excl, uint32_t max_hits,
                         b200_job **out) {
    if (ctx == nullptr || out == nullptr) return B200_ERR_ARG;
    *out = nullptr;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->n_seq == 0) return set_err(ctx, B200_ERR_NODB, "no target DB loaded");
    if (queries == nullptr || nq <= 0 || max_hits == 0) return set_err(ctx, B200_ERR_ARG, "b200_ungapped_scan: bad arguments");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const int A = ctx->alphabet;
    // group queries by kernel configuration so that one launch covers one group (grid.y = group size)
    std::vector<std::vector<int>> groups(sizeof(kScanCfgs) / sizeof(kScanCfgs[0]) + 1);
    for (int i = 0; i < nq; i++) {
        if (queries[i].profile == nullptr || queries[i].qlen <= 0) return set_err(ctx, B200_ERR_ARG, "query without profile");
        if (queries[i].bias < 0 || queries[i].bias > 255) return set_err(ctx, B200_ERR_ARG, "profile bias outside [0,255]");
        const int c = scan_cfg_for(queries[i].qlen);
        if (queries[i].qlen > 65535) return set_err(ctx, B200_ERR_RANGE, "b200_ungapped_scan: query longer than 65535 (maxSeqLen)");
        groups[c].push_back(i);
    }
    b200_job *job = new b200_job();
    job->ctx = ctx; job->kind = 1; job->nq = nq; job->thr = min_score_excl; job->k = max_hits;
    // The G = 8 queries go four to a launch unit (quads, see ungapped_scan_kernel): sorted by length, longest first, each quad in
    // the class of its longest query.  The n mod 4 shortest stay in their own classes, as do G = 16/32 and tiled queries.
    // B200_SCAN_NO_QUADS=1 turns quads off (A/B measurements).
    std::vector<std::vector<int>> quad_groups(groups.size());
    if (getenv("B200_SCAN_NO_QUADS") == nullptr && scan_quads_fit(A)) {
        std::vector<int> g8;
        for (size_t c = 0; c < groups.size(); c++)
            if (c < sizeof(kScanCfgs) / sizeof(kScanCfgs[0]) && kScanCfgs[c].G == 8) { g8.insert(g8.end(), groups[c].begin(), groups[c].end()); groups[c].clear(); }
        std::stable_sort(g8.begin(), g8.end(), [queries](int a, int b) { return queries[a].qlen > queries[b].qlen; });
        const size_t n_quad = g8.size() / 4 * 4;
        for (size_t i = 0; i < n_quad; i += 4) {
            std::vector<int> &qg = quad_groups[scan_cfg_for(queries[g8[i]].qlen)];
            qg.insert(qg.end(), g8.begin() + i, g8.begin() + i + 4);
        }
        for (size_t i = n_quad; i < g8.size(); i++) groups[scan_cfg_for(queries[g8[i]].qlen)].push_back(g8[i]);
        for (auto &gr : groups) std::sort(gr.begin(), gr.end());
    }
    for (size_t c = 0; c < groups.size(); c++) {
        if (!quad_groups[c].empty()) job->scan_groups.push_back({(int) c, true, quad_groups[c]});
        if (!groups[c].empty()) job->scan_groups.push_back({(int) c, false, groups[c]});
    }
    std::vector<QueryDesc> h_qd;
    uint64_t raw_bytes = 0;
    for (const auto &sg : job->scan_groups)
        for (int qi : sg.queries) {
            QueryDesc d;
            memset(&d, 0, sizeof(d));
            d.qlen = queries[qi].qlen; d.bias = queries[qi].bias; d.raw_off = raw_bytes;
            raw_bytes += round_up((uint64_t) A * d.qlen, 16);
            h_qd.push_back(d);
            job->grouped_order.push_back(qi);
            job->cells += (uint64_t) d.qlen * ctx->n_res;
        }
    std::vector<int8_t> h_raw(raw_bytes, 0);
    for (int pos = 0; pos < nq; pos++)
        memcpy(h_raw.data() + h_qd[pos].raw_off, queries[job->grouped_order[pos]].profile, (size_t) A * h_qd[pos].qlen);
    cudaError_t e = job->raw.reserve(raw_bytes);
    if (e == cudaSuccess) e = job->qdesc.reserve(sizeof(QueryDesc) * nq);
    if (e == cudaSuccess) e = job->dense.reserve((size_t) nq * ctx->n_seq);
    if (e == cudaSuccess) e = job->hits.reserve((size_t) nq * max_hits * sizeof(b200_hit));
    if (e == cudaSuccess) e = job->nhits.reserve((size_t) nq * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->raw.p, h_raw.data(), raw_bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->qdesc.p, h_qd.data(), sizeof(QueryDesc) * nq, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        ctx->err = std::string("scan job staging: ") + cudaGetErrorString(e);
        job->free_all(); delete job;
        return e == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA;
    }
    *out = job;
    return B200_OK;
}

// The capacity classes present in a batch are independent launches over disjoint output rows.  They go out on the ctx stream and up
// to three side streams, largest class first: every launch is a persistent grid that fills the GPU, so a later class only gets SM
// slots as the CTAs of an earlier one run out of work units -- its start overlaps the earlier launch's tail instead of waiting for
// the last CTA (previously: one idle tail per class, five per 16-query step of config[1]).  The tiled long-query variant shares
// one boundary scratch and stays on the ctx stream.
static int scan_job_run_locked(b200_job *job) {
    b200_ctx *ctx = job->ctx;
    struct L { int cfg; bool quad; int pos, n; };   // n queries, or n quads
    std::vector<L> launches;
    int pos = 0;
    for (const auto &sg : job->scan_groups) {
        const int per = sg.quad ? 4 : 1;
        const int n = (int) sg.queries.size() / per;
        for (int s = 0; s < n; s += 32768) launches.push_back({sg.cfg, sg.quad, pos + per * s, std::min(32768, n - s)});
        pos += (int) sg.queries.size();
    }
    const int n_cfg = (int) (sizeof(kScanCfgs) / sizeof(kScanCfgs[0]));
    auto weight = [n_cfg](const L &l) { return (double) l.n * (l.quad ? 4 : 1) * (l.cfg < n_cfg ? 2.0 * kScanCfgs[l.cfg].G * kScanCfgs[l.cfg].K : 1e9); };
    std::stable_sort(launches.begin(), launches.end(), [&weight](const L &a, const L &b) { return weight(a) > weight(b); });
    const bool fan_out = launches.size() > 1 && getenv("B200_SCAN_SERIAL") == nullptr;
    if (fan_out) CU_TRY(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
    bool used[3] = {false, false, false};
    int next_side = 0;
    for (size_t i = 0; i < launches.size(); i++) {
        const L &l = launches[i];
        cudaStream_t st = ctx->stream;
        if (fan_out && i > 0 && l.cfg < n_cfg && i < (size_t) kScanCounters) {
            const int k = next_side++ % 3;
            st = ctx->side[k];
            if (!used[k]) { CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_fork, 0)); used[k] = true; }
        }
        CU_TRY(ctx, launch_scan(ctx, l.cfg, l.quad, job->raw.as<int8_t>(), job->qdesc.as<QueryDesc>() + l.pos, l.n,
                                job->dense.as<uint8_t>() + (size_t) l.pos * ctx->n_seq, st, (int) (i % kScanCounters)));
    }
    for (int k = 0; k < 3; k++)
        if (used[k]) {
            CU_TRY(ctx, cudaEventRecord(ctx->ev_join[k], ctx->side[k]));
            CU_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join[k], 0));
        }
    if ((uint64_t) job->nq * TOPK_PARTS <= 4096 && ctx->n_seq >= 65536 && getenv("B200_TOPK_SINGLE") == nullptr) {
        // few queries, many targets: the selection spread over TOPK_PARTS CTAs per query (identical output, ~30x shorter critical path)
        CU_TRY(ctx, job->part_hist.reserve(sizeof(uint32_t) * 256 * TOPK_PARTS * (size_t) job->nq));
        const dim3 grid(TOPK_PARTS, (unsigned) job->nq);
        topk_hist_kernel<<<grid, 256, 0, ctx->stream>>>(job->dense.as<uint8_t>(), (uint32_t) ctx->n_seq, job->part_hist.as<uint32_t>());
        topk_compact_kernel<<<grid, 256, 0, ctx->stream>>>(job->dense.as<uint8_t>(), (uint32_t) ctx->n_seq, job->thr, job->k,
                                                            job->part_hist.as<uint32_t>(), job->hits.as<b200_hit>(), job->nhits.as<uint32_t>());
        ctx->launches += 2;
    } else {
        topk_select_kernel<<<job->nq, 1024, 0, ctx->stream>>>(job->dense.as<uint8_t>(), (uint32_t) ctx->n_seq, job->thr, job->k,
                                                              job->hits.as<b200_hit>(), job->nhits.as<uint32_t>());
        ctx->launches++;
    }
    CU_TRY(ctx, cudaGetLastError());
    if (job->done == nullptr) CU_TRY(ctx, cudaEventCreateWithFlags(&job->done, cudaEventDisableTiming));
    CU_TRY(ctx, cudaEventRecord(job->done, ctx->stream));
    job->ran = true;
    return B200_OK;
}

int b200_scan_job_fetch(b200_job *job, b200_hit *hits, uint32_t *n_hits, uint8_t *dense) {
    if (job == nullptr || job->kind != 1) return B200_ERR_ARG;
    b200_ctx *ctx = job->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const int nq = job->nq;
    const uint32_t k = job->k;
    std::vector<b200_hit> h_hits((size_t) nq * k);
    std::vector<uint32_t> h_n(nq);
    // The download waits for THIS job's last kernel only (its event), on the copy stream: jobs enqueued after it keep the GPU busy
    // while the host collects -- what lets a caller overlap the hit-list gather of step s with the scan of step s+1.
    cudaStream_t cs = job->ran ? ctx->copy_stream : ctx->stream;
    if (job->ran) CU_TRY(ctx, cudaStreamWaitEvent(cs, job->done, 0));
    CU_TRY(ctx, cudaMemcpyAsync(h_n.data(), job->nhits.p, sizeof(uint32_t) * nq, cudaMemcpyDeviceToHost, cs));
    CU_TRY(ctx, cudaMemcpyAsync(h_hits.data(), job->hits.p, sizeof(b200_hit) * nq * k, cudaMemcpyDeviceToHost, cs));
    if (dense != nullptr) {
        for (int pos = 0; pos < nq; pos++)
            CU_TRY(ctx, cudaMemcpyAsync(dense + (size_t) job->grouped_order[pos] * ctx->n_seq,
                                        job->dense.as<uint8_t>() + (size_t) pos * ctx->n_seq, ctx->n_seq,
                                        cudaMemcpyDeviceToHost, cs));
    }
    CU_TRY(ctx, cudaStreamSynchronize(cs));
    for (int pos = 0; pos < nq; pos++) {
        const int qi = job->grouped_order[pos];
        const uint32_t n = std::min(h_n[pos], k);
        b200_hit *src = h_hits.data() + (size_t) pos * k;
        std::sort(src, src + n, [](const b200_hit &a, const b200_hit &b) {
            return a.score != b.score ? a.score > b.score : a.id < b.id;
        });
        if (hits) memcpy(hits + (size_t) qi * k, src, sizeof(b200_hit) * n);
        if (n_hits) n_hits[qi] = n;
    }
    return B200_OK;
}

int b200_ungapped_scan(b200_ctx *ctx, const b200_query *queries, int nq, int min_score_excl, uint32_t max_hits,
                       b200_hit *hits, uint32_t *n_hits, uint8_t *dense) {
    b200_job *job = nullptr;
    int rc = b200_scan_job_create(ctx, queries, nq, min_score_excl, max_hits, &job);
    if (rc != B200_OK) return rc;
    rc = b200_job_run(job);
    if (rc == B200_OK) rc = b200_scan_job_fetch(job, hits, n_hits, dense);
    b200_job_destroy(job);
    return rc;
}

// ---- A1 ---------------------------------------------------------------------------------------------
// Many queries' hit lists in one call: one upload of all profiles and hits, one launch, one download, one synchronisation --
// what QueryMatcher's OpenMP threads need so that they do not serialise on a per-query round trip (QueryMatcher.cpp:73,131).
// queries[i] owns hits [hit_offsets[i], hit_offsets[i+1]).
int b200_diag_score_batch(b200_ctx *ctx, const b200_query *queries, int nq, const uint64_t *hit_offsets, const uint32_t *ids,
                          const uint16_t *diagonals, uint8_t *counts, int32_t *raw) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->n_seq == 0) return set_err(ctx, B200_ERR_NODB, "no target DB loaded");
    if (ctx->alphabet > 31) return set_err(ctx, B200_ERR_ARG, "b200_diag_score: the resident DB is an ASCII DB (b200_db_load_ascii)");
    if (queries == nullptr || nq <= 0 || hit_offsets == nullptr) return set_err(ctx, B200_ERR_ARG, "b200_diag_score: bad arguments");
    const uint64_t n = hit_offsets[nq] - hit_offsets[0];
    if (n == 0) return B200_OK;
    if (ids == nullptr || diagonals == nullptr || counts == nullptr) return set_err(ctx, B200_ERR_ARG, "b200_diag_score: bad arguments");
    if (ctx->max_len >= 32768)
        return set_err(ctx, B200_ERR_RANGE, "b200_diag_score: sequences >= 32768 take the reference's computeLongScore path (T6)");
    std::vector<DiagQuery> h_dq(nq);
    uint64_t pbytes = 0;
    for (int i = 0; i < nq; i++) {
        if (queries[i].profile == nullptr || queries[i].qlen <= 0 || hit_offsets[i + 1] < hit_offsets[i])
            return set_err(ctx, B200_ERR_ARG, "b200_diag_score: query without profile, or hit offsets not monotone");
        if (queries[i].qlen >= 32768)
            return set_err(ctx, B200_ERR_RANGE, "b200_diag_score: sequences >= 32768 take the reference's computeLongScore path (T6)");
        h_dq[i].prof_off = pbytes; h_dq[i].hit_begin = hit_offsets[i] - hit_offsets[0]; h_dq[i].qlen = queries[i].qlen; h_dq[i].pad_ = 0;
        pbytes += round_up((uint64_t) ctx->alphabet * queries[i].qlen, 16);
    }
    const uint32_t *idp = ids + hit_offsets[0];
    const uint16_t *dgp = diagonals + hit_offsets[0];
    uint8_t *cnp = counts + hit_offsets[0];
    int32_t *rwp = raw ? raw + hit_offsets[0] : nullptr;
    for (uint64_t i = 0; i < n; i++)
        if (idp[i] >= ctx->n_seq) return set_err(ctx, B200_ERR_ARG, "b200_diag_score: target id out of range");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<int8_t> h_prof(pbytes);
    for (int i = 0; i < nq; i++) memcpy(h_prof.data() + h_dq[i].prof_off, queries[i].profile, (size_t) ctx->alphabet * queries[i].qlen);
    CU_TRY(ctx, ctx->raw.reserve(pbytes));
    CU_TRY(ctx, ctx->qdesc.reserve(sizeof(DiagQuery) * nq));
    CU_TRY(ctx, ctx->ids.reserve(n * sizeof(uint32_t)));
    CU_TRY(ctx, ctx->diags.reserve(n * sizeof(uint16_t)));
    CU_TRY(ctx, ctx->counts.reserve(n));
    if (raw) CU_TRY(ctx, ctx->rawout.reserve(n * sizeof(int32_t)));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->raw.p, h_prof.data(), pbytes, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->qdesc.p, h_dq.data(), sizeof(DiagQuery) * nq, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->ids.p, idp, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->diags.p, dgp, n * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->counts.p, cnp, n, cudaMemcpyHostToDevice, ctx->stream));
    const unsigned ctas = (unsigned) std::min<uint64_t>((n + 7) / 8, (uint64_t) ctx->sm_count * 8);
    CU_TRY(ctx, cudaEventRecord(ctx->ev[12], ctx->stream));
    diag_score_kernel<<<ctas, 256, 0, ctx->stream>>>(ctx->raw.as<int8_t>(), ctx->qdesc.as<DiagQuery>(), nq, ctx->d_res, ctx->d_off, ctx->d_len,
                                                     ctx->ids.as<uint32_t>(), ctx->diags.as<uint16_t>(), n,
                                                     ctx->counts.as<uint8_t>(), raw ? ctx->rawout.as<int32_t>() : nullptr);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaEventRecord(ctx->ev[13], ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(cnp, ctx->counts.p, n, cudaMemcpyDeviceToHost, ctx->stream));
    if (raw) CU_TRY(ctx, cudaMemcpyAsync(rwp, ctx->rawout.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_kernel_ms, ctx->ev[12], ctx->ev[13]);
    return B200_OK;
}

int b200_diag_score(b200_ctx *ctx, const b200_query *q, const uint32_t *ids, const uint16_t *diagonals, uint64_t n,
                    uint8_t *counts, int32_t *raw) {
    if (ctx == nullptr) return B200_ERR_ARG;
    if (q == nullptr) return set_err(ctx, B200_ERR_ARG, "b200_diag_score: bad arguments");
    const uint64_t offs[2] = {0, n};
    return b200_diag_score_batch(ctx, q, 1, offs, ids, diagonals, counts, raw);
}

// ---- A3-A5 ------------------------------------------------------------------------------------------
namespace {

constexpr uint32_t kPairsPerItem = 8;

struct SwPlan {
    std::vector<uint32_t> perm;  // sorted position -> caller index
    std::vector<WorkItem> items;
};

// sort pairs by (query, target length desc) and cut each query's run into CTA-sized items, longest work first
void plan_pairs(const b200_ctx *ctx, const b200_query *queries, const b200_pair *pairs, uint64_t n, const uint8_t *mask, SwPlan &plan,
                uint32_t pairs_per_item = kPairsPerItem) {
    std::vector<int32_t> qlens;
    { uint32_t mq = 0; for (uint64_t i = 0; i < n; i++) mq = std::max(mq, pairs[i].query); qlens.resize((size_t) mq + 1); for (uint32_t i = 0; i <= mq; i++) qlens[i] = queries[i].qlen; }
    // order: query ascending, target length descending, caller index ascending -- one 64-bit key per pair
    const int32_t *hl = ctx->h_len.data();
    struct Key { uint64_t k; uint32_t i; };
    std::vector<Key> keys;
    keys.reserve(n);
    for (uint64_t i = 0; i < n; i++)
        if (mask == nullptr || mask[i]) {
            Key e; e.k = ((uint64_t) pairs[i].query << 32) | (uint64_t) (0xffffu - (uint32_t) hl[pairs[i].target]); e.i = (uint32_t) i;
            keys.push_back(e);
        }
    // stable LSD radix sort on the 48 significant key bits (16 length bits, then the query index), 16 bits per pass;
    // stability keeps ties in caller order.  ~10x faster than a comparison sort at 10^5..10^6 pairs.
    {
        uint32_t maxq = 0;
        for (const Key &e : keys) maxq = std::max(maxq, (uint32_t) (e.k >> 32));
        std::vector<Key> tmp(keys.size());
        std::vector<uint32_t> hist(65536 + 1);
        const int shifts[3] = {0, 32, 48};
        const int npass = maxq > 0xffffu ? 3 : (maxq > 0 ? 2 : 1);
        for (int ps = 0; ps < npass; ps++) {
            const int sh = shifts[ps];
            std::fill(hist.begin(), hist.end(), 0u);
            for (const Key &e : keys) hist[((e.k >> sh) & 0xffffu) + 1]++;
            for (size_t b2 = 1; b2 < hist.size(); b2++) hist[b2] += hist[b2 - 1];
            for (const Key &e : keys) tmp[hist[(e.k >> sh) & 0xffffu]++] = e;
            keys.swap(tmp);
        }
    }
    plan.perm.resize(keys.size());
    for (size_t k = 0; k < keys.size(); k++) plan.perm[k] = keys[k].i;
    plan.items.clear();
    const uint32_t m = (uint32_t) plan.perm.size();
    uint32_t s = 0;
    while (s < m) {
        uint32_t e = s;
        const uint32_t qy = pairs[plan.perm[s]].query;
        while (e < m && pairs[plan.perm[e]].query == qy) e++;
        for (uint32_t p = s; p < e; p += pairs_per_item) {
            WorkItem it; it.query = qy; it.p0 = p; it.p1 = std::min(e, p + pairs_per_item); it.pad_ = (uint32_t) sw16_k_for(qlens[qy]);
            plan.items.push_back(it);
        }
        s = e;
    }
    // heaviest items first (longest-processing-time order for the dynamic item counter)
    std::vector<uint64_t> cost(plan.items.size());
    for (size_t k = 0; k < plan.items.size(); k++) {
        uint64_t c = 0;
        for (uint32_t p = plan.items[k].p0; p < plan.items[k].p1; p++) c += (uint64_t) hl[pairs[plan.perm[p]].target];
        cost[k] = c * (uint64_t) qlens[plan.items[k].query];
    }
    std::vector<uint32_t> io(plan.items.size());
    std::iota(io.begin(), io.end(), 0u);
    std::stable_sort(io.begin(), io.end(), [&cost](uint32_t a, uint32_t b) { return cost[a] > cost[b]; });
    std::vector<WorkItem> sorted(plan.items.size());
    for (size_t k = 0; k < io.size(); k++) sorted[k] = plan.items[io[k]];
    plan.items.swap(sorted);
}

// resident CTAs of the gapped kernel for a given dynamic shared-memory size (also sizes the boundary scratch)
template <int DIR>
unsigned sw_grid(b200_ctx *ctx, size_t smem, unsigned n_items) {
    int per_sm = 0;
    if (smem > 0) {
        cudaFuncSetAttribute(sw32_kernel<DIR, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sw32_kernel<DIR, true>, SW_WARPS * 32, smem) != cudaSuccess) per_sm = 1;
    } else if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sw32_kernel<DIR, false>, SW_WARPS * 32, 0) != cudaSuccess) per_sm = 1;
    per_sm = std::max(1, per_sm);
    return (unsigned) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) ctx->sm_count * per_sm, n_items));
}
unsigned sw_max_grid(const b200_ctx *ctx) { return (unsigned) ctx->sm_count * 16u; }

template <int DIR>
int launch_sw(b200_ctx *ctx, const QueryDesc *d_qd, const int8_t *d_pad, int max_Lp, const WorkItem *d_items, uint32_t n_items,
              const PairDesc *d_pairs, int go, int ge, int2 *d_bnd, int bnd_stride, int4 *d_out) {
    const int A = ctx->alphabet;
    size_t smem = (size_t) (A + 1) * max_Lp;
    int smem_profile = 1;
    if (smem > (size_t) ctx->max_smem_optin - 1024) { smem = 0; smem_profile = 0; }
    CU_TRY(ctx, ctx->counter.reserve(sizeof(unsigned)));
    CU_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, sizeof(unsigned), ctx->stream));
    const unsigned grid = sw_grid<DIR>(ctx, smem, n_items);
    if (smem_profile)
        sw32_kernel<DIR, true><<<grid, SW_WARPS * 32, smem, ctx->stream>>>(d_pad, d_qd, d_items, d_pairs, ctx->d_res, ctx->d_off,
                                                                          ctx->d_len, A, go, ge, d_bnd, bnd_stride, smem_profile,
                                                                          n_items, ctx->counter.as<unsigned>(), d_out);
    else
        sw32_kernel<DIR, false><<<grid, SW_WARPS * 32, 0, ctx->stream>>>(d_pad, d_qd, d_items, d_pairs, ctx->d_res, ctx->d_off,
                                                                        ctx->d_len, A, go, ge, d_bnd, bnd_stride, smem_profile,
                                                                        n_items, ctx->counter.as<unsigned>(), d_out);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    return B200_OK;
}

int check_pairs(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go, int ge) {
    if (ctx->n_seq == 0) return set_err(ctx, B200_ERR_NODB, "no target DB loaded");
    if (queries == nullptr || nq <= 0 || (pairs == nullptr && n > 0)) return set_err(ctx, B200_ERR_ARG, "sw: bad arguments");
    if (go < 0 || go > 255 || ge < 0 || ge > 255) return set_err(ctx, B200_ERR_ARG, "sw: gap penalties are uint8 in the reference");
    if (n >= 0xffffffffull) return set_err(ctx, B200_ERR_RANGE, "sw: more than 2^32-1 pairs in one call");
    for (uint64_t i = 0; i < n; i++)
        if (pairs[i].query >= (uint32_t) nq || pairs[i].target >= ctx->n_seq) return set_err(ctx, B200_ERR_ARG, "sw: pair index out of range");
    return B200_OK;
}

// shared body: one direction over a planned set of pairs; results (score, col, row) come back in caller order
template <int DIR>
int run_sw_pass(b200_ctx *ctx, const std::vector<QueryDesc> &h_qd, const b200_pair *pairs, const SwPlan &plan,
                const b200_sw_end *ends, int go, int ge, std::vector<int4> &res_sorted) {
    const uint32_t m = (uint32_t) plan.perm.size();
    res_sorted.assign(m, make_int4(0, -1, -1, 0));
    if (m == 0) return B200_OK;
    std::vector<PairDesc> h_pd(m);
    int max_cols = 1;
    for (uint32_t s = 0; s < m; s++) {
        const uint32_t i = plan.perm[s];
        PairDesc &d = h_pd[s];
        d.target = pairs[i].target;
        d.qend = d.dbend = d.score = 0;
        if (DIR < 0) { d.qend = ends[i].qend; d.dbend = ends[i].dbend; d.score = ends[i].score; max_cols = std::max(max_cols, d.dbend + 1); }
        else max_cols = std::max(max_cols, ctx->h_len[d.target]);
    }
    int max_Lp = 0;
    bool multi = false;
    for (const WorkItem &it : plan.items) {
        max_Lp = std::max(max_Lp, h_qd[it.query].Lp);
        if (h_qd[it.query].qlen > SW_TILE) multi = true;
    }
    const uint32_t n_items = (uint32_t) plan.items.size();
    const int bnd_stride = multi ? (int) round_up((uint64_t) max_cols, 32) + 32 : 32;
    CU_TRY(ctx, ctx->pairs.reserve(sizeof(PairDesc) * m));
    CU_TRY(ctx, ctx->items.reserve(sizeof(WorkItem) * n_items));
    CU_TRY(ctx, ctx->out4.reserve(sizeof(int4) * m));
    CU_TRY(ctx, ctx->bnd.reserve(sizeof(int2) * 2 * (size_t) bnd_stride * std::min<uint64_t>(n_items, sw_max_grid(ctx)) * SW_WARPS));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->pairs.p, h_pd.data(), sizeof(PairDesc) * m, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->items.p, plan.items.data(), sizeof(WorkItem) * n_items, cudaMemcpyHostToDevice, ctx->stream));
    int rc = launch_sw<DIR>(ctx, ctx->qdesc.as<QueryDesc>(), ctx->pad.as<int8_t>(), max_Lp, ctx->items.as<WorkItem>(), n_items,
                            ctx->pairs.as<PairDesc>(), go, ge, ctx->bnd.as<int2>(), bnd_stride, ctx->out4.as<int4>());
    if (rc != B200_OK) return rc;
    CU_TRY(ctx, cudaMemcpyAsync(res_sorted.data(), ctx->out4.p, sizeof(int4) * m, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return B200_OK;
}

// byte/word reporting rules of alignScoreEndPos (StripedSmithWaterman.cpp:892-941, T4/T5)
inline void report_end(const int4 &r, int bias, b200_sw_end &o) {
    const int score = r.x;
    if (score + bias >= 255) {
        o.score = std::min(score, 32767); o.qend = r.z; o.dbend = r.y; o.word = 1;
    } else if (score == 0) {
        o.score = 0; o.qend = 0; o.dbend = -1; o.word = 0;
    } else {
        o.score = score; o.qend = r.z; o.dbend = r.y; o.word = 0;
    }
}

}  // namespace

namespace {
int run_sw16_pass(b200_ctx *ctx, const std::vector<QueryDesc> &h_qd, const b200_query *queries, const b200_pair *pairs, uint64_t n,
                  const uint8_t *mask, const int32_t *scores, int go, int ge, std::vector<int32_t> &res, const b200_sw_end *rev_ends = nullptr);
int run_sw16_chain(b200_ctx *ctx, const std::vector<QueryDesc> &h_qd, const b200_query *queries, const b200_pair *pairs, uint64_t n,
                   const uint8_t *mask, const uint8_t *gate, bool want_start, int go, int ge, std::vector<int32_t> &score,
                   std::vector<int32_t> &endpos, std::vector<int32_t> *startpos);
}

// alignScoreEndPos for a batch: packed score kernel on every pair that is safe in int16, packed FIND pass for the end
// positions of those with a positive score, int32 kernel (score + end in one pass) for the rest.
static int sw_score_endpos_locked(b200_ctx *ctx, const std::vector<QueryDesc> &h_qd, const b200_query *queries, const b200_pair *pairs,
                                  uint64_t n, int go, int ge, b200_sw_end *out, const uint8_t *gate = nullptr,
                                  std::vector<int32_t> *startpos = nullptr, std::vector<uint8_t> *packed_out = nullptr) {
    const int A = ctx->alphabet;
    const int nq = (int) h_qd.size();
    std::vector<int> smax(nq, 1);
    std::vector<int64_t> qsum(nq, 0);
    for (size_t q_ = 0; q_ < (size_t) (nq); q_++) profile_bounds(queries[q_].profile, A, queries[q_].qlen, smax[q_], qsum[q_]);
    std::vector<uint8_t> packed(n), rest(n);
    bool any_rest = false, any_packed = false;
    for (uint64_t i = 0; i < n; i++) {
        const int qi = (int) pairs[i].query;
        const int tl = ctx->h_len[pairs[i].target];
        const bool ok = go >= ge && int16_safe(smax[qi], qsum[qi], queries[qi].qlen, tl);
        packed[i] = ok ? 1 : 0; rest[i] = ok ? 0 : 1;
        any_rest |= !ok; any_packed |= ok;
    }
    std::vector<int4> res4(n, make_int4(0, -1, -1, 0));
    if (any_packed) {
        // score -> end positions (-> start positions) as chained launches over one plan: nothing returns to the host in between
        std::vector<int32_t> score(n, 0), pos(2 * n, -1);
        if (startpos != nullptr) startpos->assign(2 * n, -1);
        int rc = run_sw16_chain(ctx, h_qd, queries, pairs, n, any_rest ? packed.data() : nullptr, gate, startpos != nullptr, go, ge,
                                score, pos, startpos);
        if (rc != B200_OK) return rc;
        for (uint64_t i = 0; i < n; i++)
            if (packed[i] && score[i] > 0) res4[i] = make_int4(score[i], pos[2 * i], pos[2 * i + 1], 0);
    }
    if (any_rest) {
        SwPlan plan;
        plan_pairs(ctx, queries, pairs, n, rest.data(), plan);
        std::vector<int4> res;
        int rc = run_sw_pass<1>(ctx, h_qd, pairs, plan, nullptr, go, ge, res);
        if (rc != B200_OK) return rc;
        for (uint32_t s = 0; s < plan.perm.size(); s++) res4[plan.perm[s]] = res[s];
    }
    for (uint64_t i = 0; i < n; i++) report_end(res4[i], queries[pairs[i].query].bias, out[i]);
    if (packed_out != nullptr) packed_out->swap(packed);
    return B200_OK;
}

int b200_sw_score_endpos(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go,
                         int ge, b200_sw_end *out) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (out == nullptr) return set_err(ctx, B200_ERR_ARG, "sw: out is NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);
    if (rc != B200_OK) return rc;
    return sw_score_endpos_locked(ctx, h_qd, queries, pairs, n, go, ge, out);
}

static int sw_startpos_locked(b200_ctx *ctx, const b200_query *queries, const std::vector<QueryDesc> &h_qd, const b200_pair *pairs, uint64_t n, int go,
                              int ge, const b200_sw_end *ends, const uint8_t *gate, b200_sw_aln *out, const uint8_t *skip = nullptr) {
    std::vector<uint8_t> mask(n);
    for (uint64_t i = 0; i < n; i++) {
        out[i].score = ends[i].score; out[i].qend = ends[i].qend; out[i].dbend = ends[i].dbend; out[i].word = ends[i].word;
        out[i].qstart = -1; out[i].dbstart = -1;
        mask[i] = (ends[i].dbend != -1 && (gate == nullptr || gate[i]) && (skip == nullptr || !skip[i])) ? 1 : 0;
        if (mask[i]) {
            const int ql = h_qd[pairs[i].query].qlen, tl = ctx->h_len[pairs[i].target];
            if (ends[i].qend < 0 || ends[i].qend >= ql || ends[i].dbend < 0 || ends[i].dbend >= tl || ends[i].score <= 0)
                return set_err(ctx, B200_ERR_ARG, "sw_startpos: end positions outside the sequences");
        }
    }
    // packed reverse pass where the forward pass was packed too (same int16 safety argument), int32 kernel otherwise
    const int A = ctx->alphabet;
    std::vector<int> smax(h_qd.size(), 1);
    std::vector<int64_t> qsum(h_qd.size(), 0);
    for (size_t q_ = 0; q_ < (size_t) (h_qd.size()); q_++) profile_bounds(queries[q_].profile, A, queries[q_].qlen, smax[q_], qsum[q_]);
    std::vector<uint8_t> packed(n, 0), rest(n, 0);
    bool any_packed = false, any_rest = false;
    for (uint64_t i = 0; i < n; i++) {
        if (!mask[i]) continue;
        const int qi = (int) pairs[i].query;
        const bool ok = go >= ge && int16_safe(smax[qi], qsum[qi], queries[qi].qlen, ctx->h_len[pairs[i].target]);
        packed[i] = ok; rest[i] = !ok;
        any_packed |= ok; any_rest |= !ok;
    }
    if (any_packed) {
        std::vector<int32_t> pos(2 * n, -1);
        int rc = run_sw16_pass(ctx, h_qd, queries, pairs, n, packed.data(), nullptr, go, ge, pos, ends);
        if (rc != B200_OK) return rc;
        for (uint64_t i = 0; i < n; i++) {
            if (!packed[i]) continue;
            if (pos[2 * i] < 0 || pos[2 * i] > 0xfffe) return set_err(ctx, B200_ERR_ARG, "sw_startpos: reverse pass did not reproduce the forward score");
            out[i].dbstart = ends[i].dbend - pos[2 * i];
            out[i].qstart = ends[i].qend - pos[2 * i + 1];
        }
    }
    if (any_rest) {
        SwPlan plan;
        plan_pairs(ctx, queries, pairs, n, rest.data(), plan);
        std::vector<int4> res;
        int rc = run_sw_pass<-1>(ctx, h_qd, pairs, plan, ends, go, ge, res);
        if (rc != B200_OK) return rc;
        for (uint32_t s2 = 0; s2 < plan.perm.size(); s2++) {
            const uint32_t i = plan.perm[s2];
            if (res[s2].x != ends[i].score) return set_err(ctx, B200_ERR_ARG, "sw_startpos: reverse pass did not reproduce the forward score");
            out[i].dbstart = ends[i].dbend - res[s2].y;
            out[i].qstart = ends[i].qend - res[s2].z;
        }
    }
    return B200_OK;
}

int b200_sw_startpos(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go, int ge,
                     const b200_sw_end *ends, b200_sw_aln *out) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (ends == nullptr || out == nullptr) return set_err(ctx, B200_ERR_ARG, "sw_startpos: NULL argument");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);
    if (rc != B200_OK) return rc;
    return sw_startpos_locked(ctx, queries, h_qd, pairs, n, go, ge, ends, nullptr, out);
}

int b200_sw_align(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go, int ge,
                  const uint8_t *gate, b200_sw_aln *out) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (out == nullptr) return set_err(ctx, B200_ERR_ARG, "sw: out is NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);
    if (rc != B200_OK) return rc;
    std::vector<b200_sw_end> ends(n);
    std::vector<int32_t> startpos;
    std::vector<uint8_t> packed;
    rc = sw_score_endpos_locked(ctx, h_qd, queries, pairs, n, go, ge, ends.data(), gate, &startpos, &packed);
    if (rc != B200_OK) return rc;
    // the packed pairs already carry their start positions; the int32 reverse kernel covers the rest
    rc = sw_startpos_locked(ctx, queries, h_qd, pairs, n, go, ge, ends.data(), gate, out, packed.data());
    if (rc != B200_OK) return rc;
    if (!startpos.empty())
        for (uint64_t i = 0; i < n; i++) {
            if (!packed[i] || ends[i].dbend == -1 || (gate != nullptr && !gate[i])) continue;
            if (startpos[2 * i] < 0 || startpos[2 * i] > 0xfffe)
                return set_err(ctx, B200_ERR_CUDA, "sw_align: reverse pass did not reproduce the forward score");
            out[i].dbstart = ends[i].dbend - startpos[2 * i];
            out[i].qstart = ends[i].qend - startpos[2 * i + 1];
        }
    return B200_OK;
}

// ---- resident SW job (forward score + end positions) -----------------------------------------------------
int b200_sw_job_create(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go, int ge,
                       b200_job **out) {
    if (ctx == nullptr || out == nullptr) return B200_ERR_ARG;
    *out = nullptr;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return set_err(ctx, B200_ERR_ARG, "sw job: no pairs");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);  // fills ctx->raw/qdesc/pad; the job takes copies below
    if (rc != B200_OK) return rc;
    b200_job *job = new b200_job();
    job->ctx = ctx; job->kind = 2; job->go = go; job->ge = ge; job->n_pairs = n; job->nq = nq;
    SwPlan plan;
    plan_pairs(ctx, queries, pairs, n, nullptr, plan);
    job->perm = plan.perm;
    job->h_pairs.assign(pairs, pairs + n);
    job->h_qlen.resize(nq); job->h_bias.resize(nq);
    for (int i = 0; i < nq; i++) { job->h_qlen[i] = queries[i].qlen; job->h_bias[i] = queries[i].bias; }
    std::vector<PairDesc> h_pd(n);
    int max_cols = 1, max_Lp = 0;
    bool multi = false;
    for (uint32_t s = 0; s < n; s++) {
        const uint32_t i = plan.perm[s];
        h_pd[s].target = pairs[i].target; h_pd[s].qend = h_pd[s].dbend = h_pd[s].score = 0;
        max_cols = std::max(max_cols, ctx->h_len[pairs[i].target]);
        job->cells += (uint64_t) queries[pairs[i].query].qlen * (uint64_t) ctx->h_len[pairs[i].target];
    }
    for (const WorkItem &it : plan.items) {
        max_Lp = std::max(max_Lp, h_qd[it.query].Lp);
        if (h_qd[it.query].qlen > SW_TILE) multi = true;
    }
    job->n_items = (uint32_t) plan.items.size();
    job->bnd_stride = multi ? (int) round_up((uint64_t) max_cols, 32) + 32 : 32;
    job->smem_bytes = max_Lp;
    const size_t pad_bytes = h_qd.back().p16_off + (size_t) (ctx->alphabet + 1) * h_qd.back().Lp;
    cudaError_t e = job->pad.reserve(pad_bytes);
    if (e == cudaSuccess) e = job->qdesc.reserve(sizeof(QueryDesc) * nq);
    if (e == cudaSuccess) e = job->pairs.reserve(sizeof(PairDesc) * n);
    if (e == cudaSuccess) e = job->items.reserve(sizeof(WorkItem) * job->n_items);
    if (e == cudaSuccess) e = job->out4.reserve(sizeof(int4) * n);
    if (e == cudaSuccess) e = job->bnd.reserve(sizeof(int2) * 2 * (size_t) job->bnd_stride * std::min<uint64_t>(job->n_items, sw_max_grid(ctx)) * SW_WARPS);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->pad.p, ctx->pad.p, pad_bytes, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->qdesc.p, h_qd.data(), sizeof(QueryDesc) * nq, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->pairs.p, h_pd.data(), sizeof(PairDesc) * n, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->items.p, plan.items.data(), sizeof(WorkItem) * job->n_items, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        ctx->err = std::string("sw job staging: ") + cudaGetErrorString(e);
        job->free_all(); delete job;
        return e == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA;
    }
    *out = job;
    return B200_OK;
}


// ---- score-only batch (packed int16x2 fast path + int32 fallback) ---------------------------------------------
namespace {

template <int WARPS, int MODE>
int launch_sw16_w(b200_ctx *ctx, const QueryDesc *d_qd, const int8_t *d_pad, size_t smem, int smem_profile, const WorkItem *d_items,
                  uint32_t n_items, const PairDesc *d_pairs, int go, int ge, uint2 *d_bnd, int bnd_stride, int32_t *d_out,
                  const int32_t *dv_score = nullptr, const int32_t *dv_pos = nullptr) {
    int per_sm = 0;
    if (smem_profile) {
        CU_TRY(ctx, cudaFuncSetAttribute(sw16_kernel<true, WARPS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sw16_kernel<true, WARPS, MODE>, WARPS * 32, smem) != cudaSuccess) per_sm = 1;
    } else if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sw16_kernel<false, WARPS, MODE>, WARPS * 32, 0) != cudaSuccess) per_sm = 1;
    per_sm = std::max(1, per_sm);
    const unsigned grid = (unsigned) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) ctx->sm_count * per_sm, n_items));
    if (smem_profile)
        sw16_kernel<true, WARPS, MODE><<<grid, WARPS * 32, smem, ctx->stream>>>(d_pad, d_qd, d_items, d_pairs, ctx->d_res, ctx->d_off,
                                                                         ctx->d_len, ctx->alphabet, go, ge, d_bnd, bnd_stride, n_items,
                                                                         ctx->counter.as<unsigned>(), d_out, dv_score, dv_pos);
    else
        sw16_kernel<false, WARPS, MODE><<<grid, WARPS * 32, 0, ctx->stream>>>(d_pad, d_qd, d_items, d_pairs, ctx->d_res, ctx->d_off,
                                                                       ctx->d_len, ctx->alphabet, go, ge, d_bnd, bnd_stride, n_items,
                                                                       ctx->counter.as<unsigned>(), d_out, dv_score, dv_pos);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    return B200_OK;
}

int sw16_warps() {  // CTA width of the packed kernel (pairs per item = 2 x warps); B200_SW16_WARPS overrides for experiments
    static int w = 0;
    if (w == 0) {
        const char *e = getenv("B200_SW16_WARPS");
        w = (e != nullptr && atoi(e) == 4) ? 4 : 8;
    }
    return w;
}

int launch_sw16(b200_ctx *ctx, const QueryDesc *d_qd, const int8_t *d_pad, int max_Lp, const WorkItem *d_items, uint32_t n_items,
                const PairDesc *d_pairs, int go, int ge, uint2 *d_bnd, int bnd_stride, int32_t *d_out, int mode = 0,
                const int32_t *dv_score = nullptr, const int32_t *dv_pos = nullptr) {
    size_t smem = (size_t) (ctx->alphabet + 1) * max_Lp;
    int smem_profile = 1;
    if (smem > (size_t) ctx->max_smem_optin - 1024) { smem = 0; smem_profile = 0; }
    CU_TRY(ctx, ctx->counter.reserve(sizeof(unsigned)));
    CU_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, sizeof(unsigned), ctx->stream));
    if (mode == 1) return launch_sw16_w<8, 1>(ctx, d_qd, d_pad, smem, smem_profile, d_items, n_items, d_pairs, go, ge, d_bnd, bnd_stride, d_out, dv_score, dv_pos);
    if (mode == 2) return launch_sw16_w<8, 2>(ctx, d_qd, d_pad, smem, smem_profile, d_items, n_items, d_pairs, go, ge, d_bnd, bnd_stride, d_out, dv_score, dv_pos);
    if (sw16_warps() == 4)
        return launch_sw16_w<4, 0>(ctx, d_qd, d_pad, smem, smem_profile, d_items, n_items, d_pairs, go, ge, d_bnd, bnd_stride, d_out);
    return launch_sw16_w<8, 0>(ctx, d_qd, d_pad, smem, smem_profile, d_items, n_items, d_pairs, go, ge, d_bnd, bnd_stride, d_out);
}

}  // namespace


namespace {

// packed (int16x2) kernel over the pairs selected by `mask`: score mode (scores == nullptr; res[i] = score) or FIND mode
// (scores[i] = known score > 0; res[2i], res[2i+1] = end column, end row).  Results land at the caller's pair index.
// rev_ends != nullptr: reverse (start position) pass from the given end positions; res[2i], res[2i+1] = reverse column, row.
int run_sw16_pass(b200_ctx *ctx, const std::vector<QueryDesc> &h_qd, const b200_query *queries, const b200_pair *pairs, uint64_t n,
                  const uint8_t *mask, const int32_t *scores, int go, int ge, std::vector<int32_t> &res, const b200_sw_end *rev_ends) {
    const bool find = scores != nullptr || rev_ends != nullptr;
    SwPlan plan;
    plan_pairs(ctx, queries, pairs, n, mask, plan, 2u * (uint32_t) (find ? 8 : sw16_warps()));
    const uint32_t m = (uint32_t) plan.perm.size();
    if (m == 0) return B200_OK;
    std::vector<PairDesc> h_pd(m);
    int max_cols = 1, max_Lp = 0;
    bool multi = false;
    for (uint32_t s = 0; s < m; s++) {
        const uint32_t i = plan.perm[s];
        h_pd[s].target = pairs[i].target; h_pd[s].qend = 0; h_pd[s].dbend = 0; h_pd[s].score = scores ? scores[i] : 0;
        if (rev_ends) { h_pd[s].qend = rev_ends[i].qend; h_pd[s].dbend = rev_ends[i].dbend; h_pd[s].score = rev_ends[i].score; }
        max_cols = std::max(max_cols, ctx->h_len[pairs[i].target]);
        max_Lp = std::max(max_Lp, h_qd[pairs[i].query].Lp);
        if (h_qd[pairs[i].query].qlen > 512) multi = true;
    }
    const uint32_t n_items = (uint32_t) plan.items.size();
    const int bnd_stride = multi ? (int) round_up((uint64_t) max_cols, 32) + 32 : 32;
    CU_TRY(ctx, ctx->pairs.reserve(sizeof(PairDesc) * m));
    CU_TRY(ctx, ctx->items.reserve(sizeof(WorkItem) * n_items));
    CU_TRY(ctx, ctx->out4.reserve(sizeof(int32_t) * 2 * (size_t) m));
    CU_TRY(ctx, ctx->bnd.reserve(sizeof(int2) * 2 * (size_t) bnd_stride * std::min<uint64_t>(n_items, sw_max_grid(ctx)) * 8));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->pairs.p, h_pd.data(), sizeof(PairDesc) * m, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->items.p, plan.items.data(), sizeof(WorkItem) * n_items, cudaMemcpyHostToDevice, ctx->stream));
    int rc = launch_sw16(ctx, ctx->qdesc.as<QueryDesc>(), ctx->pad.as<int8_t>(), max_Lp, ctx->items.as<WorkItem>(), n_items,
                         ctx->pairs.as<PairDesc>(), go, ge, ctx->bnd.as<uint2>(), bnd_stride, ctx->out4.as<int32_t>(), rev_ends ? 2 : (scores ? 1 : 0));
    if (rc != B200_OK) return rc;
    std::vector<int32_t> h((size_t) m * (find ? 2 : 1));
    CU_TRY(ctx, cudaMemcpyAsync(h.data(), ctx->out4.p, sizeof(int32_t) * h.size(), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t s = 0; s < m; s++) {
        const uint32_t i = plan.perm[s];
        if (find) { res[2 * (size_t) i] = h[2 * (size_t) s]; res[2 * (size_t) i + 1] = h[2 * (size_t) s + 1]; }
        else res[i] = h[s];
    }
    return B200_OK;
}

// score -> FIND -> (reverse) over ONE plan and ONE upload: each launch reads the previous one's output on the device in plan
// order (dv_score / dv_pos), so the host only sees the final scores and positions.  PairDesc.qend carries the gate of the
// reverse pass.  score[i], endpos[2i..], startpos[2i..] land at the caller's pair index for the pairs selected by mask.
int run_sw16_chain(b200_ctx *ctx, const std::vector<QueryDesc> &h_qd, const b200_query *queries, const b200_pair *pairs, uint64_t n,
                   const uint8_t *mask, const uint8_t *gate, bool want_start, int go, int ge, std::vector<int32_t> &score,
                   std::vector<int32_t> &endpos, std::vector<int32_t> *startpos) {
    static const bool trace = getenv("B200_TRACE") != nullptr;   // stderr timing of the phases (development aid)
    const auto t_begin = std::chrono::steady_clock::now();
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    SwPlan plan;
    plan_pairs(ctx, queries, pairs, n, mask, plan, 2u * (uint32_t) sw16_warps());
    const auto t_plan = std::chrono::steady_clock::now();
    const uint32_t m = (uint32_t) plan.perm.size();
    if (m == 0) return B200_OK;
    std::vector<PairDesc> h_pd(m);
    int max_cols = 1, max_Lp = 0;
    bool multi = false;
    for (uint32_t s = 0; s < m; s++) {
        const uint32_t i = plan.perm[s];
        h_pd[s].target = pairs[i].target; h_pd[s].qend = (gate == nullptr || gate[i]) ? 1 : 0; h_pd[s].dbend = 0; h_pd[s].score = 0;
        max_cols = std::max(max_cols, ctx->h_len[pairs[i].target]);
        max_Lp = std::max(max_Lp, h_qd[pairs[i].query].Lp);
        if (h_qd[pairs[i].query].qlen > 512) multi = true;
    }
    const uint32_t n_items = (uint32_t) plan.items.size();
    const int bnd_stride = multi ? (int) round_up((uint64_t) max_cols, 32) + 32 : 32;
    const size_t words = (size_t) m * (want_start ? 5 : 3);   // [score | end (col,row) | start (col,row)]
    CU_TRY(ctx, ctx->pairs.reserve(sizeof(PairDesc) * m));
    CU_TRY(ctx, ctx->items.reserve(sizeof(WorkItem) * n_items));
    CU_TRY(ctx, ctx->out4.reserve(sizeof(int32_t) * words));
    CU_TRY(ctx, ctx->bnd.reserve(sizeof(int2) * 2 * (size_t) bnd_stride * std::min<uint64_t>(n_items, sw_max_grid(ctx)) * 8));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->pairs.p, h_pd.data(), sizeof(PairDesc) * m, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(ctx->items.p, plan.items.data(), sizeof(WorkItem) * n_items, cudaMemcpyHostToDevice, ctx->stream));
    int32_t *d_score = ctx->out4.as<int32_t>(), *d_end = d_score + m, *d_start = d_score + 3 * (size_t) m;
    if (trace) { for (auto &e : ev) cudaEventCreate(&e); cudaEventRecord(ev[0], ctx->stream); }
    for (int mode = 0; mode <= (want_start ? 2 : 1); mode++) {
        int rc = launch_sw16(ctx, ctx->qdesc.as<QueryDesc>(), ctx->pad.as<int8_t>(), max_Lp, ctx->items.as<WorkItem>(), n_items,
                             ctx->pairs.as<PairDesc>(), go, ge, ctx->bnd.as<uint2>(), bnd_stride,
                             mode == 0 ? d_score : (mode == 1 ? d_end : d_start), mode, mode ? d_score : nullptr, mode == 2 ? d_end : nullptr);
        if (rc != B200_OK) return rc;
        if (trace) cudaEventRecord(ev[mode + 1], ctx->stream);
    }
    const auto t_launch = std::chrono::steady_clock::now();
    std::vector<int32_t> h(words);
    CU_TRY(ctx, cudaMemcpyAsync(h.data(), ctx->out4.p, sizeof(int32_t) * words, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    const int32_t *he = h.data() + m, *hs = h.data() + 3 * (size_t) m;
    for (uint32_t s = 0; s < m; s++) {
        const size_t i = plan.perm[s];
        score[i] = h[s];
        endpos[2 * i] = he[2 * (size_t) s]; endpos[2 * i + 1] = he[2 * (size_t) s + 1];
        if (want_start) { (*startpos)[2 * i] = hs[2 * (size_t) s]; (*startpos)[2 * i + 1] = hs[2 * (size_t) s + 1]; }
    }
    if (trace) {
        const auto t_end = std::chrono::steady_clock::now();
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
            return std::chrono::duration<double, std::milli>(b - a).count(); };
        float k[3] = {0, 0, 0};
        for (int mode = 0; mode <= (want_start ? 2 : 1); mode++) cudaEventElapsedTime(&k[mode], ev[mode], ev[mode + 1]);
        fprintf(stderr, "[b200 trace] sw16 chain: %u pairs, plan %.2f ms, stage+launch %.2f ms, kernels score %.2f / find %.2f / reverse %.2f ms, "
                        "wait+d2h+scatter %.2f ms, total %.2f ms\n", m, ms(t_begin, t_plan), ms(t_plan, t_launch), k[0], k[1], k[2],
                ms(t_launch, t_end), ms(t_begin, t_end));
        for (auto &e : ev) cudaEventDestroy(e);
    }
    return B200_OK;
}

}  // namespace

int b200_sw_score_job_create(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go,
                             int ge, b200_job **out) {
    if (ctx == nullptr || out == nullptr) return B200_ERR_ARG;
    *out = nullptr;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return set_err(ctx, B200_ERR_ARG, "sw score job: no pairs");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);
    if (rc != B200_OK) return rc;
    const int A = ctx->alphabet;
    // int16 safety: a local alignment cannot score more than min(qlen,tlen) * (largest profile entry)
    std::vector<int> smax(nq, 1);
    std::vector<int64_t> qsum(nq, 0);
    for (size_t q_ = 0; q_ < (size_t) (nq); q_++) profile_bounds(queries[q_].profile, A, queries[q_].qlen, smax[q_], qsum[q_]);
    b200_job *job = new b200_job();
    job->ctx = ctx; job->kind = 3; job->go = go; job->ge = ge; job->n_pairs = n; job->nq = nq;
    const int klass[2] = {1, 0};  // 1: packed int16x2 kernel (any rows-per-lane flavour), 0: int32 fallback
    std::vector<uint8_t> mask(n);
    int max_cols = 1;
    bool multi = false;
    uint32_t max_items = 1;
    cudaError_t e = cudaSuccess;
    for (int c = 0; c < 2 && e == cudaSuccess; c++) {
        bool any = false;
        for (uint64_t i = 0; i < n; i++) {
            const int qi = (int) pairs[i].query;
            const int tl = ctx->h_len[pairs[i].target];
            const bool packed_ok = go >= ge && int16_safe(smax[qi], qsum[qi], queries[qi].qlen, tl);
            const int k = packed_ok ? 1 : 0;
            mask[i] = (k == klass[c]) ? 1 : 0;
            any |= mask[i] != 0;
            if (c == 0) job->cells += (uint64_t) queries[qi].qlen * (uint64_t) tl;
        }
        if (!any) continue;
        SwPlan plan;
        plan_pairs(ctx, queries, pairs, n, mask.data(), plan, klass[c] ? 2u * (uint32_t) sw16_warps() : kPairsPerItem);
        b200_job::Part *pt = new b200_job::Part();
        job->parts.push_back(pt);
        pt->K = klass[c];
        pt->perm = plan.perm;
        pt->n_pairs = (uint32_t) plan.perm.size();
        pt->n_items = (uint32_t) plan.items.size();
        max_items = std::max(max_items, pt->n_items);
        std::vector<PairDesc> h_pd(pt->n_pairs);
        for (uint32_t sidx = 0; sidx < pt->n_pairs; sidx++) {
            const uint32_t i = plan.perm[sidx];
            h_pd[sidx].target = pairs[i].target; h_pd[sidx].qend = h_pd[sidx].dbend = h_pd[sidx].score = 0;
            max_cols = std::max(max_cols, ctx->h_len[pairs[i].target]);
            pt->max_Lp = std::max(pt->max_Lp, h_qd[pairs[i].query].Lp);
            if (queries[pairs[i].query].qlen > (klass[c] ? 512 : SW_TILE)) multi = true;
        }
        e = pt->pairs.reserve(sizeof(PairDesc) * pt->n_pairs);
        if (e == cudaSuccess) e = pt->items.reserve(sizeof(WorkItem) * pt->n_items);
        if (e == cudaSuccess) e = pt->out.reserve(sizeof(int4) * pt->n_pairs);
        if (e == cudaSuccess) e = cudaMemcpyAsync(pt->pairs.p, h_pd.data(), sizeof(PairDesc) * pt->n_pairs, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(pt->items.p, plan.items.data(), sizeof(WorkItem) * pt->n_items, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    job->bnd_stride = multi ? (int) round_up((uint64_t) max_cols, 32) + 32 : 32;
    const size_t pad_bytes = h_qd.back().p16_off + (size_t) (A + 1) * h_qd.back().Lp;
    if (e == cudaSuccess) e = job->pad.reserve(pad_bytes);
    if (e == cudaSuccess) e = job->qdesc.reserve(sizeof(QueryDesc) * nq);
    if (e == cudaSuccess) e = job->bnd.reserve(sizeof(int2) * 2 * (size_t) job->bnd_stride * std::min<uint64_t>(max_items, sw_max_grid(ctx)) * 8);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->pad.p, ctx->pad.p, pad_bytes, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(job->qdesc.p, h_qd.data(), sizeof(QueryDesc) * nq, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        ctx->err = std::string("sw score job staging: ") + cudaGetErrorString(e);
        job->free_all(); delete job;
        return e == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA;
    }
    *out = job;
    return B200_OK;
}

static int sw_score_job_run_locked(b200_job *job) {
    b200_ctx *ctx = job->ctx;
    for (b200_job::Part *pt : job->parts) {
        int rc;
        if (pt->K > 0)
            rc = launch_sw16(ctx, job->qdesc.as<QueryDesc>(), job->pad.as<int8_t>(), pt->max_Lp, pt->items.as<WorkItem>(),
                             pt->n_items, pt->pairs.as<PairDesc>(), job->go, job->ge, job->bnd.as<uint2>(), job->bnd_stride,
                             pt->out.as<int32_t>());
        else
            rc = launch_sw<1>(ctx, job->qdesc.as<QueryDesc>(), job->pad.as<int8_t>(), pt->max_Lp, pt->items.as<WorkItem>(),
                              pt->n_items, pt->pairs.as<PairDesc>(), job->go, job->ge, job->bnd.as<int2>(), job->bnd_stride,
                              pt->out.as<int4>());
        if (rc != B200_OK) return rc;
    }
    return B200_OK;
}

int b200_sw_score_job_fetch(b200_job *job, int32_t *scores) {
    if (job == nullptr || job->kind != 3 || scores == nullptr) return B200_ERR_ARG;
    b200_ctx *ctx = job->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    for (b200_job::Part *pt : job->parts) {
        if (pt->K > 0) {
            std::vector<int32_t> h(pt->n_pairs);
            CU_TRY(ctx, cudaMemcpyAsync(h.data(), pt->out.p, sizeof(int32_t) * pt->n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            for (uint32_t s = 0; s < pt->n_pairs; s++) scores[pt->perm[s]] = h[s];
        } else {
            std::vector<int4> h(pt->n_pairs);
            CU_TRY(ctx, cudaMemcpyAsync(h.data(), pt->out.p, sizeof(int4) * pt->n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            for (uint32_t s = 0; s < pt->n_pairs; s++) scores[pt->perm[s]] = std::min(h[s].x, 32767);
        }
    }
    return B200_OK;
}

int b200_sw_score(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go, int ge,
                  int32_t *scores) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (scores == nullptr) return set_err(ctx, B200_ERR_ARG, "sw: scores is NULL");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);
    if (rc != B200_OK) return rc;
    const int A = ctx->alphabet;
    std::vector<int> smax(nq, 1);
    std::vector<int64_t> qsum(nq, 0);
    for (size_t q_ = 0; q_ < (size_t) (nq); q_++) profile_bounds(queries[q_].profile, A, queries[q_].qlen, smax[q_], qsum[q_]);
    std::vector<uint8_t> packed(n), rest(n);
    bool any_rest = false, any_packed = false;
    for (uint64_t i = 0; i < n; i++) {
        const int qi = (int) pairs[i].query;
        const bool ok = go >= ge && int16_safe(smax[qi], qsum[qi], queries[qi].qlen, ctx->h_len[pairs[i].target]);
        packed[i] = ok ? 1 : 0; rest[i] = ok ? 0 : 1;
        any_rest |= !ok; any_packed |= ok;
    }
    std::vector<int32_t> sc(n, 0);
    if (any_packed) {
        rc = run_sw16_pass(ctx, h_qd, queries, pairs, n, any_rest ? packed.data() : nullptr, nullptr, go, ge, sc);
        if (rc != B200_OK) return rc;
    }
    if (any_rest) {
        SwPlan plan;
        plan_pairs(ctx, queries, pairs, n, rest.data(), plan);
        std::vector<int4> res;
        rc = run_sw_pass<1>(ctx, h_qd, pairs, plan, nullptr, go, ge, res);
        if (rc != B200_OK) return rc;
        for (uint32_t s2 = 0; s2 < plan.perm.size(); s2++) sc[plan.perm[s2]] = std::min(res[s2].x, 32767);
    }
    memcpy(scores, sc.data(), sizeof(int32_t) * n);
    return B200_OK;
}

// End positions for pairs whose score is already known (a host that gates on the score between the two steps, as
// b200_align_batch does with the E-value): packed FIND pass for the int16-safe pairs, int32 score+end kernel for the rest.
int b200_sw_endpos(b200_ctx *ctx, const b200_query *queries, int nq, const b200_pair *pairs, uint64_t n, int go, int ge,
                   const int32_t *scores, b200_sw_end *out) {
    if (ctx == nullptr) return B200_ERR_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_pairs(ctx, queries, nq, pairs, n, go, ge);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (scores == nullptr || out == nullptr) return set_err(ctx, B200_ERR_ARG, "sw_endpos: NULL argument");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<QueryDesc> h_qd;
    rc = stage_queries(ctx, queries, nq, true, h_qd);
    if (rc != B200_OK) return rc;
    const int A = ctx->alphabet;
    std::vector<int> smax(nq, 1);
    std::vector<int64_t> qsum(nq, 0);
    for (size_t q_ = 0; q_ < (size_t) (nq); q_++) profile_bounds(queries[q_].profile, A, queries[q_].qlen, smax[q_], qsum[q_]);
    std::vector<uint8_t> need(n, 0), rest(n, 0);
    bool any_rest = false, any_need = false;
    for (uint64_t i = 0; i < n; i++) {
        const int qi = (int) pairs[i].query;
        const bool ok = go >= ge && int16_safe(smax[qi], qsum[qi], queries[qi].qlen, ctx->h_len[pairs[i].target]);
        if (scores[i] < 0) return set_err(ctx, B200_ERR_ARG, "sw_endpos: negative score");
        if (ok) { need[i] = scores[i] > 0 ? 1 : 0; any_need |= need[i] != 0; }
        else { rest[i] = 1; any_rest = true; }
    }
    std::vector<int4> res4(n, make_int4(0, -1, -1, 0));
    if (any_need) {
        std::vector<int32_t> pos(2 * n, -1);
        rc = run_sw16_pass(ctx, h_qd, queries, pairs, n, need.data(), scores, go, ge, pos);
        if (rc != B200_OK) return rc;
        for (uint64_t i = 0; i < n; i++) {
            if (!need[i]) continue;
            if (pos[2 * i] < 0 || pos[2 * i] > 0xfffe) return set_err(ctx, B200_ERR_ARG, "sw_endpos: a given score is not the pair's alignment score");
            res4[i] = make_int4(scores[i], pos[2 * i], pos[2 * i + 1], 0);
        }
    }
    if (any_rest) {
        SwPlan plan;
        plan_pairs(ctx, queries, pairs, n, rest.data(), plan);
        std::vector<int4> res;
        rc = run_sw_pass<1>(ctx, h_qd, pairs, plan, nullptr, go, ge, res);
        if (rc != B200_OK) return rc;
        for (uint32_t s2 = 0; s2 < plan.perm.size(); s2++) res4[plan.perm[s2]] = res[s2];
    }
    for (uint64_t i = 0; i < n; i++) report_end(res4[i], queries[pairs[i].query].bias, out[i]);
    return B200_OK;
}

int b200_job_run(b200_job *job) {
    if (job == nullptr) return B200_ERR_ARG;
    b200_ctx *ctx = job->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (job->kind == 1) return scan_job_run_locked(job);
    if (job->kind == 3) return sw_score_job_run_locked(job);
    if (job->kind == 2)
        return launch_sw<1>(ctx, job->qdesc.as<QueryDesc>(), job->pad.as<int8_t>(), job->smem_bytes, job->items.as<WorkItem>(),
                            job->n_items, job->pairs.as<PairDesc>(), job->go, job->ge, job->bnd.as<int2>(), job->bnd_stride,
                            job->out4.as<int4>());
    return B200_ERR_ARG;
}

int b200_sw_job_fetch(b200_job *job, b200_sw_end *out) {
    if (job == nullptr || job->kind != 2 || out == nullptr) return B200_ERR_ARG;
    b200_ctx *ctx = job->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<int4> res(job->n_pairs);
    CU_TRY(ctx, cudaMemcpyAsync(res.data(), job->out4.p, sizeof(int4) * job->n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t s = 0; s < job->n_pairs; s++) {
        const uint32_t i = job->perm[s];
        report_end(res[s], job->h_bias[job->h_pairs[i].query], out[i]);
    }
    return B200_OK;
}

uint64_t b200_job_cells(const b200_job *job) { return job ? job->cells : 0; }

void b200_job_destroy(b200_job *job) {
    if (job == nullptr) return;
    {
        std::lock_guard<std::mutex> lk(job->ctx->mu);
        cudaSetDevice(job->ctx->device);
        cudaStreamSynchronize(job->ctx->stream);
        job->free_all();
    }
    delete job;
}

