// filter.cu -- bit-parallel semi-global kernel (the hot kernel of the :semiglobal path).
//
// One warp per read, one lane per barcode: every lane advances a Myers/Hyyro
// bit-vector column automaton (unit costs, free start and end in the read) for
// its barcode over the read's search range, G independent barcodes per lane for
// ILP.  The barcode match tables (Peq) live in shared memory, transposed so that
// a warp's 32 lanes read 32 consecutive words; the read is streamed once per warp,
// translated to table offsets and broadcast from shared memory.
//
// Barcode rows are TOP-ALIGNED in the W*32-bit vector (row m = the MSB).  The
// unused low bits are "phantom" rows that match every byte and start with a zero
// vertical delta, which keeps them at distance 0 forever, i.e. they are the free
// row 0 of the reference DP (classification.jl:215, :288-295).  With row m in
// the MSB the +-1 update of D[m][j] is the carry-out of the shifts Ph+Ph / Mh+Mh
// (add.cc / addc / subc), so a column costs 13 integer instructions per word.
//
// What the kernel produces per read (DESIGN.md "filter + literal split"):
//   * d_b = min_j D_unit[m_b][j]  for every barcode -- a lower bound of the
//     reference's weighted distance whenever the costs are "benign", so
//     {b : d_b <= floor(allowed_b / min_cost)} is a superset of the barcodes the
//     reference can accept under ANY running threshold (classification.jl:661);
//   * in the exact regime (unit costs, no start/end constraint, score-only) d_b is
//     the reference's distance itself and the running-threshold selection
//     (classification.jl:632-713) is replayed in-warp over the candidates;
//   * otherwise the candidates are queued for the literal kernel.
#include <algorithm>
#include <math_constants.h>

#include "bdx_internal.h"
#include "literal.cuh"

namespace bdx {

constexpr int kFilterWarps = 4;
constexpr int kTile = 256;  // columns staged per pass over the read

template <int W>
struct BV {
    uint32_t w[W];
};

// ---- score update + shift of the horizontal delta vectors -------------------------------
// D[m][j] - D[m][j-1] is +1 when the MSB of Ph is set, -1 when the MSB of Mh is set.
// `mid` = score - msb(mh) is min(D[m][j-1], D[m][j]) (the score moves by at most one per
// column), so taking the running minimum of `mid` at every SECOND column covers both.
// ptxas turns the two updates into LEA.HI on the alu pipe and the shifts into IMAD.IADD on the fma
// pipe; carry-chain (add.cc / subc) and mad.hi codings of the same update measured slower on B200
// (profiles/r01_filter_variants.jsonl) and are gone.
enum { kMyers = 0, kShiftAnd = 5 };  // kShiftAnd: :exact -- Shift-And automaton instead of the edit-distance automaton

template <int CODING>
__device__ __forceinline__ void shift_score(uint32_t ph, uint32_t mh, uint32_t two, uint32_t &phs,
                                            uint32_t &mhs, int &score, int &mid)
{
    (void)two;
    mid = score - (int)(mh >> 31);
    score = mid + (int)(ph >> 31);
    phs = ph << 1;
    mhs = mh << 1;
}

// One column of the automaton for one barcode.  Eq: match mask of this read byte.
template <int CODING>
__device__ __forceinline__ void myers_col(const BV<1> &Eq, BV<1> &Pv, BV<1> &Mv, uint32_t two, int &score,
                                          int &mid)
{
    const uint32_t eq = Eq.w[0], pv = Pv.w[0], mv = Mv.w[0];
    const uint32_t xv = eq | mv;
    const uint32_t xh = ((((eq & pv) + pv) ^ pv) | eq);
    const uint32_t ph = mv | ~(xh | pv);
    const uint32_t mh = pv & xh;
    uint32_t phs, mhs;
    shift_score<CODING>(ph, mh, two, phs, mhs, score, mid);
    Pv.w[0] = mhs | ~(xv | phs);
    Mv.w[0] = phs & xv;
}

template <int CODING>
__device__ __forceinline__ void myers_col(const BV<2> &Eq, BV<2> &Pv, BV<2> &Mv, uint32_t two, int &score,
                                          int &mid)
{
    const uint32_t eq0 = Eq.w[0], eq1 = Eq.w[1], pv0 = Pv.w[0], pv1 = Pv.w[1], mv0 = Mv.w[0], mv1 = Mv.w[1];
    const uint32_t xv0 = eq0 | mv0, xv1 = eq1 | mv1;
    uint32_t t0, t1;
    asm("{\n\t"
        "add.cc.u32 %0, %2, %3;\n\t"
        "addc.u32 %1, %4, %5;\n\t"
        "}"
        : "=&r"(t0), "=r"(t1)
        : "r"(eq0 & pv0), "r"(pv0), "r"(eq1 & pv1), "r"(pv1));
    const uint32_t xh0 = (t0 ^ pv0) | eq0, xh1 = (t1 ^ pv1) | eq1;
    const uint32_t ph0 = mv0 | ~(xh0 | pv0), ph1 = mv1 | ~(xh1 | pv1);
    const uint32_t mh0 = pv0 & xh0, mh1 = pv1 & xh1;
    uint32_t phs1, mhs1;
    shift_score<CODING>(ph1, mh1, two, phs1, mhs1, score, mid);   // row m = MSB of the high word
    phs1 |= ph0 >> 31;
    mhs1 |= mh0 >> 31;
    const uint32_t phs0 = ph0 << 1, mhs0 = mh0 << 1;
    Pv.w[0] = mhs0 | ~(xv0 | phs0);
    Pv.w[1] = mhs1 | ~(xv1 | phs1);
    Mv.w[0] = phs0 & xv0;
    Mv.w[1] = phs1 & xv1;
}

template <int W>
__device__ __forceinline__ void init_rows(int m, BV<W> &Pv, BV<W> &Mv)
{
    // vertical delta +1 on the m real rows (D[i][start-1] = i, classification.jl:278-279
    // with indel = 1), 0 on the phantom rows below them
    if (W == 1) {
        Pv.w[0] = m <= 0 ? 0u : (m >= 32 ? 0xFFFFFFFFu : (0xFFFFFFFFu << (32 - m)));
    } else {
        if (m <= 32) {
            Pv.w[1] = m <= 0 ? 0u : (m == 32 ? 0xFFFFFFFFu : (0xFFFFFFFFu << (32 - m)));
            Pv.w[0] = 0u;
        } else {
            Pv.w[1] = 0xFFFFFFFFu;
            Pv.w[0] = m >= 64 ? 0xFFFFFFFFu : (0xFFFFFFFFu << (64 - m));
        }
    }
#pragma unroll
    for (int k = 0; k < W; k++) Mv.w[k] = 0u;
}

// One read column for the G barcodes of a lane.  TRACK: 0 = automaton only (column before
// min_end_pos), 1 = best = min(best, D[m][j]), 2 = best = min(best, mid) which covers
// columns j-1 and j at once.
template <int W, int G, int CODING, int TRACK>
__device__ __forceinline__ void column(const uint32_t *lane_base, uint32_t byte_off, int plane, uint32_t two,
                                       BV<W> (&Pv)[G], BV<W> (&Mv)[G], int (&score)[G], int (&best)[G])
{
    const uint32_t *p = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(lane_base) + byte_off);
#pragma unroll
    for (int q = 0; q < G; q++) {
        BV<W> Eq;
#pragma unroll
        for (int k = 0; k < W; k++) Eq.w[k] = p[k * plane + q * 32];
        if constexpr (CODING == kShiftAnd) {
            // R = ((R << 1) | 1) & Eq: bit i = "barcode prefix of length i+1 ends at this column".
            // The phantom low bits are all ones (Eq and the initial state), so the shifted-in
            // bit of row 1 is always 1; the MSB says "the whole barcode ends here".  best[]
            // ORs the states of the tracked columns; its sign bit marks a candidate.
            BV<W> &R = Pv[q];
            if (W == 1) {
                R.w[0] = (R.w[0] * 2u + 1u) & Eq.w[0];
            } else {
                const uint32_t hi = (R.w[W - 1] << 1) | (R.w[0] >> 31);
                R.w[0] = (R.w[0] * 2u + 1u) & Eq.w[0];
                R.w[W - 1] = hi & Eq.w[W - 1];
            }
            if (TRACK != 0) best[q] |= (int)R.w[W - 1];
        } else {
            int mid;
            myers_col<CODING>(Eq, Pv[q], Mv[q], two, score[q], mid);
            if (TRACK == 1) best[q] = min(best[q], score[q]);
            if (TRACK == 2) best[q] = min(best[q], mid);
        }
    }
}

// Shared memory carve-up (dynamic):
//   uint32 peq[W][n_classes][n_bc_pad] | uint32 stage[kFilterWarps][kTile] |
//   int16 fa[n_bc_pad] | uint8 len[n_bc_pad] | uint8 class_of[256]
#ifndef BDX_FILTER_MINBLOCKS
#define BDX_FILTER_MINBLOCKS 1
#endif
template <int W, int G, int CODING, bool PAIR>
__global__ void __launch_bounds__(kFilterWarps * 32, BDX_FILTER_MINBLOCKS)
k_filter(const __grid_constant__ DevParams P, const int pass, const uint8_t *__restrict__ seq,
         const int *__restrict__ off, const int n_reads, PassOut *__restrict__ out,
         const PassOut *__restrict__ prev_pass, uint16_t *__restrict__ cand,
         uint8_t *__restrict__ cand_cnt, unsigned long long *__restrict__ counters,
         const int *__restrict__ worklist, const int *__restrict__ n_work, int *__restrict__ wl_full,
         int *__restrict__ n_full)
{
    extern __shared__ __align__(16) uint32_t smem[];
    const DevSet &S = P.set[pass];
    const int n_pad = S.n_bc_pad;
    const int plane = S.n_classes * n_pad;          // words per bit-vector word plane
    uint32_t *peq_s = smem;
    uint32_t *stage_all = peq_s + W * plane;
    int16_t *fa_s = reinterpret_cast<int16_t *>(stage_all + kFilterWarps * kTile);
    uint8_t *len_s = reinterpret_cast<uint8_t *>(fa_s + n_pad);
    uint8_t *class_s = len_s + n_pad;

    for (int k = threadIdx.x; k < W * plane; k += blockDim.x) peq_s[k] = S.peq[k];
    for (int k = threadIdx.x; k < n_pad; k += blockDim.x) {
        fa_s[k] = (int16_t)max(-1, min(S.filt_allowed[k], 32767));
        len_s[k] = (uint8_t)(k < S.n_bc ? S.bc_off[k + 1] - S.bc_off[k] : 0);
    }
    for (int k = threadIdx.x; k < 256; k += blockDim.x) class_s[k] = S.class_of[k];
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    uint32_t *stage = stage_all + warp * kTile;
    unsigned int n_automaton = 0;
    const int warps_total = gridDim.x * kFilterWarps;
    const bool with_delta = P.min_delta != 0.0;
    const bool need_tb = S.trim_side != 0 || P.want_stats;
    const uint32_t row_bytes = (uint32_t)n_pad * 4u;
    const uint32_t two = (uint32_t)P.two;

    // With a worklist (left by k_prefilter) only the unresolved reads are visited.
    const int n_items = worklist ? *n_work : n_reads;
    for (int item = blockIdx.x * kFilterWarps + warp; item < n_items; item += warps_total) {
        const int read = worklist ? worklist[item] : item;
        if (pass == 1 && prev_pass[read].bc <= 0) {             // classification.jl:879-888
            if (lane == 0) out[read] = PassOut{kBcNotRun, 0, -1, -1};
            continue;
        }
        const int base = off[read];
        const int n = off[read + 1] - base;
        const uint8_t *r = seq + base;
        const Geometry g = pass_geometry(S, n);
        if (!g.valid) {                                          // :805-807
            if (lane == 0) out[read] = PassOut{kBcUnknown, 0, -1, -1};
            continue;
        }
        // exact regime: the filter distance IS the reference's distance (DESIGN.md)
        const bool fast = P.algo == BDX_SEMIGLOBAL && P.unit_costs && !need_tb && g.max_start_pos >= n &&
                          g.min_end_pos <= g.start_j;
        const int first_tracked = max(g.start_j, g.min_end_pos);  // hits need j >= min_end_pos (:419)
        // :hamming / :exact constrain the START to the search range; the match itself may run
        // past its end (classification.jl:490-491, :570-571)
        const int last_col = P.algo == BDX_SEMIGLOBAL ? g.end_j : min(n, g.end_j + S.max_m - 1);

        BestState bs;
        best_init(bs, P.max_error_rate);
        int n_cand = 0;

        // Reads whose columns fit one tile are staged once (not once per barcode chunk).
        const bool single_tile = last_col - g.start_j + 1 <= kTile;
        if (single_tile) {
            const int tlen = last_col - g.start_j + 1;
            __syncwarp();
            for (int t = lane; t < tlen; t += 32)
                stage[t] = (uint32_t)class_s[r[g.start_j - 1 + t]] * row_bytes;
            __syncwarp();
        }

        n_automaton++;

        for (int chunk = 0; chunk < n_pad; chunk += 32 * G) {
            BV<W> Pv[G], Mv[G];
            int score[G], best[G];
#pragma unroll
            for (int q = 0; q < G; q++) {
                const int m = len_s[chunk + q * 32 + lane];
                init_rows<W>(m, Pv[q], Mv[q]);
                score[q] = m;
                best[q] = kInf;
                if constexpr (CODING == kShiftAnd) {
#pragma unroll
                    for (int k = 0; k < W; k++) Pv[q].w[k] = ~Pv[q].w[k];   // phantom rows = 1, real rows = 0
                    best[q] = 0;
                }
            }
            const uint32_t *lane_base = peq_s + chunk + lane;

            for (int tile0 = g.start_j; tile0 <= last_col; tile0 += kTile) {
                const int tlen = min(kTile, last_col - tile0 + 1);
                if (!single_tile) {
                    __syncwarp();
                    for (int t = lane; t < tlen; t += 32)
                        stage[t] = (uint32_t)class_s[r[tile0 - 1 + t]] * row_bytes;
                    __syncwarp();
                }
                // columns before min_end_pos advance the automaton but are not hits
                int t = 0;
                const int untracked = min(tlen, max(0, first_tracked - tile0));
                for (; t < untracked; t++)
                    column<W, G, CODING, 0>(lane_base, stage[t], plane, two, Pv, Mv, score, best);
                // align to 4 so that the staged offsets can be fetched as one 128-bit load
                for (; t < tlen && (t & 3); t++)
                    column<W, G, CODING, 1>(lane_base, stage[t], plane, two, Pv, Mv, score, best);
                for (; t + 4 <= tlen; t += 4) {
                    const uint4 o4 = *reinterpret_cast<const uint4 *>(stage + t);
                    if (PAIR) {
                        column<W, G, CODING, 0>(lane_base, o4.x, plane, two, Pv, Mv, score, best);
                        column<W, G, CODING, 2>(lane_base, o4.y, plane, two, Pv, Mv, score, best);
                        column<W, G, CODING, 0>(lane_base, o4.z, plane, two, Pv, Mv, score, best);
                        column<W, G, CODING, 2>(lane_base, o4.w, plane, two, Pv, Mv, score, best);
                    } else {
                        column<W, G, CODING, 1>(lane_base, o4.x, plane, two, Pv, Mv, score, best);
                        column<W, G, CODING, 1>(lane_base, o4.y, plane, two, Pv, Mv, score, best);
                        column<W, G, CODING, 1>(lane_base, o4.z, plane, two, Pv, Mv, score, best);
                        column<W, G, CODING, 1>(lane_base, o4.w, plane, two, Pv, Mv, score, best);
                    }
                }
                for (; t < tlen; t++)
                    column<W, G, CODING, 1>(lane_base, stage[t], plane, two, Pv, Mv, score, best);
            }

            // candidates of this chunk, visited in barcode (file) order
#pragma unroll
            for (int q = 0; q < G; q++) {
                const int b0 = chunk + q * 32;
                const bool is_cand = CODING == kShiftAnd ? (best[q] < 0 && fa_s[b0 + lane] >= 0)
                                                         : best[q] <= (int)fa_s[b0 + lane];
                uint32_t mask = __ballot_sync(0xFFFFFFFFu, is_cand);
                while (mask) {
                    const int l = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const int b = b0 + l;
                    if (fast) {
                        const int d = __shfl_sync(0xFFFFFFFFu, best[q], l);
                        const int norm = S.norm[b];
                        const int allowed = allowed_from(bs.thr, norm);                      // :254
                        const double score_b = d <= allowed ? __ddiv_rn((double)d, (double)norm) : CUDART_INF;
                        best_consider(bs, with_delta, score_b, d, b + 1, -1, -1);
                    } else {
                        if (n_cand < kCandMax && lane == 0) cand[(size_t)read * kCandMax + n_cand] = (uint16_t)b;
                        n_cand++;
                    }
                }
            }
        }

        if (lane == 0) {
            if (fast) {
                out[read] = best_finish(bs, with_delta, P.min_delta);
            } else if (n_cand == 0) {
                out[read] = PassOut{kBcUnknown, 0, -1, -1};   // every barcode returns Inf (:820-821)
            } else {
                cand_cnt[read] = (uint8_t)(n_cand > kCandMax ? kCandOverflow : n_cand);
                out[read] = PassOut{kBcPending, 0, -1, -1};
                wl_full[atomicAdd(n_full, 1)] = read;     // k_literal walks this compacted list
            }
        }
    }
    if (counters && lane == 0 && n_automaton) atomicAdd(counters + 1, (unsigned long long)n_automaton);
}

// ---------------------------------------------------------------------------------------
// k_prefilter: perfect-occurrence prefilter, one thread per read.
//
// With default start / end ranges, match = 0, positive edit costs and no min_delta, a barcode that occurs verbatim
// inside the search range scores 0, the running threshold drops to 0 and no later barcode can be accepted
// (score < min_score is strict, classification.jl:658); an earlier barcode wins only with a
// score of 0 itself, i.e. if IT occurs verbatim.  So the answer for such a read is the
// lowest-index barcode with a verbatim occurrence: found by hashing the q-mers of sampled
// columns (every pf_stride-th column; pf_stride = 1: a rolling hash over every column) against
// a table of barcode q-mer hashes in shared memory, and byte-wise verification on a hit.
// Resolved reads get their PassOut here; all other reads are appended to the worklist the
// bit-parallel kernel then walks.
// ---------------------------------------------------------------------------------------
constexpr int kPfThreads = 256;
constexpr int kPfStageBytes = 48 * 1024;   // raw bytes of one group of 256 reads (<= 192 bases each)
constexpr int kPfMaxCand = 2;              // table hits remembered per read; more => leave it to the DP

// Hash scan of one read's search range.  Table hits are only RECORDED in the loop
// and verified byte by byte afterwards, when all lanes of the warp verify together (doing
// it inside the loop serialises the lanes: each finds its hit at a different column).
// Every table entry (barcode b, offset o) that the q-mer at column w hashes to names the
// candidate start w - o.  Returns the lowest barcode index with a verified verbatim occurrence,
// 0x7FFFFFFF if none, or -1 if there were more table hits than kPfMaxCand (the caller then
// leaves the read to the bit-parallel kernel, which is always correct).  found_w: the start
// of the chosen occurrence of that barcode, leftmost or (want_rightmost) rightmost.
// SAMPLED: the table may be a sampled one (k_prefilter<0>); otherwise pf_stride is 1.  STAGED: c0 points into the
// shared-memory stage.
template <bool SAMPLED, bool STAGED, typename BytePtr>
__device__ __forceinline__ int pf_scan(BytePtr c0, int ncols, const DevSet &S, const uint32_t *keys_s,
                                       const uint32_t *vals_s, const uint32_t *bitmap_s, bool want_rightmost,
                                       int &found_w)
{
    const int seed = S.pf_seed;
    const int stride = S.pf_stride;
    const int bm_log2 = S.pf_bm_log2;
    const uint32_t size_mask = (1u << S.pf_log2) - 1u;
    // The loop only REMEMBERS the (few) columns whose hash passes the first-level bitmap; the table is probed
    // after the loop, when the lanes of a warp probe together.  Probing inside the loop ran the probe for one lane
    // at a time -- each lane passes the bitmap at a different column -- and cost a fifth of the kernel's
    // instructions (ncu source view, profiles/r02_kernels_ncu_summary.txt).
    constexpr int kRec = 4;
    int rw0 = 0, rw1 = 0, rw2 = 0, rw3 = 0, n_rec = 0;
    uint32_t rh0 = 0, rh1 = 0, rh2 = 0, rh3 = 0;
    auto record = [&](int w, uint32_t h) {
        if (n_rec == 0) { rw0 = w; rh0 = h; }
        else if (n_rec == 1) { rw1 = w; rh1 = h; }
        else if (n_rec == 2) { rw2 = w; rh2 = h; }
        else if (n_rec == 3) { rw3 = w; rh3 = h; }
        n_rec++;
    };
    auto passes = [&](uint32_t h) {                          // rare: some barcode q-mer hashes here
        const uint32_t bit = pf_bit(h, bm_log2);
        return (bitmap_s[bit >> 5] >> (bit & 31)) & 1u;
    };
    if (!SAMPLED || stride == 1) {
        const uint32_t pw = S.pf_pow;
        uint32_t h = 0;
        for (int i = 0; i < seed; i++) h = h * kPfBase + (uint32_t)c0[i];
        const int nwin = ncols - seed + 1;
        const auto *c_in = c0 + seed;
#pragma unroll 4
        for (int w = 0; w < nwin - 1; w++) {
            if (passes(h)) record(w, h);
            h = (h - (uint32_t)c0[w] * pw) * kPfBase + (uint32_t)c_in[w];
        }
        if (nwin > 0 && passes(h)) record(nwin - 1, h);
    } else {
        // sampled columns are several columns apart: each q-mer (kPfMinSeed <= q <= kPfMaxSeed) is read as three
        // little-endian words, bytes q.. masked off (pf_words_hash).  From the stage: the four aligned words around
        // it, funnel-shifted (the stage has 16 bytes of slack behind the last read); from global memory: byte by byte.
        const uint32_t m1 = seed >= 8 ? 0xFFFFFFFFu : (1u << (8 * (seed - 4))) - 1u;
        const uint32_t m2 = seed >= 12 ? 0xFFFFFFFFu : (seed <= 8 ? 0u : (1u << (8 * (seed - 8))) - 1u);
        auto qmer_hash = [&](int w) {
            const auto *c = c0 + w;
            uint32_t x0, x1, x2;
            if constexpr (STAGED) {
                const uint32_t mis = (uint32_t)reinterpret_cast<uintptr_t>(c) & 3u;
                const uint32_t *a = reinterpret_cast<const uint32_t *>(c - mis);
                const uint32_t y0 = a[0], y1 = a[1], y2 = a[2], y3 = a[3];
                x0 = __funnelshift_r(y0, y1, 8 * mis);
                x1 = __funnelshift_r(y1, y2, 8 * mis);
                x2 = __funnelshift_r(y2, y3, 8 * mis);
            } else {
                x0 = (uint32_t)c[0] | (uint32_t)c[1] << 8 | (uint32_t)c[2] << 16 | (uint32_t)c[3] << 24;
                x1 = x2 = 0u;
#pragma unroll
                for (int i = 4; i < kPfMaxSeed; i++)
                    if (i < seed) (i < 8 ? x1 : x2) |= (uint32_t)c[i] << (8 * (i % 4));
            }
            return pf_words_hash(x0, x1 & m1, x2 & m2);
        };
        // the bitmap passes of up to 32 probes are collected as bits and recorded (hash recomputed) afterwards:
        // recording inside the loop made ptxas move the record registers at every probe
        const int n_probes = (ncols - seed) / stride + 1;
        for (int k0 = 0; k0 < n_probes; k0 += 32) {
            const int k1 = min(n_probes, k0 + 32);
            uint32_t pass_bits = 0;
            for (int k = k0; k < k1; k++) pass_bits |= passes(qmer_hash(k * stride)) << (k - k0);
            while (pass_bits) {
                const int k = k0 + __ffs(pass_bits) - 1;
                pass_bits &= pass_bits - 1;
                record(k * stride, qmer_hash(k * stride));
            }
        }
    }
    if (n_rec > kRec) return -1;                              // more bitmap hits than remembered: leave it to the DP
    static_assert(kPfMaxCand == 2, "candidates are kept in scalars");
    int cb0 = 0, cs0 = 0, cb1 = 0, cs1 = 0, nc = 0;     // (barcode, start); an indexed array went to local memory
#pragma unroll
    for (int k = 0; k < kRec; k++) {
        if (k >= n_rec) continue;
        const int w = k == 0 ? rw0 : (k == 1 ? rw1 : (k == 2 ? rw2 : rw3));
        const uint32_t hk = k == 0 ? rh0 : (k == 1 ? rh1 : (k == 2 ? rh2 : rh3));
        uint32_t slot = pf_slot(hk, S.pf_log2);
        for (;;) {
            const uint32_t v = vals_s[slot];
            if (v == kPfEmpty) break;
            const int s = w - pf_val_off(v);                  // candidate start
            if (keys_s[slot] == hk && s >= 0 && s + pf_val_len(v) <= ncols) {
                if (nc == 0) { cb0 = pf_val_bc(v); cs0 = s; }
                else if (nc == 1) { cb1 = pf_val_bc(v); cs1 = s; }
                nc++;
            }
            slot = (slot + 1) & size_mask;
        }
    }
    if (nc > kPfMaxCand) return -1;
    int found = 0x7FFFFFFF;
    found_w = -1;
#pragma unroll
    for (int k = 0; k < kPfMaxCand; k++) {
        // another occurrence of the SAME barcode replaces the position only when it starts further left, or further
        // right when the rightmost one is wanted (trim_side == 3, classification.jl:613-619).  Starts are compared,
        // not scan order: a barcode with an internal repeat can yield two candidates at one sampled column.
        const int cb = k == 0 ? cb0 : cb1, cs = k == 0 ? cs0 : cs1;
        if (k < nc && (cb < found || (cb == found && (want_rightmost ? cs > found_w : cs < found_w)))) {
            const int b = cb;
            const uint8_t *q = S.bc_bytes + S.bc_off[b];
            const int len = S.bc_off[b + 1] - S.bc_off[b];
            bool same = true;
            for (int i = 0; i < len; i++)
                if (q[i] != c0[cs + i]) { same = false; break; }
            if (same) {
                found = b;
                found_w = cs;
            }
        }
    }
    return found;
}

// :exact -- the same rolling-hash scan used as a CANDIDATE GENERATOR: every barcode whose
// seed-length prefix occurs at a column where the whole barcode still fits in the read is
// appended (distinct, ascending) to the read's candidate list; exact_literal then applies the
// reference's start/end/trim rules to those few barcodes (classification.jl:485-548).  The
// list is a superset of the barcodes with a valid occurrence, so the result is unchanged.
// Returns the number of distinct candidates, or kCandOverflow.
template <typename BytePtr>
__device__ __forceinline__ int pf_scan_exact(BytePtr c0, int n_starts, int cols_left, const DevSet &S,
                                             const uint32_t *keys_s, const uint32_t *vals_s,
                                             const uint32_t *bitmap_s, uint16_t *list)
{
    // c0 = first allowed start column; n_starts start columns are scanned; cols_left = read
    // columns available from c0 to the end of the read
    const int seed = S.pf_seed;
    const uint32_t pw = S.pf_pow;
    const int bm_log2 = S.pf_bm_log2;
    const uint32_t size_mask = (1u << S.pf_log2) - 1u;
    uint32_t h = 0;
    for (int i = 0; i < seed; i++) h = h * kPfBase + (uint32_t)c0[i];
    int nc = 0;
    for (int w = 0;;) {
        const uint32_t bit = pf_bit(h, bm_log2);
        if ((bitmap_s[bit >> 5] >> (bit & 31)) & 1u) {
            uint32_t slot = pf_slot(h, S.pf_log2);
            for (;;) {
                const uint32_t v = vals_s[slot];
                if (v == kPfEmpty) break;
                if (keys_s[slot] == h && w + pf_val_len(v) <= cols_left && nc != kCandOverflow) {
                    const uint16_t b = (uint16_t)pf_val_bc(v);
                    int pos = 0;                                   // sorted insert, skip duplicates
                    while (pos < nc && list[pos] < b) pos++;
                    if (pos == nc || list[pos] != b) {
                        if (nc == kCandMax) {
                            nc = kCandOverflow;
                        } else {
                            for (int k = nc; k > pos; k--) list[k] = list[k - 1];
                            list[pos] = b;
                            nc++;
                        }
                    }
                }
                slot = (slot + 1) & size_mask;
            }
        }
        if (++w >= n_starts) break;
        h = (h - (uint32_t)c0[w - 1] * pw) * kPfBase + (uint32_t)c0[w - 1 + seed];
    }
    return nc;
}

template <int MODE>   // 0: semiglobal perfect-occurrence resolve, 1: :exact candidate generation,
                      // 2: :hamming perfect-occurrence resolve (with positions)
__global__ void __launch_bounds__(kPfThreads)
k_prefilter(const __grid_constant__ DevParams P, const int pass, const uint8_t *__restrict__ seq,
            const int *__restrict__ off, const int n_reads, PassOut *__restrict__ out,
            const PassOut *__restrict__ prev_pass, int *__restrict__ worklist, int *__restrict__ n_work,
            unsigned long long *__restrict__ counters, uint16_t *__restrict__ cand, uint8_t *__restrict__ cand_cnt)
{
    extern __shared__ __align__(16) uint32_t smem[];
    const DevSet &S = P.set[pass];
    const int pf_size = 1 << S.pf_log2;
    const int bm_words = 1 << (S.pf_bm_log2 - 5);
    uint8_t *stage = reinterpret_cast<uint8_t *>(smem);                     // kPfStageBytes + 16
    uint32_t *keys_s = smem + (kPfStageBytes + 16) / 4;
    uint32_t *vals_s = keys_s + pf_size;
    uint32_t *bitmap_s = vals_s + pf_size;
    for (int k = threadIdx.x; k < pf_size; k += blockDim.x) {
        keys_s[k] = S.pf_keys[k];
        vals_s[k] = S.pf_vals[k];
    }
    for (int k = threadIdx.x; k < bm_words; k += blockDim.x) bitmap_s[k] = S.pf_bitmap[k];

    const int lane = threadIdx.x & 31;
    const int seed = S.pf_seed;
    const int n_groups = (n_reads + kPfThreads - 1) / kPfThreads;
    unsigned int n_done = 0;

    // persistent blocks: the tables are loaded once, then groups of 256 consecutive reads
    for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        const int r0 = grp * kPfThreads;
        const int r1 = min(r0 + kPfThreads, n_reads);
        // The group's reads are contiguous in the packed batch: copy them to shared memory with
        // 128-bit coalesced loads (from the enclosing 16-byte aligned window), then every
        // thread walks its own read from there.
        const int blk_base = off[r0];
        const int blk_end = off[r1];
        const uintptr_t g0 = reinterpret_cast<uintptr_t>(seq + blk_base);
        const int skew = (int)(g0 & 15);                       // stage[skew + k] = seq[blk_base + k]
        const bool staged = blk_end - blk_base + skew <= kPfStageBytes;
        __syncthreads();                                       // previous group done with `stage`
        if (staged) {
            const uint8_t *src = seq + blk_base - skew;        // 16-byte aligned
            const int total = blk_end - blk_base + skew;
            const int vecs = total >> 4;
            const uint4 *src16 = reinterpret_cast<const uint4 *>(src);
            uint4 *dst16 = reinterpret_cast<uint4 *>(stage);
            for (int k = threadIdx.x; k < vecs; k += blockDim.x) dst16[k] = __ldg(src16 + k);
            for (int k = (vecs << 4) + threadIdx.x; k < total; k += blockDim.x) stage[k] = src[k];
        }
        __syncthreads();

        const int read = r0 + threadIdx.x;
        bool resolved = false;
        if (MODE == 1) {
            // every read is finished here: NotRun / Unknown directly, else a candidate list
            if (read < n_reads) {
                resolved = true;
                if (pass == 1 && prev_pass[read].bc <= 0) {
                    out[read] = PassOut{kBcNotRun, 0, -1, -1};
                } else {
                    const int base = off[read];
                    const int n = off[read + 1] - base;
                    const Geometry g = pass_geometry(S, n);
                    // start columns: [start_j, min(end_j, n - seed + 1)] (classification.jl:490-491;
                    // max_start_pos is left to exact_literal)
                    const int n_starts = min(g.end_j, n - seed + 1) - g.start_j + 1;
                    int nc = 0;
                    uint16_t *list = cand + (size_t)read * kCandMax;
                    if (g.valid && n_starts > 0) {
                        const int cols_left = n - g.start_j + 1;
                        if (staged)
                            nc = pf_scan_exact(stage + skew + (base - blk_base) + g.start_j - 1, n_starts, cols_left, S,
                                               keys_s, vals_s, bitmap_s, list);
                        else
                            nc = pf_scan_exact(seq + base + g.start_j - 1, n_starts, cols_left, S, keys_s, vals_s,
                                               bitmap_s, list);
                    }
                    if (nc == 0) {
                        out[read] = PassOut{kBcUnknown, 0, -1, -1};    // no barcode occurs (:820-821)
                    } else {
                        cand_cnt[read] = (uint8_t)nc;
                        out[read] = PassOut{kBcPending, 0, -1, -1};
                    }
                }
            }
        } else if (read < n_reads && !(pass == 1 && prev_pass[read].bc <= 0)) {
            const int base = off[read];
            const int n = off[read + 1] - base;
            const Geometry g = pass_geometry(S, n);
            const int ncols = g.end_j - g.start_j + 1;
            if (MODE == 2) {
                // :hamming -- a placement with 0 mismatches is a verbatim occurrence whose START lies
                // in [start_j, min(end_j, max_start_pos, n - m + 1)] and whose end is >= min_end_pos
                // (classification.jl:570-586).  The scan covers every column such a placement can touch.
                const int last_start = min(g.end_j, g.max_start_pos);
                const int cols = min(n, last_start + S.max_m - 1) - g.start_j + 1;   // columns a valid placement can touch
                if (g.valid && cols >= seed) {
                    int found, w = -1;
                    const bool right = S.trim_side == 3;
                    if (staged)
                        found = pf_scan<false, true>(stage + skew + (base - blk_base) + g.start_j - 1, cols, S, keys_s, vals_s,
                                        bitmap_s, right, w);
                    else
                        found = pf_scan<false, false>(seq + base + g.start_j - 1, cols, S, keys_s, vals_s, bitmap_s, right, w);
                    if (found >= 0 && found != 0x7FFFFFFF) {
                        const int m = S.bc_off[found + 1] - S.bc_off[found];
                        const int s1 = g.start_j + w;                       // 1-based start
                        // `found` is the lowest index among ALL occurrences seen; if its chosen
                        // (leftmost / rightmost) occurrence is a valid placement it is also the
                        // reference's answer, otherwise the DP path decides
                        if (s1 <= min(last_start, n - m + 1) && s1 + m - 1 >= g.min_end_pos) {
                            out[read] = PassOut{found + 1, 0, s1, s1 + m - 1};
                            resolved = true;
                        }
                    }
                }
            } else if (g.valid && g.max_start_pos >= n && g.min_end_pos <= g.start_j && ncols >= seed) {
                // same per-read regime test as k_filter's `fast` (the cost conditions are config-level and
                // checked by the pass plan, plan.cu)
                // Positions (trimming / stats): every hit of the winning barcode scores 0, so the reference keeps
                // the first one it meets (early exit for trim 5, no later hit is strictly better otherwise,
                // classification.jl:419-436, :141-153) -- the leftmost occurrence -- or, trimming 3', the one
                // with the largest start: the rightmost occurrence.  A verbatim hit is one diagonal: start = end - m + 1.
                const bool need_tb = S.trim_side != 0 || P.want_stats;
                int found, w;
                if (staged)
                    found = pf_scan<true, true>(stage + skew + (base - blk_base) + g.start_j - 1, ncols, S, keys_s, vals_s,
                                    bitmap_s, S.trim_side == 3, w);
                else
                    found = pf_scan<true, false>(seq + base + g.start_j - 1, ncols, S, keys_s, vals_s, bitmap_s, S.trim_side == 3, w);
                if (found >= 0 && found != 0x7FFFFFFF) {
                    const int s1 = g.start_j + w, len = S.bc_off[found + 1] - S.bc_off[found];
                    out[read] = PassOut{found + 1, 0, need_tb ? s1 : -1, need_tb ? s1 + len - 1 : -1};
                    resolved = true;
                }
            }
        }
        if (MODE == 1) continue;
        // warp-aggregated append of the unresolved reads
        const bool todo = read < n_reads && !resolved;
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, todo);
        int base_slot = 0;
        if (lane == 0 && mask) base_slot = atomicAdd(n_work, __popc(mask));
        base_slot = __shfl_sync(0xFFFFFFFFu, base_slot, 0);
        if (todo) worklist[base_slot + __popc(mask & ((1u << lane) - 1u))] = read;
        n_done += __popc(__ballot_sync(0xFFFFFFFFu, resolved));
    }
    if (lane == 0 && n_done && counters) atomicAdd(counters + 0, (unsigned long long)n_done);
}

cudaError_t launch_prefilter(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                             const Scratch &sc, int sm_count, unsigned long long *counters, cudaStream_t st)
{
    const DevSet &S = P.set[pass];
    const size_t smem = prefilter_smem_bytes(S);
    auto kern = P.algo == BDX_EXACT ? k_prefilter<1> : (P.algo == BDX_HAMMING ? k_prefilter<2> : k_prefilter<0>);
    int blocks = 0;
    cudaError_t e = resident_grid((const void *)kern, kPfThreads, smem, (n + kPfThreads - 1) / kPfThreads, sm_count, &blocks);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(sc.n_work, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    kern<<<blocks, kPfThreads, smem, st>>>(P, pass, seq, off, n, sc.pass[pass], sc.pass[0], sc.worklist, sc.n_work,
                                           counters, sc.cand, sc.cand_cnt);
    return cudaGetLastError();
}

size_t filter_smem_bytes(const DevSet &S)
{
    const size_t n_pad = (size_t)S.n_bc_pad;
    size_t b = (size_t)S.words * S.n_classes * n_pad * 4;
    b += (size_t)kFilterWarps * kTile * 4;
    b += n_pad * 2 + n_pad + 256;
    return (b + 15) & ~(size_t)15;
}

template <int W, int G, int CODING, bool PAIR>
static cudaError_t launch_wgv(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                              const Scratch &sc, int sm_count, unsigned long long *counters, const int *wl, const int *n_wl,
                              cudaStream_t st)
{
    const size_t smem = filter_smem_bytes(P.set[pass]);
    auto kern = k_filter<W, G, CODING, PAIR>;
    // persistent grid: a whole number of resident blocks per SM, capped by the work
    int blocks = 0;
    const cudaError_t e = resident_grid((const void *)kern, kFilterWarps * 32, smem,
                                        ((long long)n + kFilterWarps - 1) / kFilterWarps, sm_count, &blocks);
    if (e != cudaSuccess) return e;
    kern<<<blocks, kFilterWarps * 32, smem, st>>>(P, pass, seq, off, n, sc.pass[pass], sc.pass[0],
                                                  sc.cand, sc.cand_cnt, counters, wl, n_wl, sc.wl_full, sc.n_lit + 1);
    return cudaGetLastError();
}

template <int W, int G>
static cudaError_t launch_wg(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                             const Scratch &sc, int sm_count, unsigned long long *counters, const int *wl, const int *n_wl,
                             cudaStream_t st)
{
    if (P.algo == BDX_EXACT)
        return launch_wgv<W, G, kShiftAnd, false>(P, pass, seq, off, n, sc, sm_count, counters, wl, n_wl, st);
    return launch_wgv<W, G, kMyers, true>(P, pass, seq, off, n, sc, sm_count, counters, wl, n_wl, st);
}

cudaError_t launch_filter(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                          const Scratch &sc, int sm_count, unsigned long long *counters, const int *wl, const int *n_wl,
                          cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    const DevSet &S = P.set[pass];
    const int groups = S.n_bc_pad / 32;
    const int G = groups >= 4 && groups % 4 == 0 ? 4 : (groups % 3 == 0 ? 3 : (groups % 2 == 0 ? 2 : 1));
#define BDX_CASE(W_, G_) \
    if (S.words == W_ && G == G_) return launch_wg<W_, G_>(P, pass, seq, off, n, sc, sm_count, counters, wl, n_wl, st);
    BDX_CASE(1, 1) BDX_CASE(1, 2) BDX_CASE(1, 3) BDX_CASE(1, 4)
    BDX_CASE(2, 1) BDX_CASE(2, 2) BDX_CASE(2, 3) BDX_CASE(2, 4)
#undef BDX_CASE
    return cudaErrorInvalidValue;
}

// k_prefilter's dynamic shared memory: read staging + hash table (keys, values) + first-level bitmap
size_t prefilter_smem_bytes(const DevSet &S)
{
    return kPfStageBytes + 16 + ((size_t)8 << S.pf_log2) + ((size_t)4 << (S.pf_bm_log2 - 5));
}

// sm_100: 228 KB of shared memory and 2048 threads an SM, 1 KB of it reserved per block
int prefilter_blocks_per_sm(size_t smem)
{
    return (int)std::min<size_t>(2048 / kPfThreads, (size_t)228 * 1024 / (smem + 1024));
}

}  // namespace bdx
