// seed_var.cu -- seed-and-verify for the sets and geometries k_seed (seed.cu) does not take: barcodes of
// DIFFERENT lengths, and search geometries with a constrained barcode start or end (barcode_start_range /
// barcode_end_range), where the reference's result for one barcode depends on the running threshold
// (classification.jl:270: the start constraint is enforced through a band whose slack is the current allowed
// distance).  Score-only passes with unit costs; one block works on groups of 128 reads.
//
//   scan    Every barcode b is cut into K_b + 1 disjoint segments of q bases (K_b = min(m_b / q - 1, allowed_b)),
//           all (barcode, segment) q-mers sit in a direct-address table (4^q buckets: at most four distinct
//           barcode bytes).  The q-mer at every column of every staged search range is looked up -- the pairs
//           (read, column) are dealt to the threads of the block, not one read per thread -- and a table entry
//           is a HIT when its diagonal is one an acceptable alignment can lie on: inside the search range,
//           ending at or after min_end_pos, starting no later than max_start_pos + allowed_b (the reference's
//           loose start bound), each widened by K_b.  Position constraints are what keeps short seeds
//           selective here (config 3: 5-mers of 384 barcodes, 25 chance hits per read instead of 55).
//   verify  The block's hits form one list; every thread verifies hits (two at a time) with the windowed
//           Myers / Hyyro automaton of k_seed over the m_b + 2 K_b columns an alignment with that intact
//           segment can occupy.  Pigeonhole: an alignment with <= K_b edits leaves a segment intact, so
//           C = {b : unit distance d_b <= K_b} is found completely and with exact distances; a barcode outside
//           C costs more than K_b edits under ANY threshold (the reference's finite results are costs of real
//           alignments inside the range), i.e. scores at least sigma = min_b (K_b + 1) / m_b.
//   decide  One thread per read replays find_best_matching_bc (classification.jl:632-713) over C in barcode
//           order.  The value of a candidate is d_b / m_b if the reference finds that alignment whatever the
//           running threshold is.  Default geometry: it does (k_filter's exact regime).  Constrained end only:
//           the DP is threshold independent but the last row takes no insertion (:213); the verification tracks
//           D'[m][j] = min(D[m-1][j] + 1, D[m-1][j-1] + sub) then.  Constrained start: sg_literal run with allowed = d_b,
//           the tightest band that can still accept the barcode; if it returns d_b the alignment lies inside
//           every wider band as well (band(a) grows with a, the Ukkonen cut-off is exact for unit costs), so
//           the value is d_b for every threshold >= d_b / m_b and "rejected" below -- which is all the replay
//           needs.  Otherwise the read is left to the exact path.
//           With best score s1 and runner-up s2 among C:  s1 < sigma is required (no unseen barcode can win or
//           tie); without min_delta that decides the read; with min_delta it is ambiguous when s2 - s1 <
//           min_delta (an unseen barcode can only lower the runner-up) and matched when both s2 - s1 and
//           sigma - s1 are >= min_delta.  An unseen barcode accepted in the reference's run lowers the
//           threshold to its score or to a candidate's, never below sigma or the runner-up, so the candidates'
//           verdicts above are unchanged.  Everything else -- no candidate, best too close to sigma, too many
//           hits -- goes on through the worklist to k_filter + k_literal, which are exact for any read.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <math_constants.h>
#include <type_traits>

#include "bdx_internal.h"
#include "literal.cuh"

namespace bdx {

constexpr int kSvThreads = 128;      // threads per block; a block works on groups of R <= 128 reads (SeedVar::group_reads)
constexpr int kSvChains = 2;         // hits a thread verifies at a time (independent dependency chains)
constexpr int kSvCand = 8;           // verified candidates kept per read
constexpr int kSvDiagBias = 64;      // hit record: read << 22 | barcode << 8 | diagonal + bias
constexpr int kSvMaxCols = 180;      // longest search range staged (longer ones take the exact path)
constexpr int kSvBig = 1 << 20;
constexpr int kSvRi = 5;             // ints per read in rinfo: L, min_end_rel, max_start_rel, flags, n_rel

// Stages `my_len` bytes starting at seq + my_start as class codes for each of the warp's 32 reads (lane l
// describes read l) -- seed_stage_warp of seed_common.cuh with a runtime slot stride.
__device__ __forceinline__ void sv_stage_warp(const uint8_t *__restrict__ seq, long long my_start, int my_len,
                                              uint8_t *warp_slots, int stride, const uint8_t *class_s, int lane)
{
    for (int r0 = 0; r0 < 32; r0 += 4) {
        uint32_t w[4][2];
        int mis[4], len[4], nw[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const long long start = __shfl_sync(0xFFFFFFFFu, my_start, r0 + j);
            len[j] = __shfl_sync(0xFFFFFFFFu, my_len, r0 + j);
            const uintptr_t addr = reinterpret_cast<uintptr_t>(seq + start);
            mis[j] = (int)(addr & 3u);
            nw[j] = len[j] ? (mis[j] + len[j] + 3) >> 2 : 0;
            const uint32_t *base = reinterpret_cast<const uint32_t *>(addr - (uintptr_t)mis[j]);
            w[j][0] = lane < nw[j] ? __ldg(base + lane) : 0u;
            w[j][1] = lane + 32 < nw[j] ? __ldg(base + lane + 32) : 0u;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            uint8_t *dst = warp_slots + (size_t)(r0 + j) * stride;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int wi = lane + 32 * h;
                if (wi >= nw[j]) continue;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int idx = 4 * wi + k - mis[j];
                    if (idx >= 0 && idx < len[j]) dst[idx] = class_s[(w[j][h] >> (8 * k)) & 0xFFu];
                }
            }
        }
    }
}

// Shared-memory carve-up (bytes); the same arithmetic on the host (launch) and the device (kernel).
// The block's hit list holds hit_rows rows of kSvThreads records; the decide phase reuses it as sg_literal's DP
// columns [row][thread], max_m + 2 rows (sets whose geometry can bound the start get at least that many: tables.cu).

enum { kSvPeq = 0, kSvHits, kSvCandL, kSvRinfo, kSvCandN, kSvCtr, kSvBinfo, kSvClass, kSvPlanes, kSvBplanes, kSvSlot, kSvParts };

// words of one bit plane of a read's search range (3-gram filter): the columns -32 .. slot_cols + 63, odd so that the
// planes of consecutive reads start in different banks; 0 = no filter
__host__ __device__ inline int sv_plane_words(int slot_cols, int qgram_filter) { return qgram_filter ? ((slot_cols + 32) / 32 + 3) | 1 : 0; }

__host__ __device__ inline size_t sv_smem_layout(int W, int plane, int n_pad,
                                                 int slot_stride, int R, int hit_rows, int pl_words, size_t off[kSvParts])
{
    size_t o = 0;
    off[kSvPeq] = o; o += (size_t)W * plane * 4;                          // Peq, transposed to [word][barcode][class]
    off[kSvHits] = o; o += (size_t)kSvThreads * hit_rows * 4;                     // hit list / DP columns [row][thread]
    off[kSvCandL] = o; o += (size_t)R * kSvCand * 4;                      // verified candidates per read
    off[kSvRinfo] = o; o += (size_t)kSvThreads * kSvRi * 4;               // per read: L, min_end_rel, max_start_rel, flags, n_rel
    off[kSvCandN] = o; o += ((size_t)kSvThreads + 4) * 4;                 // per read: number of candidates; later their offsets
    off[kSvCtr] = o; o += 32;
    off[kSvBinfo] = o; o += (size_t)n_pad * 4;                            // per barcode: m | K << 8 | allowed0 << 16
    off[kSvClass] = o; o += 256;
    off[kSvPlanes] = o; o += (size_t)R * 3 * pl_words * 4;                // per read: bit planes (absent, code bit 0, code bit 1) of the staged range
    o = (o + 7) / 8 * 8;
    off[kSvBplanes] = o; o += pl_words ? (size_t)n_pad * 8 : 0;           // per barcode: code bit 0 / bit 1 of its rows, row i at bit i
    off[kSvSlot] = o; o += (size_t)R * slot_stride + 128;                 // staged class codes (+ slack: windows are read past their end)
    return (o + 15) / 16 * 16;
}

// Windowed Myers / Hyyro verification of the block's hit list, kSvChains hits per thread and round.
// LASTROW: hits are scored as D'[m][j] = min(D[m-1][j] + 1, D[m-1][j-1] + sub) (the reference's last row takes
// no insertion, classification.jl:213) and only at columns >= min_end_pos.
template <typename WT, bool LASTROW>
__device__ __forceinline__ int sv_verify(const uint32_t *hits_s, int total, const int *rinfo_s, const uint32_t *binfo_s,
                                          const uint32_t *peq_s, int n_classes, int plane, const uint8_t *slot_s,
                                          int slot_stride, uint32_t *cand_s, int *cand_n_s, int seg, const int *cnt)
{
    constexpr int kMsb = (int)sizeof(WT) * 8 - 1;
    // seg != 0: the list is four segments of seg records whose first cnt[0..3] are live (sv_qgram_compact)
    const int n0 = seg ? cnt[0] : 0, n1 = seg ? cnt[1] : 0, n2 = seg ? cnt[2] : 0;
    auto fetch = [&](int i) {
        if (seg) {
            int w = 0;
            if (i >= n0) { i -= n0; w = 1; if (i >= n1) { i -= n1; w = 2; if (i >= n2) { i -= n2; w = 3; } } }
            i += w * seg;
        }
        return hits_s[i];
    };
    int cols = 0;                       // window columns this thread stepped its hits over (work counter)
    for (int i0 = 0; i0 < total; i0 += kSvChains * kSvThreads) {
        int score[kSvChains], best[kSvChains], hr[kSvChains], hk[kSvChains], hb[kSvChains], wl[kSvChains], ts[kSvChains];
        WT pv[kSvChains], mv[kSvChains];
        const uint8_t *col[kSvChains];          // first column of the window
        const uint32_t *row[kSvChains];         // the barcode's Peq words, indexed by class
        int wlen = 0;
#pragma unroll
        for (int u = 0; u < kSvChains; u++) {
            const int i = i0 + u * kSvThreads + (int)threadIdx.x;
            const bool live = i < total;
            const uint32_t rec = live ? fetch(i) : 0u;
            hr[u] = live ? (int)(rec >> 22) : 0;
            hb[u] = (int)((rec >> 8) & 0x3FFFu);
            const int delta = (int)(rec & 0xFFu) - kSvDiagBias;
            const uint32_t bi = binfo_s[hb[u]];
            const int m = (int)(bi & 0xFFu);
            hk[u] = live ? (int)((bi >> 8) & 0xFFu) : -1;
            const int Lr = rinfo_s[hr[u] * kSvRi + 0], min_end_rel = rinfo_s[hr[u] * kSvRi + 1];
            // 1-based relative columns an alignment with <= K edits and this segment intact can occupy
            const int c0 = live ? max(1, delta - hk[u] + 1) : 1;
            const int c1 = live ? min(Lr, delta + m + hk[u]) : 0;
            wl[u] = c1 - c0 + 1;
            ts[u] = LASTROW ? max(0, min_end_rel - c0) : 0;            // hits end at or after min_end_pos (:419)
            col[u] = slot_s + (size_t)hr[u] * slot_stride + (c0 - 1);
            row[u] = peq_s + hb[u] * n_classes;
            pv[u] = m > kMsb ? ~(WT)0 : (m <= 0 ? (WT)0 : (~(WT)0 << (kMsb + 1 - m)));   // barcode rows top-aligned
            mv[u] = 0;
            score[u] = m;
            best[u] = kInf;
            wlen = max(wlen, wl[u]);
            cols += max(wl[u], 0);
        }
        wlen = __reduce_max_sync(0xFFFFFFFFu, wlen);
        // past its own window a lane keeps stepping on whatever is staged there (never read back: `best` is frozen)
#pragma unroll 2
        for (int t = 0; t < wlen; t++) {
            WT eq[kSvChains];
#pragma unroll
            for (int u = 0; u < kSvChains; u++) {
                const uint32_t cls = col[u][t];
                eq[u] = row[u][cls];
                if (sizeof(WT) == 8) eq[u] |= (WT)row[u][plane + cls] << (kMsb - 31);
            }
#pragma unroll
            for (int u = 0; u < kSvChains; u++) {
                int up_prev = 0;
                if (LASTROW) up_prev = score[u] - (int)(pv[u] >> kMsb) + (int)(mv[u] >> kMsb);   // D[m-1][j-1]
                const WT xv = eq[u] | mv[u];
                const WT xh = ((((eq[u] & pv[u]) + pv[u]) ^ pv[u]) | eq[u]);
                const WT ph = mv[u] | ~(xh | pv[u]);
                const WT mh = pv[u] & xh;
                score[u] += (int)(ph >> kMsb) - (int)(mh >> kMsb);
                const WT phs = ph << 1, mhs = mh << 1;
                pv[u] = mhs | ~(xv | phs);
                mv[u] = phs & xv;
                int hit_score = score[u];
                if (LASTROW) {
                    const int up = score[u] - (int)(pv[u] >> kMsb) + (int)(mv[u] >> kMsb);        // D[m-1][j]
                    hit_score = min(up + 1, up_prev + 1 - (int)(eq[u] >> kMsb));
                }
                if ((unsigned)(t - ts[u]) < (unsigned)(wl[u] - ts[u])) best[u] = min(best[u], hit_score);
            }
        }
#pragma unroll
        for (int u = 0; u < kSvChains; u++)
            if (hk[u] >= 0 && best[u] <= hk[u]) {
                const int k = atomicAdd(&cand_n_s[hr[u]], 1);
                if (k < kSvCand) cand_s[hr[u] * kSvCand + k] = ((uint32_t)hb[u] << 8) | (uint32_t)best[u];
            }
    }
    return cols;
}

// 3-gram filter between the hit test and the verification (barcodes up to 32 nt over at most four bases).
// An alignment with <= K edits that contains the hit's intact segment on diagonal delta keeps all its cells on the
// diagonals delta - K .. delta + K, and every edit destroys at most three of the barcode's m - 2 overlapping 3-grams;
// so at least (m - 2) - 3 K barcode rows i must see rows i, i + 1, i + 2 matched on ONE of those diagonals.
// Bit-parallel over the rows: the read's range is kept as three bit planes (no-barcode-base, code bit 0, code bit 1;
// columns outside the range count as no-barcode-base), the barcode as two; a diagonal's match vector is
// ~((R0 ^ B0) | (R1 ^ B1) | RA) with the read planes shifted by the diagonal, its 3-gram vector M & M>>1 & M>>2,
// the union over the 2 K + 1 diagonals is counted.  ~10 instructions per diagonal where the automaton steps ~20 per
// window COLUMN (m + 2 K of them), and nine of ten chance hits end here (a random window shares ~6 of a 24-nt
// barcode's 22 3-grams where 10 are needed).  A necessary condition only: whatever passes is verified.
__device__ __forceinline__ bool sv_qgram_pass(const uint32_t *planes_s, int pl_words, const uint2 *bplanes_s, int hr, int b,
                                              int m, int K, int delta)
{
    const int need = (m - 2) - 3 * K;
    if (need <= 0) return true;
    const int biased = delta - K + 32;                      // first diagonal's column of row 0, plane bit index
    const uint32_t *pl = planes_s + (size_t)hr * 3 * pl_words + (biased >> 5);
    const int sh = biased & 31;
    const uint32_t a_lo = __funnelshift_r(pl[0], pl[1], sh), a_hi = __funnelshift_r(pl[1], pl[2], sh);
    pl += pl_words;
    const uint32_t p_lo = __funnelshift_r(pl[0], pl[1], sh), p_hi = __funnelshift_r(pl[1], pl[2], sh);
    pl += pl_words;
    const uint32_t q_lo = __funnelshift_r(pl[0], pl[1], sh), q_hi = __funnelshift_r(pl[1], pl[2], sh);
    const uint2 bp = bplanes_s[b];
    const uint32_t rows = m >= 32 ? 0xFFFFFFFFu : (1u << m) - 1u;
    uint32_t cover = 0;
    for (int k = 0; k <= 2 * K; k++) {                       // 2 K <= 2 (m - 3) / 3 < 31
        const uint32_t mis = (__funnelshift_r(p_lo, p_hi, k) ^ bp.x) | (__funnelshift_r(q_lo, q_hi, k) ^ bp.y) |
                             __funnelshift_r(a_lo, a_hi, k);
        const uint32_t mt = ~mis & rows;
        cover |= mt & (mt >> 1) & (mt >> 2);
    }
    return __popc(cover) >= need;
}

// The same test over the finished hit list (mode 2: geometries whose admissible diagonals are few, where testing inside
// the scan would run it for two or three lanes of a warp at a time).  No block-wide barrier per round: the list is cut
// into one segment per warp, each warp tests its segment 32 hits at a time and compacts the survivors to the
// segment's front (its write cursor never passes its read cursor); cnt[w] = survivors of warp w's segment.
// sv_verify then walks the four segment fronts as one list.  Returns the segment length.
__device__ __forceinline__ int sv_qgram_compact(uint32_t *hits_s, int total, const uint32_t *planes_s, int pl_words,
                                                const uint2 *bplanes_s, const uint32_t *binfo_s, int *cnt, unsigned &n_diag)
{
    static_assert(kSvThreads == 128, "four segments");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int seg = ((total + 3) / 4 + 31) & ~31;
    const int s0 = warp * seg, s1 = min(total, s0 + seg);
    int kept = 0;
    for (int i0 = s0; i0 < s1; i0 += 32) {
        const int i = i0 + lane;
        uint32_t rec = 0;
        bool keep = false;
        if (i < s1) {
            rec = hits_s[i];
            const int b = (int)((rec >> 8) & 0x3FFFu);
            const uint32_t bi = binfo_s[b];
            n_diag += 2u * ((bi >> 8) & 0xFFu) + 1u;
            keep = sv_qgram_pass(planes_s, pl_words, bplanes_s, (int)(rec >> 22), b, (int)(bi & 0xFFu), (int)((bi >> 8) & 0xFFu),
                                 (int)(rec & 0xFFu) - kSvDiagBias);
        }
        const uint32_t km = __ballot_sync(0xFFFFFFFFu, keep);        // (every lane has read its hit by now)
        if (keep) hits_s[s0 + kept + __popc(km & ((1u << lane) - 1u))] = rec;
        kept += __popc(km);
        __syncwarp();
    }
    if (lane == 0) cnt[warp] = kept;
    return seg;
}

template <int W>
__global__ void __launch_bounds__(kSvThreads, 7)
k_seed_var(const __grid_constant__ DevParams P, const int pass, const int level, const uint8_t *__restrict__ seq,
           const int *__restrict__ off, const int n_reads, PassOut *__restrict__ out,
           const PassOut *__restrict__ prev_pass, const int *__restrict__ wl_in, const int *__restrict__ n_in,
           int *__restrict__ wl_out, int *__restrict__ n_out, unsigned long long *__restrict__ counters,
           const int slot_stride, const int slot_cols)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const DevSet &S = P.set[pass];
    const SeedVar &V = S.sv[level];
    const int R = V.group_reads;                             // reads per group: threads 0 .. R-1 own one each
    const int n_pad = S.n_bc_pad;
    const int n_classes = S.n_classes;
    const int plane = n_classes * n_pad;
    size_t lo[kSvParts];
    const int pl_words = sv_plane_words(slot_cols, W == 1 && V.qgram_filter);
    sv_smem_layout(W, plane, n_pad, slot_stride, R, V.hit_rows, pl_words, lo);
    uint32_t *peq_s = reinterpret_cast<uint32_t *>(smem_raw + lo[kSvPeq]);
    uint32_t *hits_s = reinterpret_cast<uint32_t *>(smem_raw + lo[kSvHits]);
    uint32_t *cand_s = reinterpret_cast<uint32_t *>(smem_raw + lo[kSvCandL]);
    int *rinfo_s = reinterpret_cast<int *>(smem_raw + lo[kSvRinfo]);
    int *cand_n_s = reinterpret_cast<int *>(smem_raw + lo[kSvCandN]);
    int *ctr_s = reinterpret_cast<int *>(smem_raw + lo[kSvCtr]);
    // The seed tables (bucket starts + entries, a few KB) stay in global memory, i.e. in L1: copies in shared memory
    // cost one or two resident blocks per SM and measured slower (config 3: 155 -> 173 M reads/s without them)
    const uint32_t *entries_s = V.entries;
    const uint16_t *bstart_s = V.bstart;
    uint32_t *binfo_s = reinterpret_cast<uint32_t *>(smem_raw + lo[kSvBinfo]);
    uint8_t *class_s = smem_raw + lo[kSvClass];
    uint8_t *slot_s = smem_raw + lo[kSvSlot];
    uint32_t *planes_s = reinterpret_cast<uint32_t *>(smem_raw + lo[kSvPlanes]);
    uint2 *bplanes_s = reinterpret_cast<uint2 *>(smem_raw + lo[kSvBplanes]);

    // Peq arrives as [word][class][barcode] (k_filter's lanes read consecutive barcodes); a verifying thread
    // reads ONE barcode's words for changing classes, so it is kept as [word][barcode][class] here
    for (int k = threadIdx.x; k < W * plane; k += blockDim.x) {
        const int w = k / plane, rem = k - w * plane, c = rem / n_pad, b = rem - c * n_pad;
        peq_s[w * plane + b * n_classes + c] = S.peq[k];
    }
    for (int k = threadIdx.x; k < n_pad; k += blockDim.x) {
        uint32_t v = 0;
        if (k < S.n_bc)
            v = (uint32_t)(S.bc_off[k + 1] - S.bc_off[k]) | ((uint32_t)V.kdepth[k] << 8) |
                ((uint32_t)min(max(S.allowed0[k], 0), 255) << 16);
        binfo_s[k] = v;
    }
    for (int k = threadIdx.x; k < 256; k += blockDim.x) class_s[k] = S.class_of[k];
    if (pl_words)                                            // the barcodes' bit planes, row i at bit i (class c = code c - 1)
        for (int k = threadIdx.x; k < n_pad; k += blockDim.x) {
            const int m = k < S.n_bc ? S.bc_off[k + 1] - S.bc_off[k] : 0;
            uint32_t e[5] = {0u, 0u, 0u, 0u, 0u};
            for (int c = 1; c < n_classes && c < 5; c++) e[c] = S.peq[c * n_pad + k];
            const int sh = 32 - m;                           // Peq rows are top-aligned, phantom rows below them
            bplanes_s[k] = m >= 1 && m <= 32 ? make_uint2((e[2] | e[4]) >> sh, (e[3] | e[4]) >> sh) : make_uint2(0u, 0u);
        }
    for (int k = threadIdx.x; k < 128; k += blockDim.x) slot_s[(size_t)R * slot_stride + k] = 0;
    if (threadIdx.x == 0) ctr_s[5] = 0;
    __syncthreads();

    using WT = typename std::conditional<W == 1, uint32_t, unsigned long long>::type;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int n_items = wl_in ? *n_in : n_reads;
    const int n_groups = (n_items + R - 1) / R;
    const bool with_delta = P.min_delta != 0.0;
    const int hit_cap = kSvThreads * V.hit_rows;
    const bool in_scan_filter = pl_words && V.qgram_filter == 1;
    const bool dp_fits = V.hit_rows >= S.max_m + 2;          // sg_literal's column fits the (dead) hit list
    unsigned int n_done = 0;
    unsigned long long n_cols = 0;      // verified hit-columns (one Myers / Hyyro column step each), for the roofline
    unsigned long long n_scan = 0;      // (read, position) pairs scanned (thread 0 counts for the block)
    unsigned n_diag = 0;                // diagonals the 3-gram filter tested

    for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        const int item = grp * R + threadIdx.x;
        const bool have = (int)threadIdx.x < R && item < n_items;
        const int read = have ? (wl_in ? wl_in[item] : item) : 0;
        const int base = have ? off[read] : 0;
        const int n = have ? off[read + 1] - base : 0;

        bool punt = !have;       // true => the read goes on to the exact path (or is not a read at all)
        bool skip = false;       // nothing left to do for this read
        Geometry g{};
        if (have && pass == 1 && prev_pass[read].bc <= 0) {      // classification.jl:879-888
            out[read] = PassOut{kBcNotRun, 0, -1, -1};
            skip = true;
            punt = true;
        }
        if (have && !skip) {
            g = pass_geometry(S, n);
            if (!g.valid) {                                      // :805-807
                out[read] = PassOut{kBcUnknown, 0, -1, -1};
                skip = true;
                punt = true;
            } else if (g.end_j - g.start_j + 1 > slot_cols) {
                punt = true;
            }
        }
        // columns RELATIVE to the search range: relative column c (1-based) is absolute column c + sbase
        const int sbase = punt ? 0 : g.start_j - 1;
        const int L = punt ? 0 : g.end_j - g.start_j + 1;
        rinfo_s[threadIdx.x * kSvRi + 0] = L;
        rinfo_s[threadIdx.x * kSvRi + 1] = punt ? 1 : max(g.min_end_pos - sbase, -kSvBig);
        rinfo_s[threadIdx.x * kSvRi + 2] = punt ? 0 : min(g.max_start_pos - sbase, kSvBig);
        rinfo_s[threadIdx.x * kSvRi + 3] = 0;                        // flags: 1 = hit list overflow, 2 = a candidate is not robust
        rinfo_s[threadIdx.x * kSvRi + 4] = n - sbase;                // read length seen from the range start
        cand_n_s[threadIdx.x] = 0;
        if (threadIdx.x == 0) ctr_s[0] = 0;
        if (L > 0) atomicMax(&ctr_s[5], L);                      // the group's longest search range (reset at the group's end)
        if (warp * 32 < R)
            sv_stage_warp(seq, (long long)base + sbase, L, slot_s + (size_t)warp * 32 * slot_stride, slot_stride, class_s, lane);
        // Constrained end (min_end_pos inside the range): the reference's last row takes no insertion
        // (classification.jl:213), so a hit at column j is D'[m][j] = min(D[m-1][j] + 1, D[m-1][j-1] + sub), not
        // the automaton's D[m][j].  Over ALL columns the two have the same minimum, over the columns
        // >= min_end_pos they do not; D' is tracked for the whole group when any of its reads needs it.
        const int last_row_rule = __syncthreads_or(!punt && g.min_end_pos > g.start_j);
        if (pl_words) {
            // the staged ranges as bit planes, 32 columns per ballot; plane bit 32 + c is relative column c (0-based)
            for (int r = warp; r < R; r += kSvThreads / 32) {
                const int Lr = rinfo_s[r * kSvRi + 0];
                uint32_t *pl = planes_s + (size_t)r * 3 * pl_words;
                for (int w = 0; w < pl_words; w++) {
                    const int c = (w - 1) * 32 + lane;
                    uint32_t a = 0xFFFFFFFFu, b0 = 0u, b1 = 0u;
                    if (w >= 1 && (w - 1) * 32 < Lr) {
                        const uint32_t cls = c < Lr ? slot_s[(size_t)r * slot_stride + c] : 0u;
                        a = __ballot_sync(0xFFFFFFFFu, cls == 0u);
                        b0 = __ballot_sync(0xFFFFFFFFu, cls != 0u && ((cls - 1u) & 1u));
                        b1 = __ballot_sync(0xFFFFFFFFu, cls != 0u && ((cls - 1u) & 2u));
                    }
                    if (lane == 0) {
                        pl[w] = a;
                        pl[pl_words + w] = b0;
                        pl[2 * pl_words + w] = b1;
                    }
                }
            }
            __syncthreads();
        }

        // ---- scan: (read, column) pairs dealt to the lanes, two consecutive pairs each.  A pair looks its q-mer up
        // in table 0 and, with one more base, its (q + 1)-mer in table 1; the entries of a warp's 64 pairs are
        // pooled (prefix sum of the bucket sizes) and dealt out evenly again, one entry per lane and round ----
        {
            const int q0 = V.q, q1 = V.q2;                               // q1 = 0: one table
            const uint16_t *bst0 = bstart_s, *bst1 = bstart_s + V.bstart2;
            const int n_pos = max(ctr_s[5] - q0 + 1, 0);                 // positions of the group's longest search range
            const uint32_t pos_recip = 0xFFFFFFFFu / (uint32_t)max(n_pos, 1) + 1u;   // i / n_pos == umulhi(i, recip) for i < 2^16
            const int n_pairs = R * n_pos;
            if (threadIdx.x == 0) n_scan += (unsigned)n_pairs;
            for (int base = warp * 64; base < n_pairs; base += (kSvThreads / 32) * 64) {
                uint32_t ea = 0, eb = 0, c4 = 0;   // first entries of (pair 0: table 0 | table 1 << 16), (pair 1: ...); the four bucket sizes, a byte each
                int lane_total = 0;
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int i = base + 2 * lane + u;
                    uint32_t e00 = 0, c00 = 0, e01 = 0, c01 = 0;
                    if (i < n_pairs) {
                        const int r = min((int)__umulhi((uint32_t)i, pos_recip), R - 1), p = i - r * n_pos;
                        const int Lr = rinfo_s[r * kSvRi + 0];
                        if (p + q0 <= Lr) {
                            const uint8_t *c = slot_s + (size_t)r * slot_stride + p;
                            uint32_t code = 0;
                            bool ok = true;
                            for (int k = 0; k < q0; k++) {
                                const uint32_t cl = c[k];
                                ok = ok && cl != 0;                       // a byte that occurs in no barcode: no seed here
                                code |= ((cl - 1u) & 3u) << (2 * k);
                            }
                            if (ok) {
                                e00 = bst0[code];
                                c00 = bst0[code + 1] - e00;
                                if (q1 && p + q1 <= Lr && c[q0] != 0) {
                                    const uint32_t code1 = code | ((((uint32_t)c[q0] - 1u) & 3u) << (2 * q0));
                                    e01 = bst1[code1];
                                    c01 = bst1[code1 + 1] - e01;
                                }
                            }
                        }
                    }
                    if (u == 0) ea = e00 | (e01 << 16);
                    else eb = e00 | (e01 << 16);
                    c4 |= (c00 | (c01 << 8)) << (16 * u);
                    lane_total += (int)(c00 + c01);
                }
                int incl = lane_total;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if (lane >= o) incl += t;
                }
                const int total_e = __shfl_sync(0xFFFFFFFFu, incl, 31);
                const int my_excl = incl - lane_total;
                for (int j0 = 0; j0 < total_e; j0 += 32) {
                    const int j = j0 + lane;
                    int ow = 0;                                            // owner = first lane whose inclusive prefix exceeds j
#pragma unroll
                    for (int step = 16; step >= 1; step >>= 1) {
                        const int probe = __shfl_sync(0xFFFFFFFFu, incl, ow + step - 1);
                        if (probe <= j) ow += step;
                    }
                    ow = min(ow, 31);
                    const int o_excl = __shfl_sync(0xFFFFFFFFu, my_excl, ow);
                    const uint32_t oc4 = __shfl_sync(0xFFFFFFFFu, c4, ow);
                    const uint32_t oea = __shfl_sync(0xFFFFFFFFu, ea, ow), oeb = __shfl_sync(0xFFFFFFFFu, eb, ow);
                    bool hit = false;
                    uint32_t rec = 0;
                    int hr = 0;
                    if (j < total_e) {
                        // which of the owner's four buckets, and which entry of it
                        int jj = j - o_excl, which = 0;
                        const int n0 = (int)(oc4 & 0xFFu), n1 = (int)((oc4 >> 8) & 0xFFu), n2 = (int)((oc4 >> 16) & 0xFFu);
                        if (jj >= n0) { jj -= n0; which = 1; if (jj >= n1) { jj -= n1; which = 2; if (jj >= n2) { jj -= n2; which = 3; } } }
                        const uint32_t esel = which < 2 ? oea : oeb;
                        const int e0 = (int)((which & 1) ? (esel >> 16) : (esel & 0xFFFFu));
                        const int oi = base + 2 * ow + (which >> 1);                // the owner's (read, column) pair
                        hr = min((int)__umulhi((uint32_t)oi, pos_recip), R - 1);
                        const int op = oi - hr * n_pos;
                        const uint32_t ent = entries_s[e0 + jj];
                        const int b = (int)(ent >> 8), o = (int)(ent & 0xFFu);
                        const uint32_t bi = binfo_s[b];
                        const int m = (int)(bi & 0xFFu), K = (int)((bi >> 8) & 0xFFu), a0 = (int)(bi >> 16);
                        const int oL = rinfo_s[hr * kSvRi + 0], min_end_rel = rinfo_s[hr * kSvRi + 1], max_start_rel = rinfo_s[hr * kSvRi + 2];
                        const int delta = op - o;                                   // 0-based relative diagonal
                        // Diagonals (read column - barcode row) an acceptable alignment's intact segment can lie on:
                        // the segment's own cells obey the reference's band j - i <= max_start_pos + steps
                        // (classification.jl:270, :289-290; steps <= allowed_b); the rest of the barcode has to fit
                        // between the range start and end with at most K edits, and to end at or after min_end_pos
                        const int dlo = max(0, min_end_rel - m) - K;
                        const int dhi = min(max_start_rel + a0, oL - m + K);
                        hit = delta >= dlo && delta <= dhi;
                        if (hit && in_scan_filter) {
                            n_diag += 2u * (unsigned)K + 1u;
                            hit = sv_qgram_pass(planes_s, pl_words, bplanes_s, hr, b, m, K, delta);
                        }
                        rec = ((uint32_t)hr << 22) | ((uint32_t)b << 8) | (uint32_t)(delta + kSvDiagBias);
                    }
                    const uint32_t hm = __ballot_sync(0xFFFFFFFFu, hit);
                    if (hm) {
                        int hbase = 0;
                        if (lane == 0) hbase = atomicAdd(&ctr_s[0], __popc(hm));
                        hbase = __shfl_sync(0xFFFFFFFFu, hbase, 0);
                        if (hit) {
                            const int idx = hbase + __popc(hm & ((1u << lane) - 1u));
                            if (idx < hit_cap) hits_s[idx] = rec;
                            else rinfo_s[hr * kSvRi + 3] = 1;                       // this read's candidate set is incomplete
                        }
                    }
                }
            }
        }
        __syncthreads();

        // ---- verify: every thread takes hits of the block's list, two at a time ----
        {
            int total = min(ctr_s[0], hit_cap), seg = 0;
            if (pl_words && !in_scan_filter) {
                seg = sv_qgram_compact(hits_s, total, planes_s, pl_words, bplanes_s, binfo_s, ctr_s + 1, n_diag);
                __syncthreads();
                total = ctr_s[1] + ctr_s[2] + ctr_s[3] + ctr_s[4];
            }
            if (last_row_rule)
                n_cols += sv_verify<WT, true>(hits_s, total, rinfo_s, binfo_s, peq_s, n_classes, plane, slot_s, slot_stride, cand_s, cand_n_s, seg, ctr_s + 1);
            else
                n_cols += sv_verify<WT, false>(hits_s, total, rinfo_s, binfo_s, peq_s, n_classes, plane, slot_s, slot_stride, cand_s, cand_n_s, seg, ctr_s + 1);
        }
        __syncthreads();

        // ---- decide ----
        // Constrained start: every candidate is re-aligned by sg_literal in the tightest band that can still accept
        // it (allowed = d); found there => found in every wider band, i.e. its value does not depend on the running
        // threshold.  One thread per CANDIDATE (the reads' lists are flattened by a prefix sum): a group of few
        // reads would otherwise leave most of the block idle.
        const bool usable = !punt && rinfo_s[threadIdx.x * kSvRi + 3] == 0 && cand_n_s[threadIdx.x] <= kSvCand;
        // the read's verified candidates, ascending by (barcode, distance), one record per barcode: several intact
        // segments of one alignment are several hits of the same barcode
        int my_nc = 0;
        uint32_t cl[kSvCand];
        if (usable) {
            const int nc = cand_n_s[threadIdx.x];
#pragma unroll
            for (int k = 0; k < kSvCand; k++) cl[k] = k < nc ? cand_s[threadIdx.x * kSvCand + k] : 0xFFFFFFFFu;
#pragma unroll
            for (int a = 1; a < kSvCand; a++)
#pragma unroll
                for (int bq = a; bq > 0; bq--)
                    if (cl[bq] < cl[bq - 1]) {
                        const uint32_t t = cl[bq];
                        cl[bq] = cl[bq - 1];
                        cl[bq - 1] = t;
                    }
            uint32_t last = 0xFFFFFFFFu;
#pragma unroll
            for (int k = 0; k < kSvCand; k++)
                if (k < nc && (cl[k] >> 8) != last) {                 // the smaller distance of a barcode came first
                    last = cl[k] >> 8;
                    cand_s[threadIdx.x * kSvCand + my_nc++] = cl[k];
                }
        }
        const bool start_bound = !punt && g.max_start_pos < n;      // the reference's result depends on the threshold
        if (__syncthreads_or(start_bound && my_nc > 0)) {
            const Costs c{P.match, P.mismatch, P.indel, P.nindel, P.has_n};
            // DP column of sg_literal: element i of this thread at hits_s[i * kSvThreads + thread] (the hit list is dead now)
            const WsCol DP{reinterpret_cast<int *>(hits_s) + threadIdx.x, kSvThreads};
            auto check = [&](int r, int k) {
                const uint32_t rec = cand_s[r * kSvCand + k];
                const int b = (int)(rec >> 8), d = (int)(rec & 0xFFu);
                if (!dp_fits) {                                                // (never sized that way; the read takes the exact path)
                    rinfo_s[r * kSvRi + 3] = 2;
                    return;
                }
                const int qo = S.bc_off[b], m = S.bc_off[b + 1] - qo;
                // the owner's geometry in RELATIVE columns, as it left it in shared memory (sg_literal's column
                // arithmetic is translation invariant: range, max_start_pos, min_end_pos and n all shift by sbase)
                const int Lr = rinfo_s[r * kSvRi + 0], min_end_rel = rinfo_s[r * kSvRi + 1], max_start_rel = rinfo_s[r * kSvRi + 2];
                const int n_rel = rinfo_s[r * kSvRi + 4];
                const uint8_t *r1 = slot_s + (size_t)r * slot_stride - 1;     // relative column j at r1[j]
                int s_, e_;
                const int dl = sg_literal<false>(DP, DP, S.bc_cls + qo - 1, r1, m, n_rel, d, c, 0, 1, Lr, max_start_rel,
                                                 min_end_rel, s_, e_);
                if (dl != d) rinfo_s[r * kSvRi + 3] = 2;                       // not robust: the read takes the exact path
            };
            if (R > 64) {
                // a full group: most reads have exactly one candidate, a thread checks its own read's
                if (start_bound)
                    for (int k = 0; k < my_nc; k++) check(threadIdx.x, k);
            } else {
                // exclusive offsets of the reads' candidate lists (only reads with a constrained start take part)
                const int cnt = start_bound ? my_nc : 0;
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if (lane >= o) incl += t;
                }
                static_assert(kSvThreads == 128, "four warp totals in ctr_s[1..4]");
                if (lane == 31) ctr_s[1 + warp] = incl;
                __syncthreads();
                int warp_off = 0;
                for (int w = 0; w < warp; w++) warp_off += ctr_s[1 + w];
                int *coff_s = cand_n_s;                                // counts become exclusive offsets
                const int total_c = ctr_s[1] + ctr_s[2] + ctr_s[3] + ctr_s[4];
                coff_s[threadIdx.x] = warp_off + incl - cnt;
                __syncthreads();
                for (int j = threadIdx.x; j < total_c; j += kSvThreads) {
                    int lo_r = 0, hi_r = kSvThreads - 1;               // owner read: last r with coff[r] <= j
                    while (lo_r < hi_r) {
                        const int mid = (lo_r + hi_r + 1) >> 1;
                        if (coff_s[mid] <= j) lo_r = mid;
                        else hi_r = mid - 1;
                    }
                    check(lo_r, j - coff_s[lo_r]);
                }
                __syncthreads();
                cand_n_s[threadIdx.x] = my_nc;                         // (the offsets are not needed any more)
            }
            __syncthreads();
        }
        bool resolved = false;
        if (usable && rinfo_s[threadIdx.x * kSvRi + 3] == 0) {
            const int nc = my_nc;
            BestState bs;
            best_init(bs, P.max_error_rate);
#pragma unroll 1
            for (int k = 0; k < nc; k++) {
                const uint32_t rec = cand_s[threadIdx.x * kSvCand + k];
                const int b = (int)(rec >> 8), d = (int)(rec & 0xFFu);
                const int norm = S.norm[b];
                const int allowed = allowed_from(bs.thr, norm);       // :254 with the running threshold
                const double sc = d <= allowed ? __ddiv_rn((double)d, (double)norm) : CUDART_INF;
                best_consider(bs, with_delta, sc, d, b + 1, -1, -1);
            }
            if (V.complete) {
                out[read] = best_finish(bs, with_delta, P.min_delta);
                resolved = true;
            } else if (bs.min_bc != 0 && bs.min_score < V.sigma_min) {
                if (!with_delta) {
                    out[read] = best_finish(bs, false, 0.0);
                    resolved = true;
                } else if (__dsub_rn(bs.sub_min, bs.min_score) < P.min_delta) {
                    out[read] = PassOut{kBcAmbiguous, 0, -1, -1};
                    resolved = true;
                } else if (__dsub_rn(V.sigma_min, bs.min_score) >= P.min_delta) {
                    out[read] = PassOut{bs.min_bc, bs.min_dist, -1, -1};
                    resolved = true;
                }
            }
        }
        const bool todo = have && !resolved && !skip;
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, todo);
        int base_slot = 0;
        if (lane == 0 && mask) base_slot = atomicAdd(n_out, __popc(mask));
        base_slot = __shfl_sync(0xFFFFFFFFu, base_slot, 0);
        if (todo) wl_out[base_slot + __popc(mask & ((1u << lane) - 1u))] = read;
        n_done += __popc(__ballot_sync(0xFFFFFFFFu, resolved));
        if (threadIdx.x == 0) ctr_s[5] = 0;
        __syncthreads();                                             // the group's shared lists are reused
    }
    if (lane == 0 && n_done && counters) atomicAdd(counters + 2, (unsigned long long)n_done);
    if (counters) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) n_cols += __shfl_down_sync(0xFFFFFFFFu, n_cols, o);
        if (lane == 0 && n_cols) atomicAdd(counters + 3, n_cols);
        unsigned long long nd = n_diag;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) nd += __shfl_down_sync(0xFFFFFFFFu, nd, o);
        if (lane == 0 && nd) atomicAdd(counters + 8, nd);
        if (threadIdx.x == 0 && n_scan) atomicAdd(counters + 7, n_scan);
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(counters + 4, (unsigned long long)n_items);
    }
}

// longest search range any read can have (columns), or kSvMaxCols when it grows with the read
static int sv_slot_cols(const DevSet &S)
{
    const DevRange &r = S.rs;
    if (r.start_from_end == r.end_from_end) {
        const long long len = (long long)r.end_off - r.start_off + 1;
        if (len >= 1 && len <= kSvMaxCols) return (int)len;
        if (len < 1) return 1;
    }
    return kSvMaxCols;
}

struct SvLaunch {
    int slot_cols, slot_stride;
    size_t smem;
};

static SvLaunch sv_launch_params(const DevSet &S, const SeedVar &V)
{
    SvLaunch L;
    L.slot_cols = sv_slot_cols(S);
    int words = (L.slot_cols + 3) / 4;
    words |= 1;                                   // odd word stride: the slots of consecutive reads start in different banks
    L.slot_stride = words * 4;
    size_t off[kSvParts];
    const int plane = S.n_classes * S.n_bc_pad;
    L.smem = sv_smem_layout(S.words, plane, S.n_bc_pad, L.slot_stride, V.group_reads, V.hit_rows,
                            sv_plane_words(L.slot_cols, S.words == 1 && V.qgram_filter), off);
    return L;
}

size_t seed_var_smem(const DevSet &S, const SeedVar &V) { return sv_launch_params(S, V).smem; }

cudaError_t launch_seed_var(const DevParams &P, int pass, int level, const uint8_t *seq, const int *off, int n, const Scratch &sc,
                            const int *wl_in, const int *n_in, int *wl_out, int *n_out, int sm_count,
                            unsigned long long *counters, cudaStream_t st)
{
    const DevSet &S = P.set[pass];
    const SeedVar &V = S.sv[level];
    const SvLaunch L = sv_launch_params(S, V);
    auto kern = S.words == 1 ? k_seed_var<1> : k_seed_var<2>;
    int per_sm = 0;
    cudaError_t e = blocks_per_sm_cached((const void *)kern, kSvThreads, L.smem, &per_sm);
    if (e != cudaSuccess) return e;
    const int groups = (n + V.group_reads - 1) / V.group_reads;
    const int blocks = std::max(1, std::min(groups, sm_count * per_sm));
    e = cudaMemsetAsync(n_out, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    kern<<<blocks, kSvThreads, L.smem, st>>>(P, pass, level, seq, off, n, sc.pass[pass], sc.pass[0], wl_in, n_in, wl_out, n_out,
                                             counters, L.slot_stride, L.slot_cols);
    return cudaGetLastError();
}

}  // namespace bdx
