// hamming.cu -- :hamming candidate generation on bit-plane packed reads (classification.jl:557-625).
//
// Setting: one common barcode length m <= 32, at most four distinct barcode bytes, no 'N' in the barcodes
// (an 'N' there is a wildcard, :597), allowed = floor(max_error_rate * m) <= 7.  A placement with at most
// `allowed` mismatches leaves one of allowed + 1 disjoint barcode segments intact (pigeonhole; Hamming
// distance has no shifts, so the segment sits at its own offset).  Per segment a direct-address table maps the
// 2-bit code of the segment's first q bases to the barcodes that carry it.
//   * A warp packs its 32 reads with ballots: per 32 bases three words -- the two bit planes of the 2-bit base
//     code (class - 1) and an "absent from every barcode" plane (such a base mismatches every barcode
//     position, like any other byte the barcodes do not contain; bases past the end of the read are absent).
//   * One thread per read then walks the start positions hamming_align allows (:570-571, :583-586): the m-base
//     window of each plane is one funnel shift, each segment's q-gram is looked up, and every listed barcode
//     is verified with xor / or / popcount on 32-bit words: no byte loop, no early-exit divergence.
//   * Barcodes with a placement within `allowed` form the read's list (ascending), each with its best placement
//     (fewest mismatches; ties leftmost, rightmost when trimming 3', :609-620).
// The list is exactly {b : hamming_align(b) is finite at the initial threshold}; every other barcode returns Inf
// in the reference under any running threshold, and for a listed barcode hamming_align returns that best
// placement whenever it is within the threshold of its turn.  So the reference's sequential selection is
// replayed over the list right here (file order, running threshold, doubles).  Reads longer than the packed
// capacity, or with more than kCandMax acceptable barcodes, are handed to k_literal ("scan every barcode").
#include <algorithm>
#include <cstdlib>
#include <math_constants.h>

#include "bdx_internal.h"
#include "literal.cuh"

namespace bdx {

constexpr int kHpThreads = 256;
constexpr int kHpWords = 6;                  // 32-base words per plane: reads up to 192 bases
constexpr int kHpPlane = kHpWords + 1;       // + one all-absent pad word for the funnel shift

__global__ void __launch_bounds__(kHpThreads)
k_hamming_scan(const __grid_constant__ DevParams P, const int pass, const uint8_t *__restrict__ seq,
               const int *__restrict__ off, const int n_reads, PassOut *__restrict__ out,
               const PassOut *__restrict__ prev_pass, uint16_t *__restrict__ cand, uint8_t *__restrict__ cand_cnt)
{
    extern __shared__ __align__(16) uint32_t smem[];
    const DevSet &S = P.set[pass];
    const HammingPacked &H = S.hp;
    uint32_t *p0_s = smem;                                                    // [kHpPlane][threads] code bit 0
    uint32_t *p1_s = p0_s + kHpPlane * kHpThreads;                            // code bit 1
    uint32_t *pi_s = p1_s + kHpPlane * kHpThreads;                            // absent
    uint2 *bcw_s = reinterpret_cast<uint2 *>(pi_s + kHpPlane * kHpThreads);   // [n_bc] barcode planes
    uint16_t *bstart_s = reinterpret_cast<uint16_t *>(bcw_s + S.n_bc);        // [n_bstart]
    uint16_t *entries_s = bstart_s + ((H.n_bstart + 1) & ~1);                 // [n_seg][n_bc]
    // [kCandMax][threads] barcode << 12 | mismatches << 8 | start of its best placement, ascending barcode
    uint32_t *list_s = reinterpret_cast<uint32_t *>(entries_s + ((H.n_seg * S.n_bc + 1) & ~1));
    uint8_t *class_s = reinterpret_cast<uint8_t *>(list_s + kCandMax * kHpThreads);

    for (int k = threadIdx.x; k < S.n_bc; k += blockDim.x) bcw_s[k] = H.bcw[k];
    for (int k = threadIdx.x; k < H.n_bstart; k += blockDim.x) bstart_s[k] = H.bstart[k];
    for (int k = threadIdx.x; k < H.n_seg * S.n_bc; k += blockDim.x) entries_s[k] = H.entries[k];
    for (int k = threadIdx.x; k < 256; k += blockDim.x) class_s[k] = S.class_of[k];
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int m = H.m, allowed = H.allowed, n_seg = H.n_seg;
    const uint32_t len_mask = m >= 32 ? 0xFFFFFFFFu : ((1u << m) - 1u);
    const bool rightmost = S.trim_side == 3;       // ties between placements: leftmost, rightmost when trimming 3' (:613-619)
    const bool with_delta = P.min_delta != 0.0;
    const int n_groups = (n_reads + kHpThreads - 1) / kHpThreads;

    for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        const int read = grp * kHpThreads + threadIdx.x;
        const bool have = read < n_reads;
        const int base = have ? off[read] : 0;
        const int n = have ? off[read + 1] - base : 0;

        // which start positions hamming_align visits (:570-571) and the end constraint (:583-586); only the
        // columns those placements touch are packed, so a long read with a short search range fits as well
        bool skip = !have, notrun = false, none = false, toolong = false;
        int s_first = 1, s_last = 0;
        if (have) {
            if (pass == 1 && prev_pass[read].bc <= 0) {
                notrun = true;
            } else {
                const Geometry g = pass_geometry(S, n);
                s_first = max(g.start_j, max(1, g.min_end_pos - m + 1));
                s_last = min(min(g.end_j, g.max_start_pos), n - m + 1);
                if (!g.valid || s_last < s_first) none = true;
                else if (s_last - s_first + m > kHpWords * 32) toolong = true;
            }
            skip = notrun || none || toolong;
        }
        const int pbase = skip ? 0 : s_first - 1;                // packed base k = absolute column pbase + k + 1
        const int plen = skip ? 0 : s_last - s_first + m;

        // ---- pack the warp's 32 reads, one after the other: coalesced byte loads, three ballots per 32 bases ----
        __syncwarp();
        for (int r = 0; r < 32; r++) {
            const int rb = __shfl_sync(0xFFFFFFFFu, base + pbase, r);
            const int rn = __shfl_sync(0xFFFFFFFFu, plen, r);
            if (rn == 0) continue;                                // warp-uniform
            const int col = warp * 32 + r;
            uint8_t v[kHpWords];
#pragma unroll
            for (int w = 0; w < kHpWords; w++) v[w] = lane + 32 * w < rn ? seq[rb + lane + 32 * w] : (uint8_t)0;
#pragma unroll
            for (int w = 0; w < kHpWords; w++) {
                const int cls = lane + 32 * w < rn ? (int)class_s[v[w]] : 0;
                const uint32_t b0 = __ballot_sync(0xFFFFFFFFu, ((cls - 1) & 1) != 0);
                const uint32_t b1 = __ballot_sync(0xFFFFFFFFu, ((cls - 1) & 2) != 0);
                const uint32_t bi = __ballot_sync(0xFFFFFFFFu, cls == 0);
                if (lane == 0) {
                    p0_s[w * kHpThreads + col] = b0;
                    p1_s[w * kHpThreads + col] = b1;
                    pi_s[w * kHpThreads + col] = bi;
                }
            }
            if (lane == 0) {
                p0_s[kHpWords * kHpThreads + col] = 0u;
                p1_s[kHpWords * kHpThreads + col] = 0u;
                pi_s[kHpWords * kHpThreads + col] = 0xFFFFFFFFu;
            }
        }
        __syncwarp();

        if (!have) continue;
        if (notrun) {
            out[read] = PassOut{kBcNotRun, 0, -1, -1};
            continue;
        }
        if (none) {
            out[read] = PassOut{kBcUnknown, 0, -1, -1};
            continue;
        }
        if (toolong) {                                 // beyond the packed capacity: k_literal scans every barcode
            cand_cnt[read] = (uint8_t)kCandOverflow;
            out[read] = PassOut{kBcPending, 0, -1, -1};
            continue;
        }

        // ---- every start position: window, per-segment table lookup, popcount verification ----
        int nc = 0;
        const int n_starts = s_last - s_first + 1;
        for (int s = 1; s <= n_starts; s++) {                 // relative start: absolute start = s + pbase
            const int wi = (s - 1) >> 5;
            const uint32_t sh = (uint32_t)(s - 1) & 31u;
            const int i0 = wi * kHpThreads + threadIdx.x, i1 = i0 + kHpThreads;
            const uint32_t W0 = __funnelshift_r(p0_s[i0], p0_s[i1], sh);
            const uint32_t W1 = __funnelshift_r(p1_s[i0], p1_s[i1], sh);
            const uint32_t WI = __funnelshift_r(pi_s[i0], pi_s[i1], sh);
            for (int sg = 0; sg < n_seg; sg++) {
                const int o = H.seg_off[sg], q = H.seg_q[sg];
                const uint32_t qm = (1u << q) - 1u;
                if ((WI >> o) & qm) continue;                            // an absent base cannot be part of an intact seed
                const uint32_t gram = ((W0 >> o) & qm) | (((W1 >> o) & qm) << q);
                const int e1 = bstart_s[H.seg_base[sg] + gram + 1];
                for (int e = bstart_s[H.seg_base[sg] + gram]; e < e1; e++) {
                    const int b = entries_s[sg * S.n_bc + e];
                    const uint2 bw = bcw_s[b];
                    const int mm = __popc(((W0 ^ bw.x) | (W1 ^ bw.y) | WI) & len_mask);
                    if (mm > allowed || nc == kCandOverflow) continue;
                    const uint32_t item = ((uint32_t)b << 12) | ((uint32_t)mm << 8) | (uint32_t)s;
                    int pos = 0;                                         // sorted by barcode
                    while (pos < nc && (int)(list_s[pos * kHpThreads + threadIdx.x] >> 12) < b) pos++;
                    if (pos < nc && (int)(list_s[pos * kHpThreads + threadIdx.x] >> 12) == b) {
                        // the barcode's best placement so far: fewer mismatches win, ties by the start rule
                        const uint32_t old = list_s[pos * kHpThreads + threadIdx.x];
                        const int old_mm = (int)((old >> 8) & 0xFu);
                        if (mm < old_mm || (mm == old_mm && rightmost && s > (int)(old & 0xFFu)))
                            list_s[pos * kHpThreads + threadIdx.x] = item;
                        continue;
                    }
                    if (nc == kCandMax) {
                        nc = kCandOverflow;
                        continue;
                    }
                    for (int k = nc; k > pos; k--) list_s[k * kHpThreads + threadIdx.x] = list_s[(k - 1) * kHpThreads + threadIdx.x];
                    list_s[pos * kHpThreads + threadIdx.x] = item;
                    nc++;
                }
            }
        }
        if (nc == kCandOverflow) {                     // too many acceptable barcodes to list: k_literal scans them all
            cand_cnt[read] = (uint8_t)kCandOverflow;
            out[read] = PassOut{kBcPending, 0, -1, -1};
            continue;
        }
        // ---- the reference's sequential selection over the listed barcodes, in file order, with the running
        // threshold (find_best_matching_bc_*, :632-713).  For a barcode on the list hamming_align returns its
        // best placement when that is within floor(thr * m) at its turn, else Inf; unlisted barcodes return Inf
        // under every threshold. ----
        BestState bs;
        best_init(bs, P.max_error_rate);
        for (int k = 0; k < nc; k++) {
            const uint32_t item = list_s[k * kHpThreads + threadIdx.x];
            const int b = (int)(item >> 12), mm = (int)((item >> 8) & 0xFu), st = (int)(item & 0xFFu) + pbase;
            const bool ok = mm <= allowed_from(bs.thr, m);                                   // :567
            const double score = ok ? __ddiv_rn((double)mm, (double)m) : CUDART_INF;        // :607
            best_consider(bs, with_delta, score, ok ? mm : kInf, b + 1, ok ? st : -1, ok ? st + m - 1 : -1);
        }
        out[read] = best_finish(bs, with_delta, P.min_delta);
    }
}

size_t hamming_scan_smem(const DevSet &S)
{
    const HammingPacked &H = S.hp;
    size_t b = 3 * (size_t)kHpPlane * kHpThreads * 4;
    b += (size_t)S.n_bc * 8;
    b += (size_t)((H.n_bstart + 1) & ~1) * 2 + (size_t)((H.n_seg * S.n_bc + 1) & ~1) * 2;
    b += (size_t)kCandMax * kHpThreads * 4 + 256;
    return (b + 15) & ~(size_t)15;
}

cudaError_t launch_hamming_scan(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                                const Scratch &sc, int sm_count, cudaStream_t st)
{
    const DevSet &S = P.set[pass];
    const size_t smem = hamming_scan_smem(S);
    int blocks = 0;
    cudaError_t e = resident_grid((const void *)k_hamming_scan, kHpThreads, smem, (n + kHpThreads - 1) / kHpThreads,
                                  sm_count, &blocks);
    if (e != cudaSuccess) return e;
    k_hamming_scan<<<blocks, kHpThreads, smem, st>>>(P, pass, seq, off, n, sc.pass[pass], sc.pass[0], sc.cand, sc.cand_cnt);
    return cudaGetLastError();
}

}  // namespace bdx
