// seed_deep.cu -- the deepest seed level: reads whose best barcode sits at (or near) the allowed distance, and
// the proof that a read has no acceptable barcode at all.
//
// k_seed's levels stop where seeds of ONE length per level stay selective (<= 0.12 chance hits per column).
// This kernel goes to depth K_D (the allowed distance when the set is small enough) by
//   * cutting the barcode into K_D + 1 segments of m / (K_D + 1) bases, the first m % (K_D + 1) of them one base
//     longer, and hashing each with its own length -- two tables (e.g. 24 nt, K_D = 4: four 5-mers and one 4-mer
//     per barcode, 0.75 chance hits per read column for 96 barcodes instead of 1.9 with 4-mers only);
//   * walking the read in chunks of 16 columns, so that the per-thread win / hit buffers stay small although a
//     read now has ~100 hits: scan a chunk (both rolling hashes), resolve its hits, verify them pooled over the
//     warp (seed_verify, as in k_seed), fold the verified distances into the read's running best.
// It pays while the hits stay rare (bdx_config_create enables it up to 0.25 chance hits per column: small sets
// such as a single adapter, whose alternative is k_literal over the whole range); for 96 x 24 nt at depth 4 it
// measured slower than k_filter and stays off.
// Regime and exactness argument are k_seed's (seed.cu): every alignment with <= K_D edits leaves one of the
// K_D + 1 segments intact, its window is verified, so {b : d_b <= K_D} and those distances are exact.  Without
// min_delta the answer is the lowest index among the minimal d_b; if nothing is within K_D >= allowed no barcode
// is acceptable.  Used for min_delta = 0 only; reads it cannot finish go on to k_filter.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <math_constants.h>

#include "bdx_internal.h"
#include "literal.cuh"
#include "seed_common.cuh"

namespace bdx {

constexpr int kDeepChunk = 16;      // read columns per chunk: at most 2 * 16 bitmap hits -> kSeedMaxWins

struct DeepTab {                    // one seed table in shared (or global) memory
    const uint32_t *bitmap, *bstart, *entries, *ekeys;
    int q, log2, bm_log2;
    uint32_t pow;
};

template <int W>
__global__ void __launch_bounds__(kSeedThreads)
k_seed_deep(const __grid_constant__ DevParams P, const int pass, const uint8_t *__restrict__ seq,
            const int *__restrict__ off, PassOut *__restrict__ out, const PassOut *__restrict__ prev_pass,
            const int *__restrict__ worklist, const int *__restrict__ n_work, int *__restrict__ worklist2,
            int *__restrict__ n_work2, unsigned long long *__restrict__ counters, uint16_t *__restrict__ cand,
            uint8_t *__restrict__ cand_cnt, int *__restrict__ wl_win, int *__restrict__ n_win)
{
    extern __shared__ __align__(16) uint32_t smem[];
    const DevSet &S = P.set[pass];
    const bool need_tb = S.trim_side != 0 || P.want_stats;
    const int n_pad = S.n_bc_pad;
    const int plane = S.n_classes * n_pad;
    uint32_t *peq_s = smem;                                     // [W][n_classes][n_pad]
    uint32_t *cur = peq_s + W * plane;
    for (int k = threadIdx.x; k < W * plane; k += blockDim.x) peq_s[k] = S.peq[k];
    DeepTab tab[2];
    const int n_tabs = S.sdd_n;
#pragma unroll
    for (int t = 0; t < 2; t++) {
        const SeedLevel &SL = S.sdd[t < n_tabs ? t : 0];
        const int n_buckets = 1 << SL.log2, bm_words = 1 << (SL.bm_log2 - 5);
        uint32_t *bm = cur, *bs = bm + bm_words, *en = bs + n_buckets + 1, *ek = en + SL.n_entries;
        if (t < n_tabs) {
            for (int k = threadIdx.x; k < bm_words; k += blockDim.x) bm[k] = SL.bitmap[k];
            for (int k = threadIdx.x; k <= n_buckets; k += blockDim.x) bs[k] = SL.bstart[k];
            for (int k = threadIdx.x; k < SL.n_entries; k += blockDim.x) {
                en[k] = SL.entries[k];
                ek[k] = SL.ekeys[k];
            }
            cur = ek + SL.n_entries;
        }
        tab[t] = DeepTab{bm, bs, en, ek, SL.q, SL.log2, SL.bm_log2, SL.pow};
    }
    uint32_t *hits_s = cur;                                                    // [kSeedMaxHits][kSeedThreads]
    uint16_t *wins_s = reinterpret_cast<uint16_t *>(hits_s + kSeedMaxHits * kSeedThreads);   // [kSeedMaxWins][threads]
    uint8_t *class_s = reinterpret_cast<uint8_t *>(wins_s + kSeedMaxWins * kSeedThreads);
    uint8_t *slot_s = class_s + 256;                                           // [kSeedThreads][kSeedSlot]
    for (int k = threadIdx.x; k < 256; k += blockDim.x) class_s[k] = S.class_of[k];
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int m = S.sd_m, K = S.sdd_k;
    const int n_items = *n_work;
    const int n_groups = (n_items + kSeedThreads - 1) / kSeedThreads;
    unsigned int n_done = 0;
    using WT = typename std::conditional<W == 1, uint32_t, unsigned long long>::type;

    for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        const int item = grp * kSeedThreads + threadIdx.x;
        const bool have = item < n_items;
        const int read = have ? worklist[item] : 0;
        const int base = have ? off[read] : 0;
        const int n = have ? off[read + 1] - base : 0;

        bool punt = !have, skip = false;
        Geometry g{};
        if (have && pass == 1 && prev_pass[read].bc <= 0) {      // classification.jl:879-888
            out[read] = PassOut{kBcNotRun, 0, -1, -1};
            skip = true;
            punt = true;
        }
        if (have && !skip) {
            g = pass_geometry(S, n);
            if (!(g.valid && g.max_start_pos >= n && g.min_end_pos <= g.start_j) || g.end_j - g.start_j + 1 > kSeedSlot - 3)
                punt = true;
        }
        // columns relative to the search range, as in k_seed
        const int sbase = punt ? 0 : g.start_j - 1;
        const int L = punt ? 0 : g.end_j - g.start_j + 1;

        const int skew = seed_slot_skew(seq, (long long)base + sbase);          // the slot keeps the source alignment
        uint8_t *my_slot = slot_s + (size_t)threadIdx.x * kSeedSlot + skew;
        __syncwarp();
        seed_stage_warp(seq, (long long)base + sbase, L, slot_s + (size_t)warp * 32 * kSeedSlot, class_s, lane);
        __syncwarp();

        // rolling hashes of both tables, carried from chunk to chunk; h[t] is the hash of the q-mer at column `p`
        uint32_t h[2] = {0u, 0u};
#pragma unroll
        for (int t = 0; t < 2; t++)
            if (t < n_tabs && !punt && L >= tab[t].q)
                for (int i = 0; i < tab[t].q; i++) h[t] = h[t] * kPfBase + (uint32_t)my_slot[i];

        int best_d = kInf, best_b = 0x7FFFFFFF, w_lo = 0x7FFFFFFF, w_hi = 0;
        const int my_cols = punt ? 0 : L;
        const int max_cols = __reduce_max_sync(0xFFFFFFFFu, my_cols);
        for (int c0 = 0; c0 < max_cols; c0 += kDeepChunk) {
            // ---- phase 1: the chunk's columns whose q-mer passes a table's bitmap ----
            int n_wins = 0;
            if (!punt) {
                const int c1 = min(c0 + kDeepChunk, L);
                for (int p = c0; p < c1; p++) {
#pragma unroll
                    for (int t = 0; t < 2; t++) {
                        if (t >= n_tabs || p + tab[t].q > L) continue;
                        const uint32_t bit = pf_bit(h[t], tab[t].bm_log2);
                        if ((tab[t].bitmap[bit >> 5] >> (bit & 31)) & 1u) {
                            if (n_wins < kSeedMaxWins) wins_s[n_wins * kSeedThreads + threadIdx.x] = (uint16_t)(p | (t << 8));
                            n_wins++;
                        }
                        if (p + tab[t].q < L)       // roll on to column p + 1
                            h[t] = (h[t] - (uint32_t)my_slot[p] * tab[t].pow) * kPfBase + (uint32_t)my_slot[p + tab[t].q];
                    }
                }
                if (n_wins > kSeedMaxWins) punt = true;
            }
            // ---- phase 2 (lock step): bucket walk, key check, (barcode, diagonal) hits of this chunk ----
            int n_hits = 0;
            {
                const int my_wins = punt ? 0 : n_wins;
                const int max_wins = __reduce_max_sync(0xFFFFFFFFu, my_wins);
                for (int k = 0; k < max_wins; k++) {
                    if (k >= my_wins) continue;
                    const int wv = wins_s[k * kSeedThreads + threadIdx.x];
                    const int p = wv & 0xFF, t = wv >> 8;
                    const DeepTab &T = tab[t];
                    uint32_t hh = 0;
                    for (int i = 0; i < T.q; i++) hh = hh * kPfBase + (uint32_t)my_slot[p + i];
                    const uint32_t bucket = pf_slot(hh, T.log2);
                    const uint32_t e1 = T.bstart[bucket + 1];
                    for (uint32_t e = T.bstart[bucket]; e < e1; e++) {
                        if (T.ekeys[e] != hh) continue;
                        const uint32_t ent = T.entries[e];
                        const int delta = p - (int)(ent & 0xFFu);
                        const uint32_t b = ent >> 8;
                        bool merged = false;
                        const int have_hits = min(n_hits, kSeedMaxHits);
                        for (int j = 0; j < have_hits && !merged; j++) {
                            const uint32_t old = hits_s[j * kSeedThreads + threadIdx.x];
                            if ((old >> 13) != b) continue;
                            const int dmin = (int)(old & 0x3FFu) - 256, span = (int)((old >> 10) & 0x7u);
                            const int lo = min(dmin, delta), hi = max(dmin + span, delta);
                            if (hi - lo <= K) {
                                hits_s[j * kSeedThreads + threadIdx.x] = hit_pack(b, hi - lo, lo);
                                merged = true;
                            }
                        }
                        if (merged) continue;
                        if (n_hits < kSeedMaxHits) hits_s[n_hits * kSeedThreads + threadIdx.x] = hit_pack(b, 0, delta);
                        n_hits++;
                    }
                }
                if (n_hits > kSeedMaxHits) punt = true;
            }
            // ---- verify the chunk's hits, pooled over the warp ----
            const int my_hits = punt ? 0 : n_hits;
            int incl = my_hits;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += t;
            }
            const int total_hits = __shfl_sync(0xFFFFFFFFu, incl, 31);
            __syncwarp();
            {
                const SeedVerifyCtx vc{hits_s + warp * 32, peq_s, slot_s + (size_t)warp * 32 * kSeedSlot, n_pad, plane, m, K,
                                       m + 4 * K + 1, total_hits};
                int i0 = 0;
                for (; i0 + 32 < total_hits; i0 += 64) seed_verify<2, WT>(vc, i0, lane, incl, 1, L, skew);
                if (i0 < total_hits) seed_verify<1, WT>(vc, i0, lane, incl, 1, L, skew);
            }
            __syncwarp();
            // ---- fold into the read's running best (smallest distance, lowest index among equals) and the
            // columns that hold its best alignments ----
            for (int k = 0; k < my_hits; k++) {
                const uint32_t rec = hits_s[k * kSeedThreads + threadIdx.x];
                const int d = (int)((rec >> 27) & 0xFu), b = (int)((rec >> 13) & 0x3FFFu);
                if (d > K) continue;
                const int dmin = (int)(rec & 0x3FFu) - 256, span = (int)((rec >> 10) & 0x7u);
                const int lo = dmin + 1 - K, hi = dmin + span + m + 2 * K;
                if (d < best_d || (d == best_d && b < best_b)) {
                    best_d = d;
                    best_b = b;
                    w_lo = lo;
                    w_hi = hi;
                } else if (d == best_d && b == best_b) {
                    w_lo = min(w_lo, lo);
                    w_hi = max(w_hi, hi);
                }
            }
            __syncwarp();
        }

        // ---- decide (as k_seed without min_delta) ----
        bool resolved = false, queued = false;
        if (!punt) {
            if (best_d <= K) {
                const int norm = S.norm[best_b];
                const double sc = __ddiv_rn((double)best_d, (double)norm);
                if (best_d <= allowed_from(P.max_error_rate, norm) && sc <= P.max_error_rate) {
                    if (need_tb) {
                        const int a_lo = max(w_lo - 2 + sbase, 1), a_hi = min(w_hi + 2 + sbase, n);   // absolute columns
                        cand[(size_t)read * kCandMax] = (uint16_t)best_b;
                        cand[(size_t)read * kCandMax + 1] = (uint16_t)a_lo;
                        cand[(size_t)read * kCandMax + 2] = (uint16_t)a_hi;
                        cand_cnt[read] = (uint8_t)(a_hi <= 65535 ? kCandWindow : 1);
                        out[read] = PassOut{kBcPending, 0, -1, -1};
                        queued = true;
                    } else {
                        out[read] = PassOut{best_b + 1, best_d, -1, -1};
                    }
                    resolved = true;
                }
            } else if (K >= S.allowed0[0]) {
                out[read] = PassOut{kBcUnknown, 0, -1, -1};    // nothing within the allowed distance
                resolved = true;
            }
        }
        {
            const uint32_t qm = __ballot_sync(0xFFFFFFFFu, queued);
            int qb = 0;
            if (lane == 0 && qm) qb = atomicAdd(n_win, __popc(qm));
            qb = __shfl_sync(0xFFFFFFFFu, qb, 0);
            if (queued) wl_win[qb + __popc(qm & ((1u << lane) - 1u))] = read;
        }
        const bool todo = have && !resolved && !skip;
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, todo);
        int base_slot = 0;
        if (lane == 0 && mask) base_slot = atomicAdd(n_work2, __popc(mask));
        base_slot = __shfl_sync(0xFFFFFFFFu, base_slot, 0);
        if (todo) worklist2[base_slot + __popc(mask & ((1u << lane) - 1u))] = read;
        n_done += __popc(__ballot_sync(0xFFFFFFFFu, resolved));
    }
    if (lane == 0 && n_done && counters) atomicAdd(counters + 2, (unsigned long long)n_done);
}

size_t deep_smem(const DevSet &S)
{
    size_t words = (size_t)S.words * S.n_classes * S.n_bc_pad + (size_t)kSeedMaxHits * kSeedThreads;
    for (int t = 0; t < S.sdd_n; t++)
        words += ((size_t)1 << (S.sdd[t].bm_log2 - 5)) + ((size_t)1 << S.sdd[t].log2) + 1 + 2 * (size_t)S.sdd[t].n_entries;
    return words * 4 + (size_t)kSeedMaxWins * kSeedThreads * 2 + 256 + (size_t)kSeedThreads * kSeedSlot + 16;
}

cudaError_t launch_seed_deep(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n, const Scratch &sc,
                             const int *wl_in, const int *n_in, int *wl_out, int *n_out, int sm_count,
                             unsigned long long *counters, cudaStream_t st)
{
    const DevSet &S = P.set[pass];
    const size_t smem = deep_smem(S);
    auto kern = S.words == 1 ? k_seed_deep<1> : k_seed_deep<2>;
    int blocks = 0;
    cudaError_t e = resident_grid((const void *)kern, kSeedThreads, smem, (n + kSeedThreads - 1) / kSeedThreads, sm_count,
                                  &blocks);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(n_out, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    kern<<<blocks, kSeedThreads, smem, st>>>(P, pass, seq, off, sc.pass[pass], sc.pass[0], wl_in, n_in, wl_out, n_out, counters,
                                             sc.cand, sc.cand_cnt, sc.wl_win, sc.n_lit);
    return cudaGetLastError();
}

}  // namespace bdx
