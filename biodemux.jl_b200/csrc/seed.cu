// seed.cu -- depth-limited seed-and-verify for :semiglobal in the exact regime.
//
// Setting: unit costs, default barcode start / end ranges (a barcode's result then does not depend on the
// running threshold), a barcode set of one common length m <= 64 without wildcard rows.  With min_delta = 0
// k_prefilter has already resolved the reads with a verbatim barcode occurrence; otherwise the first level
// takes every read.  A level resolves reads whose best barcode is within K edits, without running the
// full-range automaton:
//
//   * Pigeonhole: cut every barcode into K + 1 disjoint segments.  An alignment with <= K edits
//     leaves at least one segment untouched, so its first q bytes occur verbatim in the read at
//     column p = s + o + shift, |shift| <= K (s = alignment start, o = segment offset).
//   * Only the columns of the read's search range are staged (as class codes); every staged column's
//     q-mer is hashed (rolling polynomial hash) into a first-level bitmap and a CSR bucket table of
//     (barcode, o) entries; a hit fixes the diagonal delta = p - o.  Hits of one barcode on diagonals
//     <= K apart join one record whose window is the union of theirs.
//   * Each record is verified with the same Myers/Hyyro automaton as k_filter, but only over the
//     window of columns that can hold such an alignment.  A window is a sub-range of the search range
//     with free start and end, so its minimum is >= the full-range distance d_b, and for d_b <= K some
//     hit window contains an optimal alignment: min over the hit windows == d_b exactly whenever
//     d_b <= K.  The hits of a warp's 32 reads are pooled and spread evenly over the lanes
//     (seed_common.cuh); the verified distance goes back into the record.
//   * Hence the set {b : d_b <= K} and those distances are known exactly.  Non-empty: the reference's
//     winner is the lowest index among the minimal d_b (classification.jl:658); with min_delta the
//     read is decided when the runner-up is known (second-smallest d_b <= K) or provably far, else it
//     moves on; with trimming / stats the winner is queued for k_literal together with the columns
//     that hold all its best alignments.  Empty and K >= allowed at the last level: no barcode is
//     acceptable.  Everything else goes on through the other worklist (next level, then k_filter).
//
// Two levels (bdx_config_create): long, very selective seeds first, then the deepest level that is still
// selective.  One thread per read; wins and hits are first collected, then resolved / verified in lock
// step (doing it inside the scan would serialise the lanes of a warp, see k_prefilter).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <math_constants.h>
#include <type_traits>

#include "bdx_internal.h"
#include "literal.cuh"

#include "seed_common.cuh"

namespace bdx {

// the reference's acceptance of a barcode at distance d (classification.jl:254, :658, :696): the DP allows d
// (floor(fl(thr * norm))) and the score passes (fl(d / norm) <= thr).  Near the threshold either check can fail
// while the other passes.
__device__ __forceinline__ bool seed_accepts(int d, int norm, double max_error_rate)
{
    return d <= allowed_from(max_error_rate, norm) && __ddiv_rn((double)d, (double)norm) <= max_error_rate;
}

// TAB_SMEM: the CSR bucket table (bstart / entries / ekeys) is copied to shared memory; large sets read it
// from global memory instead (it is touched only on first-level bitmap hits).
template <bool TAB_SMEM, int W>      // W: 32-bit words per barcode row vector (1: up to 32 nt, 2: up to 64)
__global__ void __launch_bounds__(kSeedThreads)
k_seed(const __grid_constant__ DevParams P, const int pass, const int level, const uint8_t *__restrict__ seq,
       const int *__restrict__ off, const int n_reads, PassOut *__restrict__ out,
       const PassOut *__restrict__ prev_pass, const int *__restrict__ worklist,
       const int *__restrict__ n_work, int *__restrict__ worklist2, int *__restrict__ n_work2,
       unsigned long long *__restrict__ counters, uint16_t *__restrict__ cand, uint8_t *__restrict__ cand_cnt,
       int *__restrict__ wl_win, int *__restrict__ n_win)
{
    extern __shared__ __align__(16) uint32_t smem[];
    const DevSet &S = P.set[pass];
    const SeedLevel &SL = S.sd[level];
    // with trimming / stats the winner's alignment positions are needed too: the read is handed to k_literal
    // with the winner as its only candidate (in this regime a barcode's result does not depend on the running
    // threshold, so evaluating it alone gives the reference's positions)
    const bool need_tb = S.trim_side != 0 || P.want_stats;
    const int n_pad = S.n_bc_pad;
    const int n_buckets = 1 << SL.log2;
    const int bm_words = 1 << (SL.bm_log2 - 5);
    const int plane = S.n_classes * n_pad;
    uint32_t *peq_s = smem;                                     // [W][n_classes][n_pad]
    uint32_t *bitmap_s = peq_s + W * plane;
    uint32_t *tab_s = bitmap_s + bm_words;
    const uint32_t *bstart_s = TAB_SMEM ? tab_s : SL.bstart;    // [n_buckets + 1]
    const uint32_t *entries_s = TAB_SMEM ? tab_s + n_buckets + 1 : SL.entries;             // [n_entries]
    const uint32_t *ekeys_s = TAB_SMEM ? tab_s + n_buckets + 1 + SL.n_entries : SL.ekeys;  // [n_entries] full hashes
    const int max_hits = SL.max_hits;                           // rows of the per-read hit list (sized by the host per level)
    uint32_t *hits_s = TAB_SMEM ? tab_s + n_buckets + 1 + 2 * SL.n_entries : tab_s;        // [max_hits][kSeedThreads]
    uint8_t *wins_s = reinterpret_cast<uint8_t *>(hits_s + max_hits * kSeedThreads);   // [kSeedMaxWins][threads]
    uint8_t *class_s = wins_s + kSeedMaxWins * kSeedThreads;
    uint8_t *slot_s = class_s + 256;                            // [kSeedThreads][kSeedSlot] class codes

    for (int k = threadIdx.x; k < W * plane; k += blockDim.x) peq_s[k] = S.peq[k];
    for (int k = threadIdx.x; k < bm_words; k += blockDim.x) bitmap_s[k] = SL.bitmap[k];
    if (TAB_SMEM) {
        for (int k = threadIdx.x; k <= n_buckets; k += blockDim.x) tab_s[k] = SL.bstart[k];
        for (int k = threadIdx.x; k < SL.n_entries; k += blockDim.x) {
            tab_s[n_buckets + 1 + k] = SL.entries[k];
            tab_s[n_buckets + 1 + SL.n_entries + k] = SL.ekeys[k];
        }
    }
    for (int k = threadIdx.x; k < 256; k += blockDim.x) class_s[k] = S.class_of[k];
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int m = S.sd_m, K = SL.k, q = SL.q;
    const bool last_level = level == S.sd_levels - 1;
    const uint32_t pw = SL.pow;
    const int bm_log2 = SL.bm_log2;
    const int n_items = worklist ? *n_work : n_reads;         // no worklist: every read of the batch
    const bool with_delta = P.min_delta != 0.0;
    const int n_groups = (n_items + kSeedThreads - 1) / kSeedThreads;
    unsigned int n_done = 0;

    unsigned long long scan_cols = 0, ver_cols = 0;      // work counters for the roofline: q-mers probed, window columns verified
    for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        const int item = grp * kSeedThreads + threadIdx.x;
        const bool have = item < n_items;
        const int read = have ? (worklist ? worklist[item] : item) : 0;
        const int base = have ? off[read] : 0;
        const int n = have ? off[read + 1] - base : 0;

        bool punt = !have;       // true => this read goes to the next stage (or is not a read at all)
        bool skip = false;       // pass 2 of a read whose pass 1 did not match: nothing to do
        Geometry g{};
        if (have && pass == 1 && prev_pass[read].bc <= 0) {      // classification.jl:879-888
            out[read] = PassOut{kBcNotRun, 0, -1, -1};
            skip = true;
            punt = true;
        }
        if (have && !skip) {
            g = pass_geometry(S, n);
            // the regime test of k_filter's `fast` / k_prefilter<0>; the search range has to fit the slot
            // (the read itself may be much longer: only the columns of its search range are staged)
            if (!(g.valid && g.max_start_pos >= n && g.min_end_pos <= g.start_j) || g.end_j - g.start_j + 1 > kSeedSlot - 3)
                punt = true;
        }
        // From here on columns are RELATIVE to the search range: column c of the range (1-based, 1 = start_j)
        // is absolute column c + sbase and lives in my_slot[c - 1].
        const int sbase = punt ? 0 : g.start_j - 1;
        const int L = punt ? 0 : g.end_j - g.start_j + 1;

        // ---- stage the search ranges of the warp's 32 reads as class codes, coalesced: four reads at a time,
        // all their global loads issued before the first table lookup / store ----
        const int skew = seed_slot_skew(seq, (long long)base + sbase);          // the slot keeps the source alignment
        uint8_t *my_slot = slot_s + (size_t)threadIdx.x * kSeedSlot + skew;
        __syncwarp();
        seed_stage_warp(seq, (long long)base + sbase, L, slot_s + (size_t)warp * 32 * kSeedSlot, class_s, lane);
        __syncwarp();

        // ---- scan, phase 1: remember the columns whose q-mer passes the first-level bitmap.
        // (Doing the bucket walk right here would serialise the lanes of a warp: every lane hits
        // at different columns.  The divergent part is kept to one shared-memory store.) ----
        int n_wins = 0;
        if (!punt) {
            const int p0 = 0;                          // 0-based (relative) column of the first q-mer
            const int p1 = L - q;                      // last one that lies inside the search range
            if (p1 >= p0) {
                scan_cols += (unsigned)(p1 - p0 + 1);
                uint32_t h = 0;
                for (int i = 0; i < q; i++) h = h * kPfBase + (uint32_t)my_slot[p0 + i];
                auto probe = [&](int p) {
                    const uint32_t bit = pf_bit(h, bm_log2);
                    if ((bitmap_s[bit >> 5] >> (bit & 31)) & 1u) {
                        if (n_wins < kSeedMaxWins) wins_s[n_wins * kSeedThreads + threadIdx.x] = (uint8_t)p;
                        n_wins++;
                    }
                };
                const uint8_t *c_in = my_slot + q;
#pragma unroll 4
                for (int p = p0; p < p1; p++) {
                    probe(p);
                    h = (h - (uint32_t)my_slot[p] * pw) * kPfBase + (uint32_t)c_in[p];
                }
                probe(p1);
            }
            if (n_wins > kSeedMaxWins) punt = true;
        }

        // ---- scan, phase 2 (lock step over the remembered columns): bucket walk, key check,
        // (barcode, diagonal) hits ----
        int n_hits = 0;
        {
            const int my_wins = punt ? 0 : n_wins;
            const int max_wins = __reduce_max_sync(0xFFFFFFFFu, my_wins);
            for (int k = 0; k < max_wins; k++) {
                if (k >= my_wins) continue;
                const int p = wins_s[k * kSeedThreads + threadIdx.x];
                uint32_t h = 0;
                for (int i = 0; i < q; i++) h = h * kPfBase + (uint32_t)my_slot[p + i];
                const uint32_t bucket = pf_slot(h, SL.log2);
                const uint32_t e1 = bstart_s[bucket + 1];
                for (uint32_t e = bstart_s[bucket]; e < e1; e++) {
                    if (ekeys_s[e] != h) continue;                      // bucket-mate with another q-mer
                    const uint32_t ent = entries_s[e];
                    // 32-bit hash collisions are harmless: a false hit only costs a verification
                    const int delta = p - (int)(ent & 0xFFu);           // 0-based diagonal
                    const uint32_t b = ent >> 8;
                    // Several intact segments of one alignment hit the same barcode on diagonals at most K apart.
                    // When such a hit follows directly on the previous one of this read (the usual case: a read
                    // has one real match and few chance hits) it joins that record, whose window becomes the
                    // union of theirs (still a sub-range with free ends, and it contains every alignment either
                    // window contained).  Otherwise it gets a record of its own: every record is verified in its
                    // own window and the barcode's distance is the minimum over its records, so a missed merge
                    // only costs a verification.  (Searching ALL earlier records for a partner ran at 5 of 32
                    // lanes and cost 12 % of the kernel's instructions, profiles/r02_kernels_ncu_summary.txt.)
                    if (n_hits > 0 && n_hits <= max_hits) {
                        const uint32_t old = hits_s[(n_hits - 1) * kSeedThreads + threadIdx.x];
                        if ((old >> 13) == b) {
                            const int dmin = (int)(old & 0x3FFu) - 256, span = (int)((old >> 10) & 0x7u);
                            const int lo = min(dmin, delta), hi = max(dmin + span, delta);
                            if (hi - lo <= K) {
                                hits_s[(n_hits - 1) * kSeedThreads + threadIdx.x] = hit_pack(b, hi - lo, lo);
                                continue;
                            }
                        }
                    }
                    if (n_hits < max_hits) hits_s[n_hits * kSeedThreads + threadIdx.x] = hit_pack(b, 0, delta);
                    n_hits++;
                }
            }
            if (n_hits > max_hits) punt = true;
        }

        // ---- verify: the warp pools the hits of its 32 reads and spreads them evenly over the lanes
        // (a lane's own read has 0..max_hits hits; verifying per lane would leave most lanes idle) ----
        const int my_hits = punt ? 0 : n_hits;
        int incl = my_hits;                                      // inclusive prefix sum over the lanes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        const int total_hits = __shfl_sync(0xFFFFFFFFu, incl, 31);
        if (lane == 0) ver_cols += (unsigned)(total_hits * (m + 2 * K));    // the least window a hit has to be stepped over
        __syncwarp();
        {
            const int win = m + 4 * K + 1;                   // columns [dmin + 1 - K, dmin + span + m + 2K], span <= K
            using WT = typename std::conditional<W == 1, uint32_t, unsigned long long>::type;
            const SeedVerifyCtx vc{hits_s + warp * 32, peq_s, slot_s + (size_t)warp * 32 * kSeedSlot, n_pad, plane, m, K, win,
                                   total_hits};
            int i0 = 0;
            for (; i0 + 32 < total_hits; i0 += 64) seed_verify<2, WT>(vc, i0, lane, incl, 1, L, skew);
            if (i0 < total_hits) seed_verify<1, WT>(vc, i0, lane, incl, 1, L, skew);
        }
        __syncwarp();
        // ---- the read's own hits, now with distances: d_b = min over the hit groups of barcode b.
        // best = smallest distance, lowest index among equals; second = smallest d_b of any OTHER barcode ----
        int best_d = kInf, best_b = 0x7FFFFFFF, second_d = kInf;
        for (int k = 0; k < my_hits; k++) {
            const uint32_t rec = hits_s[k * kSeedThreads + threadIdx.x];
            const int d = (int)((rec >> 27) & 0xFu), b = (int)((rec >> 13) & 0x3FFFu);
            if (d > K) continue;
            if (d < best_d || (d == best_d && b < best_b)) {
                best_d = d;
                best_b = b;
            }
        }
        if (with_delta)
            for (int k = 0; k < my_hits; k++) {
                const uint32_t rec = hits_s[k * kSeedThreads + threadIdx.x];
                const int d = (int)((rec >> 27) & 0xFu), b = (int)((rec >> 13) & 0x3FFFu);
                if (d <= K && b != best_b) second_d = min(second_d, d);
            }

        // ---- decide ----
        bool resolved = false, queued = false;      // queued: winner handed to k_literal for its positions
        if (!punt) {
            if (best_d <= K) {
                // acceptance exactly as find_best_matching_bc_* does it for this barcode (classification.jl:254,
                // :658, :696); with one common length the earlier, worse barcodes the reference may accept first
                // cannot change the final winner
                const int norm = S.norm[best_b];
                const double sc = __ddiv_rn((double)best_d, (double)norm);
                if (best_d <= allowed_from(P.max_error_rate, norm) && sc <= P.max_error_rate) {
                    bool decided = true, ambiguous = false;
                    if (with_delta) {
                        // delta = second-best score - best score (:711).  Every barcode within K edits is known
                        // exactly; an unseen runner-up is more than K edits away.  A runner-up counts only if the
                        // reference accepts it (:696): both checks pass, as for the best.  With one common length
                        // both are monotone in the distance, so when the nearest one fails, every farther one
                        // fails too and sub_min stays Inf
                        if (second_d <= K) {
                            const double sc2 = __ddiv_rn((double)second_d, (double)norm);
                            ambiguous = seed_accepts(second_d, norm, P.max_error_rate) && __dsub_rn(sc2, sc) < P.min_delta;
                        } else if (seed_accepts(K + 1, norm, P.max_error_rate)) {
                            const double sc2 = __ddiv_rn((double)(K + 1), (double)norm);
                            decided = !(__dsub_rn(sc2, sc) < P.min_delta);      // safe whatever the runner-up is
                        }
                    }
                    if (decided) {
                        if (ambiguous) {
                            out[read] = PassOut{kBcAmbiguous, 0, -1, -1};
                        } else if (need_tb) {
                            // columns that hold every best alignment of the winner: the union of the windows
                            // of its hit groups that verified at the best distance (any column where it
                            // scores best_d ends an alignment with an intact segment, i.e. lies in one of them)
                            int lo = 0x7FFFFFFF, hi = 0;
                            for (int k = 0; k < my_hits; k++) {
                                const uint32_t rec = hits_s[k * kSeedThreads + threadIdx.x];
                                if ((int)((rec >> 27) & 0xFu) != best_d || (int)((rec >> 13) & 0x3FFFu) != best_b) continue;
                                const int dmin = (int)(rec & 0x3FFu) - 256, span = (int)((rec >> 10) & 0x7u);
                                lo = min(lo, dmin + 1 - K);
                                hi = max(hi, dmin + span + m + 2 * K);
                            }
                            cand[(size_t)read * kCandMax] = (uint16_t)best_b;
                            const int w_lo = max(lo - 2 + sbase, 1), w_hi = min(hi + 2 + sbase, n);   // absolute columns
                            cand[(size_t)read * kCandMax + 1] = (uint16_t)w_lo;
                            cand[(size_t)read * kCandMax + 2] = (uint16_t)w_hi;
                            // (columns beyond the uint16 slots: k_literal aligns the winner over the whole range)
                            cand_cnt[read] = (uint8_t)(w_hi <= 65535 ? kCandWindow : 1);
                            out[read] = PassOut{kBcPending, 0, -1, -1};
                            queued = true;
                        } else {
                            out[read] = PassOut{best_b + 1, best_d, -1, -1};
                        }
                        resolved = true;
                    }
                }
            } else if (last_level && K >= S.allowed0[0]) {
                out[read] = PassOut{kBcUnknown, 0, -1, -1};    // nothing within the allowed distance
                resolved = true;
            }
        }
        {   // warp-aggregated append of the queued winners to k_literal's list
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
    if (counters) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) scan_cols += __shfl_down_sync(0xFFFFFFFFu, scan_cols, o);
        if (lane == 0) {
            if (scan_cols) atomicAdd(counters + 5, scan_cols);
            if (ver_cols) atomicAdd(counters + 6, ver_cols);
        }
    }
}

static size_t seed_tab_words(const SeedLevel &L) { return ((size_t)1 << L.log2) + 1 + 2 * (size_t)L.n_entries; }

static size_t seed_smem(const DevSet &S, const SeedLevel &L, bool tab_smem)
{
    size_t words = (size_t)S.words * S.n_classes * S.n_bc_pad + ((size_t)1 << (L.bm_log2 - 5)) + (tab_smem ? seed_tab_words(L) : 0) +
                   (size_t)L.max_hits * kSeedThreads;
    return words * 4 + (size_t)kSeedMaxWins * kSeedThreads + 256 + (size_t)kSeedThreads * kSeedSlot + 16;
}

// the CSR table goes to shared memory while the whole carve-up stays small enough for >= 3 blocks per SM
static bool seed_tab_in_smem(const DevSet &S, const SeedLevel &L) { return seed_smem(S, L, true) <= 72 * 1024; }

size_t seed_smem(const DevSet &S, const SeedLevel &L) { return seed_smem(S, L, seed_tab_in_smem(S, L)); }

cudaError_t launch_seed(const DevParams &P, int pass, int level, const uint8_t *seq, const int *off, int n,
                        const Scratch &sc, const int *wl_in, const int *n_in, int *wl_out, int *n_out, int sm_count,
                        unsigned long long *counters, cudaStream_t st)
{
    const DevSet &S = P.set[pass];
    const SeedLevel &L = S.sd[level];
    const bool tab = seed_tab_in_smem(S, L);
    const size_t smem = seed_smem(S, L, tab);
    auto kern = S.words == 1 ? (tab ? k_seed<true, 1> : k_seed<false, 1>) : (tab ? k_seed<true, 2> : k_seed<false, 2>);
    int blocks = 0;     // groups of n reads: an upper bound, the worklist is <= n
    cudaError_t e = resident_grid((const void *)kern, kSeedThreads, smem, (n + kSeedThreads - 1) / kSeedThreads, sm_count,
                                  &blocks);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(n_out, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    kern<<<blocks, kSeedThreads, smem, st>>>(P, pass, level, seq, off, n, sc.pass[pass], sc.pass[0], wl_in, n_in, wl_out, n_out,
                                             counters, sc.cand, sc.cand_cnt, sc.wl_win, sc.n_lit);
    return cudaGetLastError();
}

}  // namespace bdx
