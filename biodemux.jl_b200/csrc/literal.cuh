// literal.cuh -- scalar device implementations that keep the reference's control
// flow cell for cell.  They evaluate ONE (read, barcode) pair under the *running*
// threshold, exactly like the Julia functions they follow, and are used
//   * for every candidate the bit-parallel filter kernel lets through, and
//   * for whole barcode sets when no filter applies (:hamming, :exact, exotic costs).
// Everything order- or threshold-dependent in the reference (SURVEY.md section 9) lives
// here, so bit-exactness does not depend on the fast kernels' algebra.
//
// Cells are int32 (the reference uses Int64): config creation bounds every cost
// by 2^20 and barcode length by 256, so no cell exceeds 2^29 = kInf.
#pragma once

#include <math_constants.h>

#include "bdx_internal.h"

namespace bdx {

struct Costs {
    int match, mismatch, indel, nindel;
    int has_n;
};

// floor(Int, max_error * normalization_length)  (classification.jl:254, :567) as an
// IEEE double multiply (no contraction), clamped to +-2^28 which is beyond any
// reachable cell value and therefore indistinguishable from the unclamped Int64.
// The host (allowed0, tables.cu) must get the same value as every kernel.
__host__ __device__ __forceinline__ int allowed_from(double max_error, int norm)
{
#ifdef __CUDA_ARCH__
    double x = floor(__dmul_rn(max_error, (double)norm));
#else
    volatile double prod = max_error * (double)norm;   // stored as a double: no fused multiply-add on the host
    double x = floor(prod);
#endif
    if (!(x < 268435456.0)) return 268435456;  // also catches NaN/Inf
    if (x < -268435456.0) return -268435456;
    return (int)x;
}

// resolve(dr, len)  (classification.jl:96-100) with Julia's UnitRange normalisation
__host__ __device__ __forceinline__ void resolve_range(const DevRange &dr, int len, int &first, int &last)
{
    int s = dr.start_from_end ? len + dr.start_off : dr.start_off;
    int e = dr.end_from_end ? len + dr.end_off : dr.end_off;
    first = max(1, s);
    last = min(len, e);
    if (last < first) last = first - 1;
}

struct Geometry {
    int start_j, end_j, max_start_pos, min_end_pos;
    bool valid;
};

// match_barcode_pass range prologue (classification.jl:795-807)
__host__ __device__ __forceinline__ Geometry pass_geometry(const DevSet &S, int n)
{
    int rf, rl, bf, bl, ef, el;
    resolve_range(S.rs, n, rf, rl);
    resolve_range(S.bs, n, bf, bl);
    resolve_range(S.be, n, ef, el);
    Geometry g;
    g.start_j = max(rf, max(bf, 1));
    g.end_j = min(rl, min(el, n));
    g.max_start_pos = bl;
    g.min_end_pos = ef;
    g.valid = !(g.start_j > g.end_j || g.start_j > g.max_start_pos || g.end_j < g.min_end_pos);
    return g;
}

// The columns of a read of length n that a classification can depend on (bdx_submit_windows): per pass that runs,
// :semiglobal [start_j, end_j] (sg_literal reads no other column); :hamming / :exact [start_j, last + max_m - 1]
// with last = min(end_j, max_start_pos), the furthest column a start position's comparison reaches.  exact_literal
// may scan beyond, but an occurrence it finds outside the window gives kInf whatever the bytes are (findprev:
// every start in [first, last] is tried before any start < first; findnext: every one before any > last).
// sp = lo1, hi1, lo2, hi2 (1-based, inclusive, hi < lo = empty), sorted and merged when they overlap or touch.
// Returns the number of window columns.
__host__ __device__ __forceinline__ int read_windows(const DevParams &P, int n, int sp[4])
{
    int lo[2] = {1, 1}, hi[2] = {0, 0};
    for (int p = 0; p < (P.is_dual ? 2 : 1); p++) {
        const DevSet &S = P.set[p];
        const Geometry g = pass_geometry(S, n);
        if (!g.valid) continue;
        lo[p] = g.start_j;
        hi[p] = P.algo == BDX_SEMIGLOBAL ? g.end_j : min(n, min(g.end_j, g.max_start_pos) + S.max_m - 1);
        if (hi[p] < lo[p]) lo[p] = 1, hi[p] = 0;
    }
    const bool e0 = hi[0] < lo[0], e1 = hi[1] < lo[1];
    if (e0 || (!e1 && lo[1] < lo[0])) {          // the non-empty / leftmost span first
        int t = lo[0]; lo[0] = lo[1]; lo[1] = t;
        t = hi[0]; hi[0] = hi[1]; hi[1] = t;
    }
    if (hi[1] >= lo[1] && lo[1] <= hi[0] + 1) {  // overlapping or touching: one span
        hi[0] = max(hi[0], hi[1]);
        lo[1] = 1, hi[1] = 0;
    }
    sp[0] = lo[0], sp[1] = hi[0], sp[2] = lo[1], sp[3] = hi[1];
    return max(0, hi[0] - lo[0] + 1) + max(0, hi[1] - lo[1] + 1);
}

// semiglobal_alignment_core (classification.jl:238-445).  q1 / r1 are 1-based
// (pointer to the byte before the first).  Returns the integer score or kInf;
// TB selects TracebackOutput(trim_side) vs ScoreOnly.
// Workspace column (SemiGlobalWorkspace.DP / .origin, classification.jl:1-6): element i of this
// thread lives at base[i * stride] -- stride 1 for thread-local arrays, stride = block size for
// the shared-memory layout [row][thread] (conflict-free: a warp touches 32 consecutive words).
struct WsCol {
    int *base;
    int stride;
    __device__ __forceinline__ int &operator[](int i) const { return base[i * stride]; }
};

// win_first / win_last (optional): a column window that is known to hold EVERY minimum-score alignment of this
// barcode, start to end (k_seed derives it from the verified seed hits).  The DP then runs over the window
// only.  Nothing outside can change the result: update_result keeps minimum-score hits only (:141-153), all of
// which end inside the window; a cell on a minimum-score path has the same value as in the full DP (a cheaper
// path into it from outside would give a cheaper alignment), and a tie at such a cell against a path from
// outside would make that path a minimum-score alignment itself -- which the window contains by construction.
// The column before an inner window start stands for "free start here": cost indel * i like the true first
// column, labelled with its own column number, which is the label the reference gives an alignment that
// opens with skipped barcode bases there (previous_score_origin = j, :287, :305).
template <bool TB>
__device__ int sg_literal(const WsCol DP, const WsCol OR, const uint8_t *q1, const uint8_t *r1, int m, int n,
                          int allowed_error, const Costs &c, int trim_side, int range_first,
                          int range_last, int max_start_pos, int min_end_pos, int &out_s, int &out_e,
                          int win_first = 0, int win_last = 0x7FFFFFFF)
{
    out_s = -1;
    out_e = -1;
    if (m == 0 || n == 0) return kInf;                               // :250-252
    int res_score = kInf, res_s = -1, res_e = -1;                     // init_result :130-136
    const int min_cost = c.has_n ? min(c.indel, c.nindel) : c.indel;
    const int steps = allowed_error / min_cost;                       // :170-176 (truncating div)
    const int min_valid_start = min_end_pos - (m + steps) + 1;        // :259
    if (min_valid_start > max_start_pos) return kInf;                 // :261-263
    if (min_valid_start > range_first) range_first = max(range_first, min_valid_start);  // :266-268
    const int band_offset = max(m - n - steps, -max_start_pos - steps);                  // :270

    const bool inner_start = win_first > range_first;
    if (inner_start) range_first = win_first;
    range_last = min(range_last, win_last);
    for (int i = 1; i <= m; i++) {                                    // :278-283
        DP[i] = c.indel * i;
        if (TB) OR[i] = inner_start ? range_first - 1 : 1 - i;
    }
    int lact = min(allowed_error + 1, m);                             // :286
    for (int j = range_first; j <= range_last; j++) {
        int prev_o = j, prev, fact, cur_o = 0;
        if (j + band_offset >= 1) {                                   // :289-295
            fact = j + band_offset;
            prev = allowed_error;
        } else {
            fact = 1;
            prev = 0;
        }
        if (fact > lact) break;                                       // :297-299
        const uint8_t rj = r1[j];
        int ins, del, sub;
        // --- first computed row: step_scores (:208-236, :303-335)
        {
            const int i = fact;
            const uint8_t qi = q1[i];
            const bool is_n = c.has_n && qi == (uint8_t)'N';
            const int cost = is_n ? c.nindel : c.indel;
            ins = (i == m) ? (c.has_n ? DP[i] + kInf : kInf) : DP[i] + cost;   // :213 / :229
            del = prev + cost;
            sub = (i == 1 ? 0 : DP[i - 1]) + ((qi == rj || is_n) ? c.match : c.mismatch);
            if (TB) {
                int best = del, bo = prev_o;
                const int sub_o = (i == 1) ? j : OR[i - 1];
                if (sub < best) { best = sub; bo = sub_o; }
                if (ins < best) { best = ins; bo = OR[i]; }
                cur_o = bo;
            }
            if (i != 1) {
                DP[i - 1] = prev;
                if (TB) OR[i - 1] = prev_o;
            }
            prev = min(ins, min(del, sub));
            if (TB) prev_o = cur_o;
        }
        // --- interior rows: step_scores_main (:178-206, :338-373)
        const int limit = (lact == m) ? m - 1 : lact;
        for (int i = fact + 1; i <= limit; i++) {
            const uint8_t qi = q1[i];
            const bool is_n = c.has_n && qi == (uint8_t)'N';
            const int cost = is_n ? c.nindel : c.indel;
            ins = DP[i] + cost;
            del = prev + cost;
            sub = DP[i - 1] + ((qi == rj || is_n) ? c.match : c.mismatch);
            if (TB) {
                int best = del, bo = prev_o;
                if (sub < best) { best = sub; bo = OR[i - 1]; }
                if (ins < best) { best = ins; bo = OR[i]; }
                cur_o = bo;
            }
            DP[i - 1] = prev;
            if (TB) OR[i - 1] = prev_o;
            prev = min(ins, min(del, sub));
            if (TB) prev_o = cur_o;
        }
        // --- last row, no insertion (:376-409)
        if (lact == m && lact > fact) {
            const uint8_t qi = q1[m];
            const bool is_n = c.has_n && qi == (uint8_t)'N';
            const int cost = is_n ? c.nindel : c.indel;
            ins = c.has_n ? DP[m] + kInf : kInf;
            del = prev + cost;
            sub = DP[m - 1] + ((qi == rj || is_n) ? c.match : c.mismatch);
            if (TB) {
                int best = del, bo = prev_o;
                if (sub < best) { best = sub; bo = OR[m - 1]; }
                if (ins < best) { best = ins; bo = OR[m]; }
                cur_o = bo;
            }
            DP[m - 1] = prev;
            if (TB) OR[m - 1] = prev_o;
            prev = min(ins, min(del, sub));
            if (TB) prev_o = cur_o;
        }
        DP[lact] = prev;                                              // :412-415
        if (TB) OR[lact] = prev_o;

        if (lact == m && prev <= allowed_error) {                     // :417-438
            lact -= 1;
            if (j >= min_end_pos) {
                if (prev == 0 && (!TB || trim_side == 5)) {           // :420-429 early exit
                    if (TB) { out_s = prev_o; out_e = j; }
                    return 0;
                }
                if (TB) {                                             // update_result :142-153
                    if (prev < res_score) {
                        res_score = prev; res_s = prev_o; res_e = j;
                    } else if (prev == res_score && trim_side == 3 && prev_o > res_s) {
                        res_s = prev_o; res_e = j;
                    }
                } else {
                    res_score = min(res_score, prev);                 // :138-140
                }
            }
        }
        while (lact > 0 && DP[lact] > allowed_error) lact -= 1;       // :439-442
        lact += 1;
    }
    if (TB) { out_s = res_s; out_e = res_e; }
    return res_score >= kInf ? kInf : res_score;                      // :155-168
}

// hamming_align (classification.jl:557-625).  Returns mismatches or kInf.
__device__ __forceinline__ int hamming_literal(const uint8_t *q, int m, const uint8_t *r, int n, int allowed,
                                               int range_first, int range_last, int max_start_pos,
                                               int min_end_pos, int trim_side, int &out_s, int &out_e)
{
    out_s = -1;
    out_e = -1;
    int best = kInf;
    const int first = max(range_first, 1);                                   // :570
    const int last = min(range_last, min(max_start_pos, n - m + 1));         // :571
    for (int j = first; j <= last; j++) {
        const int end_pos = j + m - 1;
        if (end_pos < min_end_pos) continue;                                 // :583-586
        int mm = 0;
        bool failed = false;
        for (int k = 0; k < m; k++) {
            const uint8_t qc = q[k], rc = r[j - 1 + k];
            if (qc != rc && qc != 0x4E) {                                    // :597
                if (++mm > allowed) { failed = true; break; }
            }
        }
        if (!failed) {
            // score = mm / m with one m: ordering of scores == ordering of mm (:607-620)
            if (mm < best) {
                best = mm; out_s = j; out_e = end_pos;
            } else if (mm == best && trim_side == 3 && j > out_s) {
                out_s = j; out_e = end_pos;
            }
        }
    }
    return best;
}

// exact_align (classification.jl:485-548).  Returns 0 or kInf.
__device__ __forceinline__ bool bytes_equal(const uint8_t *a, const uint8_t *b, int m)
{
    for (int k = 0; k < m; k++)
        if (a[k] != b[k]) return false;
    return true;
}

__device__ __forceinline__ int exact_literal(const uint8_t *q, int m, const uint8_t *r, int n,
                                             int range_first, int range_last, int max_start_pos,
                                             int min_end_pos, int trim_side, int &out_s, int &out_e)
{
    out_s = -1;
    out_e = -1;
    const int first = max(range_first, 1);                                   // :490
    const int last = min(range_last, min(max_start_pos, n - m + 1));         // :491
    if (last < first) return kInf;
    if (trim_side == 3) {
        // findprev(q, r, last + m - 1): rightmost occurrence ending at or before that index,
        // then ONE validity check -- it does not search further left (:499-515)
        for (int s = min(last + m - 1, n) - m + 1; s >= 1; s--) {
            if (bytes_equal(q, r + s - 1, m)) {
                if (s >= first && s + m - 1 >= min_end_pos) { out_s = s; out_e = s + m - 1; return 0; }
                return kInf;
            }
        }
        return kInf;
    }
    // findnext from `first`, keep scanning while the occurrence ends too early (:519-546)
    for (int s = first; s + m - 1 <= n; s++) {
        if (bytes_equal(q, r + s - 1, m)) {
            if (s > last) return kInf;
            if (s + m - 1 >= min_end_pos) { out_s = s; out_e = s + m - 1; return 0; }
        }
    }
    return kInf;
}

// Running best / second-best of find_best_matching_bc_{no,with}_delta (:632-713).
struct BestState {
    double thr, min_score, sub_min;
    int min_bc, min_dist, s, e;
};

__device__ __forceinline__ void best_init(BestState &b, double max_error_rate)
{
    b.thr = max_error_rate;
    b.min_score = CUDART_INF;
    b.sub_min = CUDART_INF;
    b.min_bc = 0;
    b.min_dist = 0;
    b.s = -1;
    b.e = -1;
}

__device__ __forceinline__ void best_consider(BestState &b, bool with_delta, double score, int dist, int bc,
                                              int s, int e)
{
    if (!with_delta) {
        if (score <= b.thr && score < b.min_score) {                  // :658-664
            b.min_score = score;
            b.min_bc = bc;
            b.min_dist = dist;
            b.thr = fmin(b.thr, b.min_score);
            b.s = s;
            b.e = e;
        }
    } else if (score <= b.thr) {                                      // :696-708
        if (score < b.min_score) {
            b.sub_min = b.min_score;
            b.min_score = score;
            b.min_bc = bc;
            b.min_dist = dist;
            b.thr = fmin(b.thr, b.sub_min);
            b.s = s;
            b.e = e;
        } else if (score < b.sub_min) {
            b.sub_min = score;
            b.thr = fmin(b.thr, b.sub_min);
        }
    }
}

// status decision of match_barcode_pass (:820-824)
__device__ __forceinline__ PassOut best_finish(const BestState &b, bool with_delta, double min_delta)
{
    PassOut o;
    o.dist = 0;
    o.start = -1;
    o.end = -1;
    if (b.min_bc == 0) {
        o.bc = kBcUnknown;
        return o;
    }
    const double delta = with_delta ? __dsub_rn(b.sub_min, b.min_score) : CUDART_INF;  // :666, :711
    if (delta < min_delta) {
        o.bc = kBcAmbiguous;
        return o;
    }
    o.bc = b.min_bc;
    o.dist = b.min_dist;
    o.start = b.s;
    o.end = b.e;
    return o;
}

}  // namespace bdx
