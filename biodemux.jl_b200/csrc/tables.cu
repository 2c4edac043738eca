// tables.cu -- host-side barcode tables of a bdx_config (built once per config, uploaded per device by
// bdx_api.cu): the byte -> class map and the Peq match masks of the bit-parallel kernels, the hash table of
// the perfect-occurrence prefilter, the seed tables of k_seed / k_seed_deep / k_seed_var and the bit planes of
// the packed Hamming scan.  Pure host code.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>

#include "api_internal.h"

using namespace bdx;

static int narrow_range(const bdx_range &in, DevRange &out, const char *name)
{
    const int64_t lim = 1ll << 30;
    if (in.start_offset > lim || in.start_offset < -lim || in.end_offset > lim || in.end_offset < -lim)
        return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": range offset out of bounds");
    out.start_off = (int)in.start_offset;
    out.start_from_end = in.start_from_end ? 1 : 0;
    out.end_off = (int)in.end_offset;
    out.end_from_end = in.end_from_end ? 1 : 0;
    return BDX_OK;
}

static int host_allowed(double max_error, int norm)
{
    // floor(Int, max_error * normalization_length), classification.jl:254 (same clamp as the device)
    volatile double prod = max_error * (double)norm;
    double x = std::floor(prod);
    if (!(x < 268435456.0)) return 268435456;
    if (x < -268435456.0) return -268435456;
    return (int)x;
}

namespace {

// what the builders below share
struct Build {
    const bdx_params &p;
    HostSet &hs;
    uint32_t debug;
    bool sg;          // :semiglobal
    bool benign;      // costs for which the unit-cost filter is a superset filter (DESIGN.md)
    int min_m;        // shortest barcode
};

// byte classes, Peq match masks and candidate thresholds of the bit-parallel kernels (filter.cu)
void build_filter_tables(const Build &B)
{
    const bdx_params &p = B.p;
    HostSet &hs = B.hs;
    const bool sg = B.sg, benign = B.benign;
    const int min_m = B.min_m;
    (void)p; (void)sg; (void)benign; (void)min_m;
    // ---- bit-parallel filter tables (semiglobal only) ----
    const int groups = (hs.n_bc + 31) / 32;
    int gpad = groups;
    if (groups > 4) {
        const int m3 = (groups + 2) / 3 * 3, m4 = (groups + 3) / 4 * 4;
        gpad = m4 <= m3 ? m4 : m3;
    }
    hs.n_bc_pad = gpad * 32;
    memset(hs.class_of, 0, sizeof(hs.class_of));
    hs.n_classes = 1;
    for (uint8_t c : hs.bytes)
        if (!hs.class_of[c]) hs.class_of[c] = (uint8_t)hs.n_classes++;
    hs.words = hs.max_m <= 32 ? 1 : (hs.max_m <= 32 * kMaxFilterWords ? 2 : 0);
    // The unit-cost filter is also a superset filter for :hamming (Hamming distance >= edit
    // distance; a barcode N is a wildcard there, classification.jl:597) and :exact (distance 0).
    // Tiny sets are cheaper to scan with the literal kernel than to spread over 32 lanes: they get the tables
    // (for the thread-per-read prefilter / seed kernels) but not the filter kernel.
    if ((sg && !benign) || (B.debug & BDX_DEBUG_NO_FILTER) || hs.n_classes > 64) hs.words = 0;
    hs.use_filter = hs.words > 0 && hs.n_bc >= 8;

    hs.allowed0.assign(hs.n_bc_pad, -1);
    hs.filt_allowed.assign(hs.n_bc_pad, -1);
    int64_t min_cost = std::min(p.mismatch, p.indel);
    if (p.has_nindel) min_cost = std::min(min_cost, p.nindel);
    for (int b = 0; b < hs.n_bc; b++) {
        hs.allowed0[b] = host_allowed(p.max_error_rate, hs.norm[b]);
        if (p.algorithm == BDX_EXACT)
            hs.filt_allowed[b] = p.max_error_rate >= 0.0 ? 0 : -1;          // score 0.0 <= thr (:658, :696)
        else if (p.algorithm == BDX_HAMMING)
            hs.filt_allowed[b] = hs.allowed0[b] < 0 ? -1 : hs.allowed0[b];  // floor(thr * m) (:567)
        else if (benign)
            hs.filt_allowed[b] = hs.allowed0[b] < 0 ? -1 : (int)(hs.allowed0[b] / min_cost);
    }
    if (hs.words) {
        const int W = hs.words;
        const size_t plane = (size_t)hs.n_classes * hs.n_bc_pad;
        hs.peq.assign((size_t)W * plane, 0u);
        for (int b = 0; b < hs.n_bc_pad; b++) {
            const int m = b < hs.n_bc ? hs.off[b + 1] - hs.off[b] : 0;
            const int first_row_bit = W * 32 - m;  // bit of barcode row 1; lower bits are phantom rows
            for (int c = 0; c < hs.n_classes; c++) {
                uint64_t v = first_row_bit >= 64 ? ~0ull : ((1ull << first_row_bit) - 1);  // phantom rows match
                if (W == 1) v &= 0xFFFFFFFFull;
                for (int i = 0; i < m; i++) {
                    const uint8_t q = hs.bytes[hs.off[b] + i];
                    // wildcard rows: NScoring (:196-203) and hamming_align (:597); literal in :exact
                    const bool is_n = q == (uint8_t)'N' && ((sg && p.has_nindel) || p.algorithm == BDX_HAMMING);
                    if (is_n || (c != 0 && hs.class_of[q] == c)) v |= 1ull << (first_row_bit + i);
                }
                hs.peq[0 * plane + (size_t)c * hs.n_bc_pad + b] = (uint32_t)v;
                if (W == 2) hs.peq[1 * plane + (size_t)c * hs.n_bc_pad + b] = (uint32_t)(v >> 32);
            }
        }
    }
}

// hash table of whole-barcode prefixes: k_prefilter (filter.cu)
void build_prefilter(const Build &B)
{
    const bdx_params &p = B.p;
    HostSet &hs = B.hs;
    const bool sg = B.sg, benign = B.benign;
    const int min_m = B.min_m;
    (void)p; (void)sg; (void)benign; (void)min_m;
    // ---- perfect-occurrence prefilter table (semiglobal, no wildcard rows) ----
    hs.bc_cls.resize(hs.bytes.size());
    for (size_t k = 0; k < hs.bytes.size(); k++) hs.bc_cls[k] = hs.class_of[hs.bytes[k]];
    const bool ex = p.algorithm == BDX_EXACT;   // :exact keeps duplicates (each index is a candidate)
    // :hamming treats every barcode N as a wildcard (classification.jl:597): no table then
    const bool hm = p.algorithm == BDX_HAMMING &&
                    std::find(hs.bytes.begin(), hs.bytes.end(), (uint8_t)'N') == hs.bytes.end();
    if (hs.words && ((sg && !p.has_nindel) || ex || hm) && min_m >= kPfMinSeed && !(B.debug & BDX_DEBUG_NO_PREFILTER)) {
        const int seed = std::min(min_m, kPfMaxSeed);
        hs.pf_seed = seed;
        uint32_t pw = 1;
        for (int i = 1; i < seed; i++) pw *= kPfBase;
        hs.pf_pow = pw;
        int lg = 4;
        while ((1 << lg) < 2 * hs.n_bc) lg++;
        hs.pf_log2 = lg;
        const uint32_t size = 1u << lg;
        hs.pf_keys.assign(size, 0u);
        hs.pf_vals.assign(size, kPfEmpty);
        int bl = 13;                                    // >= 512 bits per barcode, 8 KB .. 32 KB
        while (bl < 18 && (1 << bl) < 512 * hs.n_bc) bl++;
        hs.pf_bm_log2 = bl;
        hs.pf_bitmap.assign((size_t)1 << (bl - 5), 0u);
        for (int b = 0; b < hs.n_bc; b++) {            // ascending: the lowest index of identical sequences stays
            const int m = hs.off[b + 1] - hs.off[b];
            uint32_t h = 0;
            for (int i = 0; i < seed; i++) h = h * kPfBase + (uint32_t)hs.bytes[hs.off[b] + i];
            const uint32_t bit = pf_bit(h, bl);
            hs.pf_bitmap[bit >> 5] |= 1u << (bit & 31);
            uint32_t slot = pf_slot(h, lg);
            bool dup = false;
            while (hs.pf_vals[slot] != kPfEmpty) {
                const uint32_t v = hs.pf_vals[slot];
                const int ob = (int)(v & 0xFFFFu);
                if (!ex && (int)(v >> 16) == m &&
                    memcmp(&hs.bytes[hs.off[ob]], &hs.bytes[hs.off[b]], (size_t)m) == 0) {
                    dup = true;
                    break;
                }
                slot = (slot + 1) & (size - 1);
            }
            if (!dup) {
                hs.pf_keys[slot] = h;
                hs.pf_vals[slot] = ((uint32_t)m << 16) | (uint32_t)b;
            }
        }
        hs.pf_enabled = 1;
    }
}

// pigeonhole seed levels of k_seed (seed.cu)
void build_seed_levels(const Build &B)
{
    const bdx_params &p = B.p;
    HostSet &hs = B.hs;
    const bool sg = B.sg, benign = B.benign;
    const int min_m = B.min_m;
    (void)p; (void)sg; (void)benign; (void)min_m;
    // ---- :semiglobal depth-limited seeds (seed.cu): uniform barcode length, no wildcard rows ----
    if (hs.pf_enabled && sg && hs.words >= 1 && min_m == hs.max_m && hs.allowed0[0] >= 1 && hs.n_bc < (1 << 14) &&
        !(B.debug & BDX_DEBUG_NO_SEEDS)) {
        const int m = hs.max_m, allowed = hs.allowed0[0];
        const double alpha = std::max(2, hs.n_classes - 1);
        // chance hits per read column of level k: entries / alphabet^q with q = min(12, m / (k + 1))
        auto q_of = [&](int k) { return std::min(12, m / (k + 1)); };
        auto rate_of = [&](int k) { return (double)hs.n_bc * (k + 1) / std::pow(alpha, q_of(k)); };
        // deepest level whose seeds are long enough to be selective (q >= 6, <= 0.12 chance hits per column)
        int K = 0;
        for (int k = 1; k <= std::min(allowed, 7); k++)   // hit records keep the diagonal span in 3 bits
            if (q_of(k) >= 6 && rate_of(k) <= 0.12) K = k;
        // a shallower level with far fewer chance hits in front of it pays when the deep one has many
        int K0 = 0;
        if (K >= 2 && rate_of(K) > 0.02 && !(B.debug & BDX_DEBUG_ONE_SEED_LEVEL))
            for (int k = 1; k < K; k++)
                if (rate_of(k) <= 0.01) K0 = k;
        hs.sd_m = m;
        for (int K_l : {K0, K}) {
            if (K_l < 1) continue;
            HostSet::HostSeedLevel &L = hs.sd[hs.sd_levels++];
            const int seg = m / (K_l + 1), q = std::min(12, seg);
            L.k = K_l;
            L.q = q;
            // rows of k_seed's per-read hit list: three times the chance hits expected on 150 columns + two records
            // per true segment + slack.  (A fixed 28 rows cost 14 KB of shared memory per block -- one resident
            // block per SM less for 96 barcodes, whose lists never hold more than a handful.)
            L.max_hits = std::max(12, std::min(28, (int)std::ceil(3.0 * 150.0 * rate_of(K_l)) + 2 * (K_l + 1) + 4));
            uint32_t pw = 1;
            for (int i = 1; i < q; i++) pw *= kPfBase;
            L.pow = pw;
            const size_t n_entries = (size_t)hs.n_bc * (K_l + 1);
            int lg = 8;
            while (lg < 14 && (size_t)(1 << lg) < n_entries) lg++;
            L.log2 = lg;
            int bl = 13;                                // ~64 bits per entry: 4 KB for 96 barcodes
            while (bl < 18 && ((size_t)1 << bl) < 64 * n_entries) bl++;
            L.bm_log2 = bl;
            L.bitmap.assign((size_t)1 << (bl - 5), 0u);
            std::vector<std::vector<std::pair<uint32_t, uint32_t>>> buckets((size_t)1 << lg);
            for (int b = 0; b < hs.n_bc; b++)
                for (int i = 0; i <= K_l; i++) {
                    const int o = i * seg;
                    uint32_t h = 0;
                    for (int k = 0; k < q; k++) h = h * kPfBase + (uint32_t)hs.bc_cls[hs.off[b] + o + k];
                    const uint32_t bit = pf_bit(h, bl);
                    L.bitmap[bit >> 5] |= 1u << (bit & 31);
                    buckets[pf_slot(h, lg)].emplace_back(((uint32_t)b << 8) | (uint32_t)o, h);
                }
            L.bstart.assign(((size_t)1 << lg) + 1, 0u);
            for (size_t k = 0; k < buckets.size(); k++) {
                L.bstart[k + 1] = L.bstart[k] + (uint32_t)buckets[k].size();
                for (auto &pr : buckets[k]) {
                    L.entries.push_back(pr.first);
                    L.ekeys.push_back(pr.second);
                }
            }
        }
    }
}

// the deepest level of k_seed_deep (seed_deep.cu)
void build_seed_deep(const Build &B)
{
    const bdx_params &p = B.p;
    HostSet &hs = B.hs;
    const bool sg = B.sg, benign = B.benign;
    const int min_m = B.min_m;
    (void)p; (void)sg; (void)benign; (void)min_m;
    // ---- deepest seed level (seed_deep.cu): depth beyond the regular levels, each segment hashed with its own
    // length.  Measured on B200: with 0.75 chance hits per column (96 x 24 nt at depth 4) it is slower than the
    // bit-parallel kernel it would replace (17 vs 11.5 ms per 10 M-read step), so it is used while the hits
    // stay rare (<= 0.25 per column) -- small sets, e.g. one adapter, whose alternative is k_literal ----
    if (hs.sd_levels > 0 && !(B.debug & BDX_DEBUG_NO_SEED_DEEP)) {
        const int m = hs.max_m, allowed = hs.allowed0[0];
        const double alpha = std::max(2, hs.n_classes - 1);
        const double deep_rate = 0.25;      // chance hits per column the deep level accepts (measured, see above)
        int KD = 0;
        for (int k = hs.sd[hs.sd_levels - 1].k + 1; k <= std::min(allowed, 7); k++) {
            const int n_seg = k + 1, base_len = m / n_seg, extra = m % n_seg;
            if (base_len < 4) break;
            double rate = 0.0;
            for (int i = 0; i < n_seg; i++) rate += hs.n_bc / std::pow(alpha, std::min(base_len + (i < extra ? 1 : 0), 8));
            if (rate <= deep_rate) KD = k;
        }
        if (KD > 0) {
            const int n_seg = KD + 1, base_len = m / n_seg, extra = m % n_seg;
            const int q_long = std::min(base_len + 1, 8), q_short = std::min(base_len, 8);
            hs.sdd_k = KD;
            // table 0: the longer seeds (if any segment is longer and that changes the seed length), table 1 / 0: the rest
            struct Seg { int off, q; };
            std::vector<Seg> segs[2];
            int o = 0;
            for (int i = 0; i < n_seg; i++) {
                const int len = base_len + (i < extra ? 1 : 0);
                const int q = std::min(len, 8);
                segs[(q == q_long && q_long != q_short) ? 0 : 1].push_back(Seg{o, q});
                o += len;
            }
            for (int t = 0; t < 2; t++) {
                if (segs[t].empty()) continue;
                HostSet::HostSeedLevel &L = hs.sdd[hs.sdd_n++];
                const int q = segs[t][0].q;
                L.k = KD;
                L.q = q;
                uint32_t pw = 1;
                for (int i = 1; i < q; i++) pw *= kPfBase;
                L.pow = pw;
                const size_t n_entries = (size_t)hs.n_bc * segs[t].size();
                int lg = 8;
                while (lg < 14 && (size_t)(1 << lg) < n_entries) lg++;
                L.log2 = lg;
                int bl = 13;
                while (bl < 18 && ((size_t)1 << bl) < 64 * n_entries) bl++;
                L.bm_log2 = bl;
                L.bitmap.assign((size_t)1 << (bl - 5), 0u);
                std::vector<std::vector<std::pair<uint32_t, uint32_t>>> buckets((size_t)1 << lg);
                for (int b = 0; b < hs.n_bc; b++)
                    for (const Seg &sg2 : segs[t]) {
                        uint32_t h = 0;
                        for (int k = 0; k < q; k++) h = h * kPfBase + (uint32_t)hs.bc_cls[hs.off[b] + sg2.off + k];
                        const uint32_t bit = pf_bit(h, bl);
                        L.bitmap[bit >> 5] |= 1u << (bit & 31);
                        buckets[pf_slot(h, lg)].emplace_back(((uint32_t)b << 8) | (uint32_t)sg2.off, h);
                    }
                L.bstart.assign(((size_t)1 << lg) + 1, 0u);
                for (size_t k = 0; k < buckets.size(); k++) {
                    L.bstart[k + 1] = L.bstart[k] + (uint32_t)buckets[k].size();
                    for (auto &pr : buckets[k]) {
                        L.entries.push_back(pr.first);
                        L.ekeys.push_back(pr.second);
                    }
                }
            }
        }
    }
}

// levels of k_seed_var (seed_var.cu)
void build_seed_var(const Build &B)
{
    const bdx_params &p = B.p;
    HostSet &hs = B.hs;
    const bool sg = B.sg, benign = B.benign;
    const int min_m = B.min_m;
    (void)p; (void)sg; (void)benign; (void)min_m;
    // ---- seed-and-verify for sets of different lengths and constrained start / end geometries (seed_var.cu):
    // K_b + 1 disjoint segments per barcode, K_b = min(m_b / q - 1, allowed_b), their first q bases in a
    // direct-address table.  Level 1: q = the shortest seed whose CHANCE hits on admissible diagonals (estimated
    // for a 150-base read) stay around two dozen per read -- position constraints keep short seeds selective.
    // Level 2 (reads level 1 could not decide): the longest seed that is COMPLETE (K_b = allowed_b for every
    // barcode, so the candidates are a superset and every verdict is final), used while verifying its chance
    // hits costs less than half the lane-per-barcode automaton over the whole range ----
    if (sg && hs.words >= 1 && !p.has_nindel && hs.n_classes - 1 <= 4 && hs.n_bc < (1 << 14) && hs.max_m <= 64 &&
        p.max_error_rate >= 0.0 && !(B.debug & BDX_DEBUG_NO_SEEDS)) {
        auto resolve = [](const DevRange &dr, int len, int &first, int &last) {      // classification.jl:96-100
            const int s = dr.start_from_end ? len + dr.start_off : dr.start_off;
            const int e = dr.end_from_end ? len + dr.end_off : dr.end_off;
            first = std::max(1, s);
            last = std::min(len, e);
            if (last < first) last = first - 1;
        };
        const int n_nom = 150;
        int rf, rl, bf, bl, ef, el;
        resolve(hs.rs, n_nom, rf, rl);
        resolve(hs.bs, n_nom, bf, bl);
        resolve(hs.be, n_nom, ef, el);
        const int start_j = std::max(rf, std::max(bf, 1)), end_j = std::min(rl, std::min(el, n_nom));
        const int L = std::max(end_j - start_j + 1, 1), sbase = start_j - 1;
        const int min_end_rel = ef - sbase, max_start_rel = bl - sbase;
        struct Est { double chance, steps; size_t n_entries; bool complete; };
        // admissible diagonals of barcode b at depth K (seed_var.cu, scan)
        auto n_diag = [&](int m, int a0, int K) {
            const int dlo = std::max(0, min_end_rel - m) - K, dhi = std::min(max_start_rel + a0, L - m + K);
            return std::max(0, dhi - dlo + 1);
        };
        auto estimate = [&](int q) {
            Est e{0.0, 0.0, 0, true};
            for (int b = 0; b < hs.n_bc; b++) {
                const int m = hs.off[b + 1] - hs.off[b], a0 = hs.allowed0[b];
                const int K = std::min(m / q - 1, a0);
                const double c = (double)(K + 1) * n_diag(m, a0, K) / std::pow(4.0, q);
                e.chance += c;
                e.steps += c * (m + 2 * K);          // columns verified for those hits
                e.n_entries += (size_t)K + 1;
                if (K < a0) e.complete = false;
            }
            return e;
        };
        // reads per group: 128 and a hit list of up to 40 rows x 128 records (seed_var.cu) that their hits -- chance
        // + a handful of true ones -- fill to about 70 %; denser levels take fewer reads per group instead.
        // The 3-gram filter between the hit test and the list pays when most hits can fail it ((m - 2) - 3 K >= 4
        // for most barcodes); about one chance hit in seven passes it then (measured: one in ten for 24 nt, K = 4).
        auto size_groups = [&](HostSet::HostSeedVar &V, double chance) {
            int strong = 0;
            for (int b = 0; b < hs.n_bc; b++)
                strong += (hs.off[b + 1] - hs.off[b] - 2) - 3 * (int)V.kdepth[(size_t)b] >= 4;
            V.qgram_filter = hs.max_m <= 32 && 2 * strong >= hs.n_bc && !(B.debug & BDX_DEBUG_NO_QGRAM_FILTER);
            // mode 1 tests inside the scan (only survivors reach the list), mode 2 over the finished list: with few
            // admissible diagonals per barcode (constrained start / end) the scan's lanes rarely hold a hit at the
            // same time and the test would run for two or three lanes of a warp
            if (V.qgram_filter) {
                double adm = 0.0, all = 0.0;
                for (int b = 0; b < hs.n_bc; b++) {
                    const int m = hs.off[b + 1] - hs.off[b], K = V.kdepth[(size_t)b];
                    adm += (double)(K + 1) * n_diag(m, hs.allowed0[b], K);
                    all += (double)(K + 1) * L;
                }
                V.qgram_filter = adm >= 0.5 * all ? 1 : 2;
            }
            const double pass = V.qgram_filter == 1 ? (0.15 * strong + (hs.n_bc - strong)) / hs.n_bc : 1.0;
            const double per_read = chance * pass + 6.0;
            // shared memory per read (staged range, its bit planes, candidates, bookkeeping) kept to ~20 KB per block:
            // five or six blocks per SM hide the scan's shuffle and shared-memory latencies, three do not
            // (measured: 0.50 -> issue slots used with three resident blocks)
            const int per_read_bytes = (L + 8) + (V.qgram_filter ? 12 * ((L + 32) / 32 + 3) : 0) + 64;
            int R = 128;
            while (R > 32 && R * per_read_bytes > 20 * 1024) R -= 32;
            auto rows_for = [&](int r) { return (int)std::ceil(per_read * r / (0.7 * 128)); };
            while (R > 8 && rows_for(R) > 40) R -= R > 32 ? 32 : 8;          // (whole warps of reads while there are several)
            V.group_reads = R;
            V.hit_rows = std::max(8, std::min(40, rows_for(R)));
            // a constrained start is re-checked by sg_literal, whose DP column (max_m + 2 entries per thread) reuses the list
            const bool can_bound_start = !(hs.bs.end_from_end && hs.bs.end_off >= 0);
            if (can_bound_start) V.hit_rows = std::max(V.hit_rows, hs.max_m + 2);
        };
        // level with ONE seed length q: K_b + 1 segments of m_b / (K_b + 1) >= q bases, K_b = min(m_b / q - 1, allowed_b)
        auto build = [&](int q, double chance) {
            HostSet::HostSeedVar &V = hs.sv[hs.sv_levels++];
            V.q = q;
            V.q2 = 0;
            V.kdepth.assign((size_t)hs.n_bc, 0);
            std::vector<std::vector<uint32_t>> buckets((size_t)1 << (2 * q));
            V.sigma_min = 1e300;
            V.complete = 1;
            for (int b = 0; b < hs.n_bc; b++) {
                const int m = hs.off[b + 1] - hs.off[b], a0 = hs.allowed0[b];
                const int K = std::min(m / q - 1, a0);
                V.kdepth[(size_t)b] = (uint8_t)K;
                if (K < a0) V.complete = 0;
                V.sigma_min = std::min(V.sigma_min, (double)(K + 1) / (double)hs.norm[b]);
                const int seg = m / (K + 1);                       // >= q: the segments are disjoint
                for (int i = 0; i <= K; i++) {
                    const int o = i * seg;
                    uint32_t code = 0;
                    for (int k = 0; k < q; k++) code |= ((uint32_t)(hs.bc_cls[hs.off[b] + o + k] - 1) & 3u) << (2 * k);
                    buckets[code].push_back(((uint32_t)b << 8) | (uint32_t)o);
                }
            }
            V.bstart.assign(buckets.size() + 1, 0);
            for (size_t k = 0; k < buckets.size(); k++) {
                if (buckets[k].size() > 255) {                     // the scan keeps bucket sizes in a byte
                    V = HostSet::HostSeedVar();
                    hs.sv_levels--;
                    return;
                }
                V.bstart[k + 1] = (uint16_t)(V.bstart[k] + buckets[k].size());
                V.entries.insert(V.entries.end(), buckets[k].begin(), buckets[k].end());
            }
            size_groups(V, chance);
        };
        // COMPLETE level (K_b = allowed_b): barcode b is cut into allowed_b + 1 segments of m_b / (allowed_b + 1) bases,
        // the first m_b % (allowed_b + 1) of them one base longer; every segment is a seed of its own length, kept
        // in one of two tables (q and q + 1: e.g. 24 nt at depth 4 = four 5-mers and one 4-mer, 2.5 x fewer chance
        // hits than five 4-mers)
        struct Seg { int b, o, q; };
        auto complete_segments = [&](int q_lo, std::vector<Seg> &segs) {
            Est e{0.0, 0.0, 0, true};
            for (int b = 0; b < hs.n_bc; b++) {
                const int m = hs.off[b + 1] - hs.off[b], a0 = hs.allowed0[b];
                const int n_seg = a0 + 1, base = m / n_seg, extra = m % n_seg;
                int o = 0;
                for (int i = 0; i < n_seg; i++) {
                    const int len = base + (i < extra ? 1 : 0);
                    const int q = (len > q_lo && q_lo < 8) ? q_lo + 1 : q_lo;
                    segs.push_back(Seg{b, o, q});
                    const double c = (double)n_diag(m, a0, a0) / std::pow(4.0, q);
                    e.chance += c;
                    e.steps += c * (m + 2 * a0);
                    o += len;
                }
            }
            e.n_entries = segs.size();
            return e;
        };
        auto build_complete = [&](int q_lo, const std::vector<Seg> &segs, double chance) {
            HostSet::HostSeedVar &V = hs.sv[hs.sv_levels++];
            bool two = false;
            for (const Seg &sg2 : segs) two = two || sg2.q != q_lo;
            V.q = q_lo;
            V.q2 = two ? q_lo + 1 : 0;
            V.kdepth.assign((size_t)hs.n_bc, 0);
            V.sigma_min = 1e300;
            V.complete = 1;
            for (int b = 0; b < hs.n_bc; b++) {
                V.kdepth[(size_t)b] = (uint8_t)hs.allowed0[b];
                V.sigma_min = std::min(V.sigma_min, (double)(hs.allowed0[b] + 1) / (double)hs.norm[b]);
            }
            for (int t = 0; t < (two ? 2 : 1); t++) {
                const int q = t ? q_lo + 1 : q_lo;
                std::vector<std::vector<uint32_t>> buckets((size_t)1 << (2 * q));
                for (const Seg &sg2 : segs) {
                    if (sg2.q != q) continue;
                    uint32_t code = 0;
                    for (int k = 0; k < q; k++) code |= ((uint32_t)(hs.bc_cls[hs.off[sg2.b] + sg2.o + k] - 1) & 3u) << (2 * k);
                    buckets[code].push_back(((uint32_t)sg2.b << 8) | (uint32_t)sg2.o);
                }
                for (size_t k = 0; k < buckets.size(); k++) {
                    if (buckets[k].size() > 255) {                 // the scan keeps bucket sizes in a byte
                        V = HostSet::HostSeedVar();
                        hs.sv_levels--;
                        return;
                    }
                    V.bstart.push_back((uint16_t)V.entries.size());
                    V.entries.insert(V.entries.end(), buckets[k].begin(), buckets[k].end());
                }
                V.bstart.push_back((uint16_t)V.entries.size());
            }
            size_groups(V, chance);
        };
        int q1 = 0;
        for (int q = 4; q <= 8 && !q1; q++) {
            if (min_m < q) break;
            const Est e = estimate(q);
            if (e.chance <= 24.0 && e.n_entries <= 65535) {
                build(q, e.chance);
                if (hs.sv_levels > 0) q1 = q;
            }
        }
        if (q1 && !hs.sv[0].complete && !(B.debug & BDX_DEBUG_ONE_SEED_LEVEL)) {
            int q_lo = 8;
            for (int b = 0; b < hs.n_bc; b++) q_lo = std::min(q_lo, (hs.off[b + 1] - hs.off[b]) / (hs.allowed0[b] + 1));
            if (q_lo >= 3) {
                std::vector<Seg> segs;
                const Est e = complete_segments(q_lo, segs);
                const double automaton_steps = (double)hs.n_bc * L;
                if (e.n_entries <= 65535 && e.steps < 0.5 * automaton_steps && e.chance <= 200.0)
                    build_complete(q_lo, segs, e.chance);
            }
        }
        // With a complete level behind them (score-only passes, plan.cu), k_seed's levels only have to
        // be cheap, not deep: its second level is dropped when its seeds are short (> 0.02 chance hits per column,
        // e.g. 96 x 24 nt at depth 3: 6-mers, 14 chance hits per read) -- the reads it resolved cost less in the
        // complete level than the level costs on all of its input (config 2: 889 -> 910 M reads/s).  Sets without a
        // complete level keep it: there its reads would fall to the lane-per-barcode automaton (config 5: 38 -> 24).
        if (hs.sv_levels > 0 && hs.sv[hs.sv_levels - 1].complete && hs.sd_levels == 2 && hs.trim_side == 0 && !p.want_stats) {
            const HostSet::HostSeedLevel &D = hs.sd[1];
            const double rate = (double)hs.n_bc * (D.k + 1) / std::pow((double)std::max(2, hs.n_classes - 1), D.q);
            if (rate > 0.02) {
                hs.sd[1] = HostSet::HostSeedLevel();
                hs.sd_levels = 1;
            }
        }
    }
}

// bit planes and direct-address seed tables of k_hamming_scan (hamming.cu)
void build_hamming_packed(const Build &B)
{
    const bdx_params &p = B.p;
    HostSet &hs = B.hs;
    const bool sg = B.sg, benign = B.benign;
    const int min_m = B.min_m;
    (void)p; (void)sg; (void)benign; (void)min_m;
    // ---- :hamming on packed words (hamming.cu): uniform length <= 32, <= 4 distinct barcode bytes, no 'N' ----
    if (!(B.debug & BDX_DEBUG_NO_HAMMING_PACKED) && p.algorithm == BDX_HAMMING && min_m == hs.max_m && hs.max_m <= 32 && hs.n_classes - 1 <= 4 && hs.n_bc <= 65535 &&
        hs.allowed0[0] >= 0 && hs.allowed0[0] <= 7 && p.max_error_rate >= 0.0 &&
        std::find(hs.bytes.begin(), hs.bytes.end(), (uint8_t)'N') == hs.bytes.end()) {
        const int m = hs.max_m, n_seg = hs.allowed0[0] + 1;
        const int seg_len = m / n_seg, extra = m % n_seg;      // the first `extra` segments are one base longer
        if (seg_len >= 2) {
            hs.hp_m = m;
            hs.hp_allowed = hs.allowed0[0];
            hs.hp_n_seg = n_seg;
            int o = 0, base = 0;
            for (int i = 0; i < n_seg; i++) {
                const int len = seg_len + (i < extra ? 1 : 0);
                hs.hp_off[i] = o;
                hs.hp_q[i] = std::min(len, 6);                  // direct-address table of 4^q buckets
                hs.hp_base[i] = base;
                base += (1 << (2 * hs.hp_q[i])) + 1;
                o += len;
            }
            auto code_of = [&](int b, int pos) { return (uint32_t)(hs.bc_cls[hs.off[b] + pos] - 1) & 3u; };
            hs.hp_bstart.assign((size_t)base, 0);
            hs.hp_entries.assign((size_t)n_seg * hs.n_bc, 0);
            for (int i = 0; i < n_seg; i++) {
                const int nb = 1 << (2 * hs.hp_q[i]);
                std::vector<std::vector<uint16_t>> buckets((size_t)nb);
                for (int b = 0; b < hs.n_bc; b++) {
                    uint32_t gram = 0;           // bit plane 0 of the q bases, then bit plane 1
                    for (int k = 0; k < hs.hp_q[i]; k++) {
                        const uint32_t c = code_of(b, hs.hp_off[i] + k);
                        gram |= (c & 1u) << k;
                        gram |= (c >> 1) << (hs.hp_q[i] + k);
                    }
                    buckets[gram].push_back((uint16_t)b);
                }
                uint16_t run = 0;
                size_t w = (size_t)i * hs.n_bc;
                for (int gidx = 0; gidx < nb; gidx++) {
                    hs.hp_bstart[(size_t)hs.hp_base[i] + gidx] = run;
                    for (uint16_t b : buckets[(size_t)gidx]) hs.hp_entries[w++] = b;
                    run = (uint16_t)(run + buckets[(size_t)gidx].size());
                }
                hs.hp_bstart[(size_t)hs.hp_base[i] + nb] = run;
            }
            hs.hp_bcw.resize((size_t)hs.n_bc);
            for (int b = 0; b < hs.n_bc; b++) {
                uint32_t w0 = 0, w1 = 0;         // the two bit planes, base k in bit k
                for (int k = 0; k < m; k++) {
                    w0 |= (code_of(b, k) & 1u) << k;
                    w1 |= (code_of(b, k) >> 1) << k;
                }
                hs.hp_bcw[(size_t)b] = make_uint2(w0, w1);
            }
            hs.hp_enabled = 1;
        }
    }
}

}  // namespace

int bdx_build_set(const bdx_params &p, const bdx_barcode_set &in, HostSet &hs, uint32_t debug, const char *name)
{
    if (in.n_barcodes <= 0 || !in.bytes || !in.offsets)
        return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": empty barcode set");
    if (in.n_barcodes > 65535) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": more than 65535 barcodes");
    if (in.trim_side != 0 && in.trim_side != 3 && in.trim_side != 5)
        return bdx_fail(BDX_ERR_INVALID, "trim_side must be 3 or 5");  // core.jl:308-313
    if (p.has_nindel && !in.lengths_no_n)
        return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": lengths_no_n required with nindel");
    hs.n_bc = in.n_barcodes;
    hs.trim_side = in.trim_side;
    int rc;
    if ((rc = narrow_range(in.ref_search_range, hs.rs, name))) return rc;
    if ((rc = narrow_range(in.barcode_start_range, hs.bs, name))) return rc;
    if ((rc = narrow_range(in.barcode_end_range, hs.be, name))) return rc;
    if (in.offsets[0] != 0) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": offsets[0] must be 0");
    hs.off.assign(in.offsets, in.offsets + in.n_barcodes + 1);
    hs.max_m = 0;
    for (int b = 0; b < hs.n_bc; b++) {
        const int m = hs.off[b + 1] - hs.off[b];
        if (m <= 0) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": empty barcode (not supported)");
        if (m > kMaxBarcodeLen) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": barcode longer than 256");
        hs.max_m = std::max(hs.max_m, m);
    }
    hs.bytes.assign(in.bytes, in.bytes + hs.off[hs.n_bc]);
    hs.norm.resize(hs.n_bc);
    for (int b = 0; b < hs.n_bc; b++) {
        const int m = hs.off[b + 1] - hs.off[b];
        // semiglobal: m, or bc_lengths_no_N under NScoring (classification.jl:460, :476, :647);
        // hamming: m (:567, :607)
        hs.norm[b] = (p.algorithm == BDX_SEMIGLOBAL && p.has_nindel) ? in.lengths_no_n[b] : m;
        if (hs.norm[b] < 0) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": negative lengths_no_n");
        // floor(Int, max_error_rate * norm) (classification.jl:254, :567) raises InexactError unless the product is a
        // number whose floor fits Int64: refused here for every barcode, as the reference would fail on its first read
        volatile double prod = p.max_error_rate * (double)hs.norm[b];
        if (p.algorithm != BDX_EXACT && !(prod >= -9223372036854775808.0 && prod < 9223372036854775808.0))
            return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": max_error_rate * length outside Int64 (the reference "
                                                             "raises InexactError on floor(Int, max_error_rate * length))");
    }
    int min_m = hs.max_m;
    for (int b = 0; b < hs.n_bc; b++) min_m = std::min(min_m, hs.off[b + 1] - hs.off[b]);
    const bool benign = p.match >= 0 && p.mismatch >= 1 && p.indel >= 1 && (!p.has_nindel || p.nindel >= p.indel);
    const Build B{p, hs, debug, p.algorithm == BDX_SEMIGLOBAL, benign, min_m};
    build_filter_tables(B);
    build_prefilter(B);
    build_seed_levels(B);
    build_seed_deep(B);
    build_seed_var(B);
    build_hamming_packed(B);
    return BDX_OK;
}

// Text description of the tables built for one barcode set (bdx_config_describe): which shortcut stages exist and
// with which parameters.  Host data only.
std::string bdx_describe_set(const HostSet &hs)
{
    char line[256];
    std::string out;
    int min_m = hs.max_m;
    for (int b = 0; b < hs.n_bc; b++) min_m = std::min(min_m, hs.off[b + 1] - hs.off[b]);
    snprintf(line, sizeof line, "set: barcodes=%d length=%d..%d classes=%d words=%d filter=%d\n", hs.n_bc, hs.n_bc ? min_m : 0,
             hs.max_m, hs.n_classes - 1, hs.words, hs.use_filter);
    out += line;
    if (hs.pf_enabled) {
        snprintf(line, sizeof line, "prefilter: seed=%d log2=%d bitmap_log2=%d\n", hs.pf_seed, hs.pf_log2, hs.pf_bm_log2);
        out += line;
    }
    for (int l = 0; l < hs.sd_levels; l++) {
        snprintf(line, sizeof line, "k_seed level %d: K=%d q=%d entries=%zu max_hits=%d\n", l + 1, hs.sd[l].k, hs.sd[l].q,
                 hs.sd[l].entries.size(), hs.sd[l].max_hits);
        out += line;
    }
    for (int l = 0; l < hs.sdd_n; l++) {
        snprintf(line, sizeof line, "k_seed_deep table %d: K=%d q=%d entries=%zu\n", l + 1, hs.sdd_k, hs.sdd[l].q, hs.sdd[l].entries.size());
        out += line;
    }
    for (int l = 0; l < hs.sv_levels; l++) {
        const HostSet::HostSeedVar &V = hs.sv[l];
        int k_lo = 255, k_hi = 0;
        for (uint8_t k : V.kdepth) {
            k_lo = std::min<int>(k_lo, k);
            k_hi = std::max<int>(k_hi, k);
        }
        snprintf(line, sizeof line, "k_seed_var level %d: q=%d q2=%d K=%d..%d complete=%d entries=%zu group_reads=%d hit_rows=%d qgram_filter=%d\n",
                 l + 1, V.q, V.q2, V.kdepth.empty() ? 0 : k_lo, k_hi, V.complete, V.entries.size(), V.group_reads, V.hit_rows,
                 V.qgram_filter);
        out += line;
    }
    if (hs.hp_enabled) {
        snprintf(line, sizeof line, "k_hamming_scan: m=%d allowed=%d segments=%d\n", hs.hp_m, hs.hp_allowed, hs.hp_n_seg);
        out += line;
    }
    return out;
}

