// tables.cu -- host-side barcode tables of a bdx_config (built once per config, uploaded per device by
// bdx_api.cu): the byte -> class map and the Peq match masks of the bit-parallel kernels, the hash table of
// the perfect-occurrence prefilter, the seed tables of k_seed / k_seed_deep / k_seed_var and the bit planes of
// the packed Hamming scan.  Pure host code.  Each builder writes its stage's scalars into the set's DevSet (the
// config's base parameter block) and its vectors into the HostSet.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>

#include "api_internal.h"
#include "literal.cuh"

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

namespace {

// kPfBase^(q-1): the weight of a q-mer's first byte in its polynomial hash
uint32_t hash_pow(int q)
{
    uint32_t pw = 1;
    for (int i = 1; i < q; i++) pw *= kPfBase;
    return pw;
}

// byte classes, Peq match masks and candidate thresholds of the bit-parallel kernels (filter.cu)
void build_filter_tables(const bdx_params &p, HostSet &hs, DevSet &D, uint32_t debug)
{
    const bool sg = p.algorithm == BDX_SEMIGLOBAL;
    // costs for which the unit-cost filter is a superset filter (DESIGN.md)
    const bool benign = p.match >= 0 && p.mismatch >= 1 && p.indel >= 1 && (!p.has_nindel || p.nindel >= p.indel);
    // ---- bit-parallel filter tables (semiglobal only) ----
    const int groups = (D.n_bc + 31) / 32;
    int gpad = groups;
    if (groups > 4) {
        const int m3 = (groups + 2) / 3 * 3, m4 = (groups + 3) / 4 * 4;
        gpad = m4 <= m3 ? m4 : m3;
    }
    D.n_bc_pad = gpad * 32;
    hs.class_of.assign(256, 0);
    D.n_classes = 1;
    for (uint8_t c : hs.bytes)
        if (!hs.class_of[c]) hs.class_of[c] = (uint8_t)D.n_classes++;
    D.words = D.max_m <= 32 ? 1 : (D.max_m <= 32 * kMaxFilterWords ? 2 : 0);
    // The unit-cost filter is also a superset filter for :hamming (Hamming distance >= edit
    // distance; a barcode N is a wildcard there, classification.jl:597) and :exact (distance 0).
    // Tiny sets are cheaper to scan with the literal kernel than to spread over 32 lanes: they get the tables
    // (for the thread-per-read prefilter / seed kernels) but not the filter kernel.
    if ((sg && !benign) || (debug & BDX_DEBUG_NO_FILTER) || D.n_classes > 64) D.words = 0;
    D.use_filter = D.words > 0 && D.n_bc >= 8;

    hs.allowed0.assign(D.n_bc_pad, -1);
    hs.filt_allowed.assign(D.n_bc_pad, -1);
    int64_t min_cost = std::min(p.mismatch, p.indel);
    if (p.has_nindel) min_cost = std::min(min_cost, p.nindel);
    for (int b = 0; b < D.n_bc; b++) {
        hs.allowed0[b] = allowed_from(p.max_error_rate, hs.norm[b]);
        if (p.algorithm == BDX_EXACT)
            hs.filt_allowed[b] = p.max_error_rate >= 0.0 ? 0 : -1;          // score 0.0 <= thr (:658, :696)
        else if (p.algorithm == BDX_HAMMING)
            hs.filt_allowed[b] = hs.allowed0[b] < 0 ? -1 : hs.allowed0[b];  // floor(thr * m) (:567)
        else if (benign)
            hs.filt_allowed[b] = hs.allowed0[b] < 0 ? -1 : (int)(hs.allowed0[b] / min_cost);
    }
    if (D.words) {
        const int W = D.words;
        const size_t plane = (size_t)D.n_classes * D.n_bc_pad;
        hs.peq.assign((size_t)W * plane, 0u);
        for (int b = 0; b < D.n_bc_pad; b++) {
            const int m = b < D.n_bc ? hs.off[b + 1] - hs.off[b] : 0;
            const int first_row_bit = W * 32 - m;  // bit of barcode row 1; lower bits are phantom rows
            for (int c = 0; c < D.n_classes; c++) {
                uint64_t v = first_row_bit >= 64 ? ~0ull : ((1ull << first_row_bit) - 1);  // phantom rows match
                if (W == 1) v &= 0xFFFFFFFFull;
                for (int i = 0; i < m; i++) {
                    const uint8_t q = hs.bytes[hs.off[b] + i];
                    // wildcard rows: NScoring (:196-203) and hamming_align (:597); literal in :exact
                    const bool is_n = q == (uint8_t)'N' && ((sg && p.has_nindel) || p.algorithm == BDX_HAMMING);
                    if (is_n || (c != 0 && hs.class_of[q] == c)) v |= 1ull << (first_row_bit + i);
                }
                hs.peq[0 * plane + (size_t)c * D.n_bc_pad + b] = (uint32_t)v;
                if (W == 2) hs.peq[1 * plane + (size_t)c * D.n_bc_pad + b] = (uint32_t)(v >> 32);
            }
        }
    }
}

// hash table of whole-barcode prefixes: k_prefilter (filter.cu)
void build_prefilter(const bdx_params &p, HostSet &hs, DevSet &D, uint32_t debug)
{
    // ---- perfect-occurrence prefilter table (semiglobal, no wildcard rows) ----
    hs.bc_cls.resize(hs.bytes.size());
    for (size_t k = 0; k < hs.bytes.size(); k++) hs.bc_cls[k] = hs.class_of[hs.bytes[k]];
    const bool sg = p.algorithm == BDX_SEMIGLOBAL;
    const bool ex = p.algorithm == BDX_EXACT;   // :exact keeps duplicates (each index is a candidate)
    // :hamming treats every barcode N as a wildcard (classification.jl:597): no table then
    const bool hm = p.algorithm == BDX_HAMMING &&
                    std::find(hs.bytes.begin(), hs.bytes.end(), (uint8_t)'N') == hs.bytes.end();
    if (D.words && ((sg && !p.has_nindel) || ex || hm) && hs.min_m >= kPfMinSeed && !(debug & BDX_DEBUG_NO_PREFILTER)) {
        const int seed = std::min(hs.min_m, kPfMaxSeed);
        D.pf_seed = seed;
        D.pf_pow = hash_pow(seed);
        int lg = 4;
        while ((1 << lg) < 2 * D.n_bc) lg++;
        D.pf_log2 = lg;
        const uint32_t size = 1u << lg;
        hs.pf_keys.assign(size, 0u);
        hs.pf_vals.assign(size, kPfEmpty);
        int bl = 13;                                    // >= 512 bits per barcode, 8 KB .. 32 KB
        while (bl < 18 && (1 << bl) < 512 * D.n_bc) bl++;
        D.pf_bm_log2 = bl;
        hs.pf_bitmap.assign((size_t)1 << (bl - 5), 0u);
        for (int b = 0; b < D.n_bc; b++) {            // ascending: the lowest index of identical sequences stays
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
        D.pf_enabled = 1;
    }
}

// a hashed seed table of k_seed / k_seed_deep: the q-mer at each offset in `offs` of every barcode (class codes),
// a first-level bitmap and CSR buckets of (barcode index << 8) | offset with the q-mer's hash
void build_hashed_level(const HostSet &hs, int n_bc, int q, const std::vector<int> &offs, SeedLevel &L,
                        HostSet::HostSeedLevel &H)
{
    L.q = q;
    L.pow = hash_pow(q);
    const size_t n_entries = (size_t)n_bc * offs.size();
    int lg = 8;
    while (lg < 14 && (size_t)(1 << lg) < n_entries) lg++;
    L.log2 = lg;
    int bl = 13;                                // ~64 bits per entry: 4 KB for 96 barcodes
    while (bl < 18 && ((size_t)1 << bl) < 64 * n_entries) bl++;
    L.bm_log2 = bl;
    H.bitmap.assign((size_t)1 << (bl - 5), 0u);
    std::vector<std::vector<std::pair<uint32_t, uint32_t>>> buckets((size_t)1 << lg);
    for (int b = 0; b < n_bc; b++)
        for (int o : offs) {
            uint32_t h = 0;
            for (int k = 0; k < q; k++) h = h * kPfBase + (uint32_t)hs.bc_cls[hs.off[b] + o + k];
            const uint32_t bit = pf_bit(h, bl);
            H.bitmap[bit >> 5] |= 1u << (bit & 31);
            buckets[pf_slot(h, lg)].emplace_back(((uint32_t)b << 8) | (uint32_t)o, h);
        }
    H.bstart.assign(((size_t)1 << lg) + 1, 0u);
    for (size_t k = 0; k < buckets.size(); k++) {
        H.bstart[k + 1] = H.bstart[k] + (uint32_t)buckets[k].size();
        for (auto &pr : buckets[k]) {
            H.entries.push_back(pr.first);
            H.ekeys.push_back(pr.second);
        }
    }
    L.n_entries = (int)H.entries.size();
}

// pigeonhole seed levels of k_seed (seed.cu)
void build_seed_levels(const bdx_params &p, HostSet &hs, DevSet &D, uint32_t debug)
{
    // ---- :semiglobal depth-limited seeds (seed.cu): uniform barcode length, no wildcard rows ----
    if (D.pf_enabled && p.algorithm == BDX_SEMIGLOBAL && D.words >= 1 && hs.min_m == D.max_m && hs.allowed0[0] >= 1 &&
        D.n_bc < (1 << 14) && !(debug & BDX_DEBUG_NO_SEEDS)) {
        const int m = D.max_m, allowed = hs.allowed0[0];
        const double alpha = std::max(2, D.n_classes - 1);
        // chance hits per read column of level k: entries / alphabet^q with q = min(12, m / (k + 1))
        auto q_of = [&](int k) { return std::min(12, m / (k + 1)); };
        auto rate_of = [&](int k) { return (double)D.n_bc * (k + 1) / std::pow(alpha, q_of(k)); };
        // deepest level whose seeds are long enough to be selective (q >= 6, <= 0.12 chance hits per column)
        int K = 0;
        for (int k = 1; k <= std::min(allowed, 7); k++)   // hit records keep the diagonal span in 3 bits
            if (q_of(k) >= 6 && rate_of(k) <= 0.12) K = k;
        // a shallower level with far fewer chance hits in front of it pays when the deep one has many
        int K0 = 0;
        if (K >= 2 && rate_of(K) > 0.02 && !(debug & BDX_DEBUG_ONE_SEED_LEVEL))
            for (int k = 1; k < K; k++)
                if (rate_of(k) <= 0.01) K0 = k;
        D.sd_m = m;
        for (int K_l : {K0, K}) {
            if (K_l < 1) continue;
            const int l = D.sd_levels++, seg = m / (K_l + 1);
            SeedLevel &L = D.sd[l];
            L.k = K_l;
            // rows of k_seed's per-read hit list: three times the chance hits expected on 150 columns + two records
            // per true segment + slack.  (A fixed 28 rows cost 14 KB of shared memory per block -- one resident
            // block per SM less for 96 barcodes, whose lists never hold more than a handful.)
            L.max_hits = std::max(12, std::min(28, (int)std::ceil(3.0 * 150.0 * rate_of(K_l)) + 2 * (K_l + 1) + 4));
            std::vector<int> offs;
            for (int i = 0; i <= K_l; i++) offs.push_back(i * seg);
            build_hashed_level(hs, D.n_bc, q_of(K_l), offs, L, hs.sd[l]);
        }
    }
}

// the deepest level of k_seed_deep (seed_deep.cu)
void build_seed_deep(HostSet &hs, DevSet &D, uint32_t debug)
{
    // ---- deepest seed level (seed_deep.cu): depth beyond the regular levels, each segment hashed with its own
    // length.  Measured on B200: with 0.75 chance hits per column (96 x 24 nt at depth 4) it is slower than the
    // bit-parallel kernel it would replace (17 vs 11.5 ms per 10 M-read step), so it is used while the hits
    // stay rare (<= 0.25 per column) -- small sets, e.g. one adapter, whose alternative is k_literal ----
    if (D.sd_levels > 0 && !(debug & BDX_DEBUG_NO_SEED_DEEP)) {
        const int m = D.max_m, allowed = hs.allowed0[0];
        const double alpha = std::max(2, D.n_classes - 1);
        const double deep_rate = 0.25;      // chance hits per column the deep level accepts (measured, see above)
        int KD = 0;
        for (int k = D.sd[D.sd_levels - 1].k + 1; k <= std::min(allowed, 7); k++) {
            const int n_seg = k + 1, base_len = m / n_seg, extra = m % n_seg;
            if (base_len < 4) break;
            double rate = 0.0;
            for (int i = 0; i < n_seg; i++) rate += D.n_bc / std::pow(alpha, std::min(base_len + (i < extra ? 1 : 0), 8));
            if (rate <= deep_rate) KD = k;
        }
        if (KD > 0) {
            const int n_seg = KD + 1, base_len = m / n_seg, extra = m % n_seg;
            const int q_long = std::min(base_len + 1, 8), q_short = std::min(base_len, 8);
            D.sdd_k = KD;
            // table 0: the longer seeds (if any segment is longer and that changes the seed length), table 1 / 0: the rest
            std::vector<int> offs[2];
            int o = 0;
            for (int i = 0; i < n_seg; i++) {
                const int len = base_len + (i < extra ? 1 : 0);
                offs[(std::min(len, 8) == q_long && q_long != q_short) ? 0 : 1].push_back(o);
                o += len;
            }
            for (int t = 0; t < 2; t++) {
                if (offs[t].empty()) continue;
                const int l = D.sdd_n++;
                D.sdd[l].k = KD;
                build_hashed_level(hs, D.n_bc, t == 0 ? q_long : q_short, offs[t], D.sdd[l], hs.sdd[l]);
            }
        }
    }
}

// a segment of barcode b at offset o whose first q bases are a k_seed_var seed
struct VarSeg { int b, o, q; };

// appends one direct-address table of k_seed_var to H: 4^q + 1 CSR row starts over the 2-bit codes of the segments
// with seed length q, absolute indices into H.entries of (barcode index << 8) | offset.  false: a bucket holds more
// than 255 entries (the scan keeps bucket sizes in a byte)
bool append_direct_table(const HostSet &hs, int q, const std::vector<VarSeg> &segs, HostSet::HostSeedVar &H)
{
    std::vector<std::vector<uint32_t>> buckets((size_t)1 << (2 * q));
    for (const VarSeg &s : segs) {
        if (s.q != q) continue;
        uint32_t code = 0;
        for (int k = 0; k < q; k++) code |= ((uint32_t)(hs.bc_cls[hs.off[s.b] + s.o + k] - 1) & 3u) << (2 * k);
        buckets[code].push_back(((uint32_t)s.b << 8) | (uint32_t)s.o);
    }
    for (const std::vector<uint32_t> &bk : buckets) {
        if (bk.size() > 255) return false;
        H.bstart.push_back((uint16_t)H.entries.size());
        H.entries.insert(H.entries.end(), bk.begin(), bk.end());
    }
    H.bstart.push_back((uint16_t)H.entries.size());
    return true;
}

// levels of k_seed_var (seed_var.cu)
void build_seed_var(const bdx_params &p, HostSet &hs, DevSet &D, uint32_t debug)
{
    // ---- seed-and-verify for sets of different lengths and constrained start / end geometries (seed_var.cu):
    // K_b + 1 disjoint segments per barcode, K_b = min(m_b / q - 1, allowed_b), their first q bases in a
    // direct-address table.  Level 1: q = the shortest seed whose CHANCE hits on admissible diagonals (estimated
    // for a 150-base read) stay around two dozen per read -- position constraints keep short seeds selective.
    // Level 2 (reads level 1 could not decide): the longest seed that is COMPLETE (K_b = allowed_b for every
    // barcode, so the candidates are a superset and every verdict is final), used while verifying its chance
    // hits costs less than half the lane-per-barcode automaton over the whole range ----
    if (p.algorithm == BDX_SEMIGLOBAL && D.words >= 1 && !p.has_nindel && D.n_classes - 1 <= 4 && D.n_bc < (1 << 14) &&
        D.max_m <= 64 && p.max_error_rate >= 0.0 && !(debug & BDX_DEBUG_NO_SEEDS)) {
        const Geometry g = pass_geometry(D, 150);
        const int L = std::max(g.end_j - g.start_j + 1, 1), sbase = g.start_j - 1;
        const int min_end_rel = g.min_end_pos - sbase, max_start_rel = g.max_start_pos - sbase;
        struct Est { double chance, steps; size_t n_entries; bool complete; };
        // admissible diagonals of barcode b at depth K (seed_var.cu, scan)
        auto n_diag = [&](int m, int a0, int K) {
            const int dlo = std::max(0, min_end_rel - m) - K, dhi = std::min(max_start_rel + a0, L - m + K);
            return std::max(0, dhi - dlo + 1);
        };
        auto estimate = [&](int q) {
            Est e{0.0, 0.0, 0, true};
            for (int b = 0; b < D.n_bc; b++) {
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
        auto size_groups = [&](SeedVar &V, const std::vector<uint8_t> &kdepth, double chance) {
            int strong = 0;
            for (int b = 0; b < D.n_bc; b++)
                strong += (hs.off[b + 1] - hs.off[b] - 2) - 3 * (int)kdepth[(size_t)b] >= 4;
            V.qgram_filter = D.max_m <= 32 && 2 * strong >= D.n_bc && !(debug & BDX_DEBUG_NO_QGRAM_FILTER);
            // mode 1 tests inside the scan (only survivors reach the list), mode 2 over the finished list: with few
            // admissible diagonals per barcode (constrained start / end) the scan's lanes rarely hold a hit at the
            // same time and the test would run for two or three lanes of a warp
            if (V.qgram_filter) {
                double adm = 0.0, all = 0.0;
                for (int b = 0; b < D.n_bc; b++) {
                    const int m = hs.off[b + 1] - hs.off[b], K = kdepth[(size_t)b];
                    adm += (double)(K + 1) * n_diag(m, hs.allowed0[b], K);
                    all += (double)(K + 1) * L;
                }
                V.qgram_filter = adm >= 0.5 * all ? 1 : 2;
            }
            const double pass = V.qgram_filter == 1 ? (0.15 * strong + (D.n_bc - strong)) / D.n_bc : 1.0;
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
            const bool can_bound_start = !(D.bs.end_from_end && D.bs.end_off >= 0);
            if (can_bound_start) V.hit_rows = std::max(V.hit_rows, D.max_m + 2);
        };
        // the next level: the tables of the segments (seed length q, and q + 1 in a second table if any segment has
        // it), barcode b's seeds complete for kdepth[b] edits.  A level whose table refuses its bucket sizes is not
        // kept: its vectors are cleared and its SeedVar stays zero.
        auto add_level = [&](int q, const std::vector<VarSeg> &segs, std::vector<uint8_t> kdepth, double chance) {
            HostSet::HostSeedVar &H = hs.sv[D.sv_levels];
            bool two = false;
            for (const VarSeg &s : segs) two = two || s.q != q;
            for (int t = 0; t < (two ? 2 : 1); t++)
                if (!append_direct_table(hs, q + t, segs, H)) {
                    H = HostSet::HostSeedVar();
                    return;
                }
            SeedVar &V = D.sv[D.sv_levels++];
            V.enabled = 1;
            V.q = q;
            V.q2 = two ? q + 1 : 0;
            V.bstart2 = (1 << (2 * q)) + 1;
            V.n_bstart = (int)H.bstart.size();
            V.n_entries = (int)H.entries.size();
            V.complete = 1;
            V.sigma_min = 1e300;
            for (int b = 0; b < D.n_bc; b++) {
                if (kdepth[(size_t)b] < hs.allowed0[b]) V.complete = 0;
                V.sigma_min = std::min(V.sigma_min, (double)(kdepth[(size_t)b] + 1) / (double)hs.norm[b]);
            }
            size_groups(V, kdepth, chance);
            H.kdepth = std::move(kdepth);
        };
        // level with ONE seed length q: K_b + 1 segments of m_b / (K_b + 1) >= q bases, K_b = min(m_b / q - 1, allowed_b)
        auto build = [&](int q, double chance) {
            std::vector<VarSeg> segs;
            std::vector<uint8_t> kdepth((size_t)D.n_bc);
            for (int b = 0; b < D.n_bc; b++) {
                const int m = hs.off[b + 1] - hs.off[b], K = std::min(m / q - 1, hs.allowed0[b]);
                kdepth[(size_t)b] = (uint8_t)K;
                const int seg = m / (K + 1);                       // >= q: the segments are disjoint
                for (int i = 0; i <= K; i++) segs.push_back(VarSeg{b, i * seg, q});
            }
            add_level(q, segs, std::move(kdepth), chance);
        };
        // COMPLETE level (K_b = allowed_b): barcode b is cut into allowed_b + 1 segments of m_b / (allowed_b + 1) bases,
        // the first m_b % (allowed_b + 1) of them one base longer; every segment is a seed of its own length, kept
        // in one of two tables (q and q + 1: e.g. 24 nt at depth 4 = four 5-mers and one 4-mer, 2.5 x fewer chance
        // hits than five 4-mers)
        auto complete_segments = [&](int q_lo, std::vector<VarSeg> &segs) {
            Est e{0.0, 0.0, 0, true};
            for (int b = 0; b < D.n_bc; b++) {
                const int m = hs.off[b + 1] - hs.off[b], a0 = hs.allowed0[b];
                const int n_seg = a0 + 1, base = m / n_seg, extra = m % n_seg;
                int o = 0;
                for (int i = 0; i < n_seg; i++) {
                    const int len = base + (i < extra ? 1 : 0);
                    const int q = (len > q_lo && q_lo < 8) ? q_lo + 1 : q_lo;
                    segs.push_back(VarSeg{b, o, q});
                    const double c = (double)n_diag(m, a0, a0) / std::pow(4.0, q);
                    e.chance += c;
                    e.steps += c * (m + 2 * a0);
                    o += len;
                }
            }
            e.n_entries = segs.size();
            return e;
        };
        int q1 = 0;
        for (int q = 4; q <= 8 && !q1; q++) {
            if (hs.min_m < q) break;
            const Est e = estimate(q);
            if (e.chance <= 24.0 && e.n_entries <= 65535) {
                build(q, e.chance);
                if (D.sv_levels > 0) q1 = q;
            }
        }
        if (q1 && !D.sv[0].complete && !(debug & BDX_DEBUG_ONE_SEED_LEVEL)) {
            int q_lo = 8;
            for (int b = 0; b < D.n_bc; b++) q_lo = std::min(q_lo, (hs.off[b + 1] - hs.off[b]) / (hs.allowed0[b] + 1));
            if (q_lo >= 3) {
                std::vector<VarSeg> segs;
                const Est e = complete_segments(q_lo, segs);
                const double automaton_steps = (double)D.n_bc * L;
                if (e.n_entries <= 65535 && e.steps < 0.5 * automaton_steps && e.chance <= 200.0)
                    add_level(q_lo, segs, std::vector<uint8_t>(hs.allowed0.begin(), hs.allowed0.begin() + D.n_bc), e.chance);
            }
        }
        // With a complete level behind them (score-only passes, plan.cu), k_seed's levels only have to
        // be cheap, not deep: its second level is dropped when its seeds are short (> 0.02 chance hits per column,
        // e.g. 96 x 24 nt at depth 3: 6-mers, 14 chance hits per read) -- the reads it resolved cost less in the
        // complete level than the level costs on all of its input (config 2: 889 -> 910 M reads/s).  Sets without a
        // complete level keep it: there its reads would fall to the lane-per-barcode automaton (config 5: 38 -> 24).
        if (D.sv_levels > 0 && D.sv[D.sv_levels - 1].complete && D.sd_levels == 2 && D.trim_side == 0 && !p.want_stats) {
            const SeedLevel &L2 = D.sd[1];
            const double rate = (double)D.n_bc * (L2.k + 1) / std::pow((double)std::max(2, D.n_classes - 1), L2.q);
            if (rate > 0.02) {
                D.sd[1] = SeedLevel();
                hs.sd[1] = HostSet::HostSeedLevel();
                D.sd_levels = 1;
            }
        }
    }
}

// bit planes and direct-address seed tables of k_hamming_scan (hamming.cu)
void build_hamming_packed(const bdx_params &p, HostSet &hs, DevSet &D, uint32_t debug)
{
    // ---- :hamming on packed words (hamming.cu): uniform length <= 32, <= 4 distinct barcode bytes, no 'N' ----
    if (!(debug & BDX_DEBUG_NO_HAMMING_PACKED) && p.algorithm == BDX_HAMMING && hs.min_m == D.max_m && D.max_m <= 32 && D.n_classes - 1 <= 4 && D.n_bc <= 65535 &&
        hs.allowed0[0] >= 0 && hs.allowed0[0] <= 7 && p.max_error_rate >= 0.0 &&
        std::find(hs.bytes.begin(), hs.bytes.end(), (uint8_t)'N') == hs.bytes.end()) {
        const int m = D.max_m, n_seg = hs.allowed0[0] + 1;
        const int seg_len = m / n_seg, extra = m % n_seg;      // the first `extra` segments are one base longer
        if (seg_len >= 2) {
            HammingPacked &H = D.hp;
            H.m = m;
            H.allowed = hs.allowed0[0];
            H.n_seg = n_seg;
            int o = 0, base = 0;
            for (int i = 0; i < n_seg; i++) {
                const int len = seg_len + (i < extra ? 1 : 0);
                H.seg_off[i] = o;
                H.seg_q[i] = std::min(len, 6);                  // direct-address table of 4^q buckets
                H.seg_base[i] = base;
                base += (1 << (2 * H.seg_q[i])) + 1;
                o += len;
            }
            auto code_of = [&](int b, int pos) { return (uint32_t)(hs.bc_cls[hs.off[b] + pos] - 1) & 3u; };
            hs.hp_bstart.assign((size_t)base, 0);
            hs.hp_entries.assign((size_t)n_seg * D.n_bc, 0);
            for (int i = 0; i < n_seg; i++) {
                const int nb = 1 << (2 * H.seg_q[i]);
                std::vector<std::vector<uint16_t>> buckets((size_t)nb);
                for (int b = 0; b < D.n_bc; b++) {
                    uint32_t gram = 0;           // bit plane 0 of the q bases, then bit plane 1
                    for (int k = 0; k < H.seg_q[i]; k++) {
                        const uint32_t c = code_of(b, H.seg_off[i] + k);
                        gram |= (c & 1u) << k;
                        gram |= (c >> 1) << (H.seg_q[i] + k);
                    }
                    buckets[gram].push_back((uint16_t)b);
                }
                uint16_t run = 0;
                size_t w = (size_t)i * D.n_bc;
                for (int gidx = 0; gidx < nb; gidx++) {
                    hs.hp_bstart[(size_t)H.seg_base[i] + gidx] = run;
                    for (uint16_t b : buckets[(size_t)gidx]) hs.hp_entries[w++] = b;
                    run = (uint16_t)(run + buckets[(size_t)gidx].size());
                }
                hs.hp_bstart[(size_t)H.seg_base[i] + nb] = run;
            }
            hs.hp_bcw.resize((size_t)D.n_bc);
            for (int b = 0; b < D.n_bc; b++) {
                uint32_t w0 = 0, w1 = 0;         // the two bit planes, base k in bit k
                for (int k = 0; k < m; k++) {
                    w0 |= (code_of(b, k) & 1u) << k;
                    w1 |= (code_of(b, k) >> 1) << k;
                }
                hs.hp_bcw[(size_t)b] = make_uint2(w0, w1);
            }
            H.n_bstart = base;
            H.enabled = 1;
        }
    }
}

}  // namespace

int bdx_build_set(const bdx_params &p, const bdx_barcode_set &in, HostSet &hs, DevSet &D, uint32_t debug, const char *name)
{
    if (in.n_barcodes <= 0 || !in.bytes || !in.offsets)
        return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": empty barcode set");
    if (in.n_barcodes > 65535) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": more than 65535 barcodes");
    if (in.trim_side != 0 && in.trim_side != 3 && in.trim_side != 5)
        return bdx_fail(BDX_ERR_INVALID, "trim_side must be 3 or 5");  // core.jl:308-313
    if (p.has_nindel && !in.lengths_no_n)
        return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": lengths_no_n required with nindel");
    D.n_bc = in.n_barcodes;
    D.trim_side = in.trim_side;
    int rc;
    if ((rc = narrow_range(in.ref_search_range, D.rs, name))) return rc;
    if ((rc = narrow_range(in.barcode_start_range, D.bs, name))) return rc;
    if ((rc = narrow_range(in.barcode_end_range, D.be, name))) return rc;
    if (in.offsets[0] != 0) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": offsets[0] must be 0");
    hs.off.assign(in.offsets, in.offsets + in.n_barcodes + 1);
    D.max_m = 0;
    hs.min_m = kMaxBarcodeLen;
    for (int b = 0; b < D.n_bc; b++) {
        const int m = hs.off[b + 1] - hs.off[b];
        if (m <= 0) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": empty barcode (not supported)");
        if (m > kMaxBarcodeLen) return bdx_fail(BDX_ERR_INVALID, std::string(name) + ": barcode longer than 256");
        D.max_m = std::max(D.max_m, m);
        hs.min_m = std::min(hs.min_m, m);
    }
    hs.bytes.assign(in.bytes, in.bytes + hs.off[D.n_bc]);
    hs.norm.resize(D.n_bc);
    for (int b = 0; b < D.n_bc; b++) {
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
    build_filter_tables(p, hs, D, debug);
    build_prefilter(p, hs, D, debug);
    build_seed_levels(p, hs, D, debug);
    build_seed_deep(hs, D, debug);
    build_seed_var(p, hs, D, debug);
    build_hamming_packed(p, hs, D, debug);
    return BDX_OK;
}

// Text description of the tables built for one barcode set (bdx_config_describe): which shortcut stages exist and
// with which parameters.  Host data only.
std::string bdx_describe_set(const HostSet &hs, const DevSet &D)
{
    char line[256];
    std::string out;
    snprintf(line, sizeof line, "set: barcodes=%d length=%d..%d classes=%d words=%d filter=%d\n", D.n_bc, hs.min_m, D.max_m,
             D.n_classes - 1, D.words, D.use_filter);
    out += line;
    if (D.pf_enabled) {
        snprintf(line, sizeof line, "prefilter: seed=%d log2=%d bitmap_log2=%d\n", D.pf_seed, D.pf_log2, D.pf_bm_log2);
        out += line;
    }
    for (int l = 0; l < D.sd_levels; l++) {
        snprintf(line, sizeof line, "k_seed level %d: K=%d q=%d entries=%d max_hits=%d\n", l + 1, D.sd[l].k, D.sd[l].q,
                 D.sd[l].n_entries, D.sd[l].max_hits);
        out += line;
    }
    for (int l = 0; l < D.sdd_n; l++) {
        snprintf(line, sizeof line, "k_seed_deep table %d: K=%d q=%d entries=%d\n", l + 1, D.sdd_k, D.sdd[l].q, D.sdd[l].n_entries);
        out += line;
    }
    for (int l = 0; l < D.sv_levels; l++) {
        const SeedVar &V = D.sv[l];
        int k_lo = 255, k_hi = 0;
        for (uint8_t k : hs.sv[l].kdepth) {
            k_lo = std::min<int>(k_lo, k);
            k_hi = std::max<int>(k_hi, k);
        }
        snprintf(line, sizeof line, "k_seed_var level %d: q=%d q2=%d K=%d..%d complete=%d entries=%d group_reads=%d hit_rows=%d qgram_filter=%d\n",
                 l + 1, V.q, V.q2, hs.sv[l].kdepth.empty() ? 0 : k_lo, k_hi, V.complete, V.n_entries, V.group_reads, V.hit_rows,
                 V.qgram_filter);
        out += line;
    }
    if (D.hp.enabled) {
        snprintf(line, sizeof line, "k_hamming_scan: m=%d allowed=%d segments=%d\n", D.hp.m, D.hp.allowed, D.hp.n_seg);
        out += line;
    }
    return out;
}
