// plan.cu -- which kernels run for a pass, on which reads and in which order: the routing policy of the library
// (DESIGN.md section 4).  Host code only; the kernel files contribute their shared-memory layout arithmetic.
#include "api_internal.h"

// Shared-memory budgets of the shortcut stages: a stage whose launch would need more is left out, and the reads go
// on to the next one.  Below the opt-in limit on purpose: each keeps its kernel at a useful occupancy.
constexpr size_t kHammingScanSmemBudget = 200 * 1024;
constexpr size_t kSeedSmemBudget = 110 * 1024;
constexpr size_t kSeedDeepSmemBudget = 96 * 1024;
constexpr size_t kSeedVarSmemBudget = 160 * 1024;

// the reference's default barcode start / end ranges: every alignment may start and end anywhere in the read
static bool default_geometry(const DevSet &S)
{
    const DevRange &bs = S.bs, &be = S.be;
    return bs.start_off <= 1 && !bs.start_from_end && bs.end_from_end && bs.end_off >= 0 && be.start_off <= 1 &&
           !be.start_from_end;
}

PassPlan plan_pass(const DevParams &P, int pass)
{
    const DevSet &S = P.set[pass];
    PassPlan plan;
    int wl = kWlNone;   // the worklist that holds the reads the steps so far left open
    auto add = [&](int kind, int stage, int level = 0, int out = kWlNone, int reads = kLitAll) {
        plan.step[plan.n++] = PlanStep{(uint8_t)kind, (uint8_t)level, (uint8_t)wl, (uint8_t)out, (uint8_t)reads, (uint8_t)stage};
        if (out != kWlNone) wl = out;
    };
    // the seed stages hand the reads they cannot finish from one worklist to the other
    auto next_wl = [&] { return wl == kWlWork2 ? kWlWork : kWlWork2; };
    auto literal = [&](int reads) { add(kStepLiteral, kStLiteral, 0, kWlNone, reads); };

    if (P.algo == BDX_HAMMING && S.hp.enabled && hamming_scan_smem(S) <= kHammingScanSmemBudget) {
        // :hamming -- packed pigeonhole scan over every start position, then the literal rules on the candidates
        add(kStepHammingScan, kStHamming);
        literal(kLitCand);
        return plan;
    }
    if (P.algo == BDX_EXACT && S.use_filter && S.pf_enabled && P.max_error_rate >= 0.0) {
        // :exact -- rolling-hash candidate generation (k_prefilter<1>) instead of the Shift-And filter kernel, then
        // the literal rules on the candidates
        add(kStepPrefilter, kStPrefilter);
        literal(kLitCand);
        return plan;
    }
    if (S.words == 0) {   // no filter tables (exotic costs, barcodes > 64 nt): k_literal over every barcode
        literal(kLitAll);
        return plan;
    }
    plan.clear_lit = true;
    // k_prefilter where every read in the exact regime may be resolved by it; without it in front (min_delta != 0)
    // the first seed stage takes every read of the batch.  :hamming produces positions, so trim / stats are fine
    // (no wildcard rows).  :semiglobal with trimming / stats: a verbatim occurrence has the positions (k_prefilter),
    // a seed-resolved read gets them from k_literal run on its single winning barcode.  Any positive edit costs will
    // do (match = 0): a verbatim occurrence is the only way to score 0, whatever a mismatch or a gap costs, and
    // score 0 beats every other barcode under the strict "<" of :658.
    if (S.pf_enabled && P.min_delta == 0.0 && P.max_error_rate >= 0.0 &&
        (P.algo == BDX_HAMMING ? S.use_filter : P.algo == BDX_SEMIGLOBAL && P.match == 0 && P.mismatch >= 1 && P.indel >= 1))
        add(kStepPrefilter, kStPrefilter, 0, kWlWork);
    // k_seed's levels: the exact regime of k_filter (unit costs, uniform length, no wildcard rows: the tables exist
    // only then); min_delta is handled, trimming / stats go through k_literal for the positions
    const bool seeds = P.algo == BDX_SEMIGLOBAL && P.unit_costs && P.max_error_rate >= 0.0;
    int levels = seeds && S.pf_enabled ? S.sd_levels : 0;
    for (int l = 0; l < levels; l++)
        if (seed_smem(S, S.sd[l]) > kSeedSmemBudget) levels = 0;
    // k_seed_var's levels serve score-only passes: in place of k_seed's levels where those do not apply (barcodes of
    // different lengths) or would refuse every read (constrained start / end), else its complete level behind them
    const bool sv = seeds && S.sv_levels >= 1 && S.trim_side == 0 && !P.want_stats;
    int sv_levels = 0;
    if (sv && !(levels > 0 && default_geometry(S) && !(P.debug & BDX_DEBUG_PREFER_SEED_VAR)))
        while (sv_levels < S.sv_levels && seed_var_smem(S, S.sv[sv_levels]) <= kSeedVarSmemBudget) sv_levels++;
    for (int l = 0; l < sv_levels; l++) add(kStepSeedVar, l == 0 ? kStSeed : kStSeedDeep, l, next_wl());
    if (sv_levels == 0 && levels > 0) {
        for (int l = 0; l < levels; l++) add(kStepSeed, kStSeed, l, next_wl());
        const int tail = S.sv_levels - 1;
        if (sv && S.sv[tail].complete && seed_var_smem(S, S.sv[tail]) <= kSeedVarSmemBudget)
            // its verdicts are final (best barcode at the allowed distance, or none at all): k_filter sees only the
            // reads it hands on (hit-list overflow)
            add(kStepSeedVar, kStSeedDeep, tail, next_wl());
        else if (S.sdd_n > 0 && P.min_delta == 0.0 && deep_smem(S) <= kSeedDeepSmemBudget)
            add(kStepSeedDeep, kStSeedDeep, 0, next_wl());   // keeps no runner-up: min_delta = 0 only
    }
    if (!S.use_filter) {
        // tiny set: no filter kernel.  What the shortcut stages left goes to k_literal over every barcode.
        if (wl == kWlNone) {
            literal(kLitAll);
        } else {
            add(kStepMarkPending, kStOther);
            // seed winners (windowed) and the scan-everything rest as separate, compacted launches
            literal(kLitWin);
            literal(kLitRest);
        }
        return plan;
    }
    add(kStepFilter, kStFilter);
    // the exact regime finishes inside the filter kernel; anything else leaves kBcPending reads with candidate
    // lists for the literal kernel
    if (!(P.algo == BDX_SEMIGLOBAL && P.unit_costs && S.trim_side == 0 && !P.want_stats && default_geometry(S))) {
        // seed winners (windowed DP) and k_filter's candidate reads as separate, compacted launches: a warp costs
        // as much as its most expensive lane
        if (wl != kWlNone && levels > 0) literal(kLitWin);
        literal(kLitFull);
    }
    return plan;
}

std::string plan_text(const PassPlan &plan)
{
    static const char *const kernel[] = {"k_hamming_scan", "k_prefilter", "k_seed", "k_seed_var", "k_seed_deep",
                                         "k_filter", "k_mark_pending", "k_literal"};
    static const char *const reads[] = {"@all", "@cand", "@win", "@full", "@rest"};
    std::string out;
    for (int i = 0; i < plan.n; i++) {
        const PlanStep &t = plan.step[i];
        out += std::string(i ? "," : "") + kernel[t.kind];
        if (t.kind == kStepSeed || t.kind == kStepSeedVar) out += "@" + std::to_string(t.level + 1);
        if (t.kind == kStepLiteral) out += reads[t.reads];
    }
    return out;
}
