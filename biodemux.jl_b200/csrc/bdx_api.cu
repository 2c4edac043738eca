// bdx_api.cu -- C ABI of libbdx (include/bdx.h): configuration, per-worker streams with
// pinned double-buffered staging, batch submission / retrieval, DemuxStats counters.
// Replaces the body of the reference's worker_task (src/core.jl:226-279).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "api_internal.h"
#include "literal.cuh"

using namespace bdx;

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local std::string g_err;

std::string &bdx_error_text() { return g_err; }
int bdx_fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}
int bdx_cuda_fail(cudaError_t e, const char *what)
{
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return BDX_ERR_CUDA;
}
static int fail(int code, const std::string &msg) { return bdx_fail(code, msg); }
static int cuda_fail(cudaError_t e, const char *what) { return bdx_cuda_fail(e, what); }

extern "C" const char *bdx_last_error(void) { return g_err.c_str(); }
extern "C" int bdx_abi_version(void) { return BDX_ABI_VERSION; }
extern "C" int bdx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---------------------------------------------------------------------------
// configuration
// ---------------------------------------------------------------------------
extern "C" int bdx_config_create(const bdx_params *p, bdx_config **out) { return bdx_config_create_debug(p, 0u, out); }

extern "C" int bdx_config_create_debug(const bdx_params *p, uint32_t debug, bdx_config **out)
{
    if (!p || !out) return fail(BDX_ERR_INVALID, "null argument");
    *out = nullptr;
    if (p->struct_size != sizeof(bdx_params) || p->abi_version != BDX_ABI_VERSION)
        return fail(BDX_ERR_INVALID, "bdx_params: struct_size / abi_version mismatch");
    if (p->algorithm < BDX_SEMIGLOBAL || p->algorithm > BDX_EXACT) return fail(BDX_ERR_INVALID, "unknown algorithm");
    const int64_t costs[4] = {p->match, p->mismatch, p->indel, p->has_nindel ? p->nindel : 1};
    for (int64_t c : costs)
        if (c > kMaxCost || c < -kMaxCost) return fail(BDX_ERR_INVALID, "cost magnitude above 2^20");
    if (p->algorithm == BDX_SEMIGLOBAL && (p->indel == 0 || (p->has_nindel && p->nindel == 0)))
        return fail(BDX_ERR_INVALID, "zero gap cost (the reference raises DivideError, classification.jl:170-176)");
    if (std::isnan(p->max_error_rate) || std::isnan(p->min_delta)) return fail(BDX_ERR_INVALID, "NaN option");

    bdx_config *cfg = new (std::nothrow) bdx_config();
    if (!cfg) return fail(BDX_ERR_NOMEM, "out of memory");
    cfg->debug = debug;
    DevParams &P = cfg->base;
    int rc = bdx_build_set(*p, p->set1, cfg->set[0], P.set[0], debug, "set1");
    if (rc == BDX_OK && p->is_dual) rc = bdx_build_set(*p, p->set2, cfg->set[1], P.set[1], debug, "set2");
    if (rc != BDX_OK) {
        delete cfg;
        return rc;
    }
    {   // 4-bit codes of the packed input: the distinct barcode bytes of both sets, in order of first appearance
        int n_codes = 1;
        bool used[256] = {};
        for (int k = 0; k < (p->is_dual ? 2 : 1) && n_codes; k++)
            for (uint8_t b : cfg->set[k].bytes)
                if (!cfg->code_of[b]) {
                    if (n_codes == 16) {                 // too many distinct bytes: no packed input for this config
                        n_codes = 0;
                        memset(cfg->code_of, 0, sizeof(cfg->code_of));
                        break;
                    }
                    cfg->code_of[b] = (uint8_t)n_codes;
                    cfg->rep_of[n_codes++] = b;
                    used[b] = true;
                }
        cfg->n_codes = n_codes;
        for (int b = 0; b < 256 && n_codes; b++)
            if (!used[b]) {                              // code 0 expands to a byte that is in no barcode
                cfg->rep_of[0] = (uint8_t)b;
                break;
            }
    }
    P.max_error_rate = p->max_error_rate;
    P.min_delta = p->min_delta;
    P.match = (int)p->match;
    P.mismatch = (int)p->mismatch;
    P.indel = (int)p->indel;
    P.nindel = p->has_nindel ? (int)p->nindel : 0;
    P.has_n = p->has_nindel ? 1 : 0;
    P.algo = p->algorithm;
    P.is_dual = p->is_dual ? 1 : 0;
    P.want_stats = p->want_stats ? 1 : 0;
    P.two = 2;
    P.debug = (int)debug;
    P.unit_costs = p->match == 0 && p->mismatch == 1 && p->indel == 1 && (!p->has_nindel || p->nindel == 1);

    // stats layout (classification.jl:736-758)
    bdx_stats_layout &L = cfg->lay;
    const int b1 = P.set[0].n_bc, b2 = p->is_dual ? P.set[1].n_bc : 0;
    const int max_m = std::max(P.set[0].max_m, p->is_dual ? P.set[1].max_m : 0);
    int max_allowed = 0;
    for (int s = 0; s < (p->is_dual ? 2 : 1); s++)
        for (int b = 0; b < P.set[s].n_bc; b++) max_allowed = std::max(max_allowed, cfg->set[s].allowed0[b]);
    L.b1 = b1;
    L.b2 = b2;
    L.pos_bias = max_m;
    L.pos_bins = 1024 + max_m + 2;
    // e - s + 1 with s >= 1 - m (origin labels of the init column, classification.jl:281) and e <= n
    L.len_bins = 1024 + max_m + 2;
    L.dist_bias = (int)std::min<int64_t>(std::max<int64_t>(0, -p->match) * max_m, 4096);
    L.dist_bins = L.dist_bias + std::min(std::max(max_allowed, 0), 4095) + 1;
    int64_t o = 4;
    L.sample_off = o;
    o += (int64_t)(b1 + 1) * (b2 + 1);
    const int bsz[2] = {b1, b2};
    for (int s = 0; s < 2; s++) {
        L.pos_off[s] = o;
        o += (int64_t)(bsz[s] + 1) * L.pos_bins;
        L.len_off[s] = o;
        o += (int64_t)(bsz[s] + 1) * L.len_bins;
        L.dist_off[s] = o;
        o += (int64_t)(bsz[s] + 1) * L.dist_bins;
    }
    L.total_len = o;
    *out = cfg;
    return BDX_OK;
}

static void free_tables(DeviceTables *t)
{
    for (void *p : t->allocs) cudaFree(p);
    delete t;
}

extern "C" void bdx_config_destroy(bdx_config *cfg)
{
    if (!cfg) return;
    for (auto &kv : cfg->per_device) {
        cudaSetDevice(kv.first);
        free_tables(kv.second);
    }
    delete cfg;
}

template <typename T>
static cudaError_t upload(DeviceTables *t, const std::vector<T> &v, const T **out)
{
    *out = nullptr;
    if (v.empty()) return cudaSuccess;
    void *d = nullptr;
    cudaError_t e = cudaMalloc(&d, v.size() * sizeof(T));
    if (e != cudaSuccess) return e;
    t->allocs.push_back(d);
    e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = (const T *)d;
    return e;
}

// sharedMemPerBlockOptin of sm_100 (227 KB); the library runs on no other architecture
constexpr size_t kSm100SmemOptin = 232448;

// A config's device parameter block without the table pointers, with the stages whose shared memory would exceed
// `smem_optin` switched off: what plan_pass decides by, on a device (get_tables) or for sm_100 (bdx_config_describe).
static DevParams host_params(const bdx_config &cfg, size_t smem_optin)
{
    DevParams P = cfg.base;
    for (int s = 0; s < (P.is_dual ? 2 : 1); s++) {
        DevSet &D = P.set[s];
        // shared-memory footprints against the opt-in limit: the prefilter's hash table and bitmap (large sets of
        // short barcodes), then the filter kernel's Peq planes
        if (D.pf_enabled && prefilter_smem_bytes(D) > smem_optin) {
            D.pf_enabled = 0;   // k_prefilter and the k_seed levels behind it are skipped; k_filter takes every read
            D.sd_levels = 0;
            D.sdd_n = 0;
        }
        if (D.words && filter_smem_bytes(D) > smem_optin) {
            D.words = 0;
            D.use_filter = 0;
            D.pf_enabled = 0;
            D.sd_levels = 0;
            D.sdd_n = 0;
            D.sv_levels = 0;
        }
    }
    return P;
}

static int get_tables(bdx_config *cfg, int device, DeviceTables **out)
{
    std::lock_guard<std::mutex> lk(cfg->mu);
    auto it = cfg->per_device.find(device);
    if (it != cfg->per_device.end()) {
        *out = it->second;
        return BDX_OK;
    }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(BDX_ERR_CUDA, "libbdx is built for sm_100a only; device compute capability too low");
    DeviceTables *t = new DeviceTables();
    t->P = host_params(*cfg, prop.sharedMemPerBlockOptin);
    t->sm_count = prop.multiProcessorCount;
    const int passes = t->P.is_dual ? 2 : 1;
    // every table of a set, paired with the DevSet pointer its device copy goes to; a level that was not built has
    // empty vectors and keeps a null pointer.  Nothing is uploaded after the first error.
    cudaError_t e = cudaSuccess;
    auto up = [&](const auto &v, auto &dev) {
        if (e == cudaSuccess) e = upload(t, v, &dev);
    };
    for (int s = 0; s < passes; s++) {
        const HostSet &hs = cfg->set[s];
        DevSet &D = t->P.set[s];
        up(hs.bytes, D.bc_bytes);
        up(hs.off, D.bc_off);
        up(hs.norm, D.norm);
        up(hs.peq, D.peq);
        up(hs.filt_allowed, D.filt_allowed);
        up(hs.allowed0, D.allowed0);
        up(hs.class_of, D.class_of);
        up(hs.pf_bitmap, D.pf_bitmap);
        up(hs.pf_keys, D.pf_keys);
        up(hs.pf_vals, D.pf_vals);
        up(hs.bc_cls, D.bc_cls);
        auto level = [&](const HostSet::HostSeedLevel &H, SeedLevel &L) {
            up(H.bstart, L.bstart);
            up(H.entries, L.entries);
            up(H.ekeys, L.ekeys);
            up(H.bitmap, L.bitmap);
        };
        for (int l = 0; l < 2; l++) level(hs.sd[l], D.sd[l]);
        for (int l = 0; l < 2; l++) level(hs.sdd[l], D.sdd[l]);
        for (int l = 0; l < 2; l++) {
            up(hs.sv[l].bstart, D.sv[l].bstart);
            up(hs.sv[l].entries, D.sv[l].entries);
            up(hs.sv[l].kdepth, D.sv[l].kdepth);
        }
        up(hs.hp_bstart, D.hp.bstart);
        up(hs.hp_entries, D.hp.entries);
        up(hs.hp_bcw, D.hp.bcw);
    }
    if (e != cudaSuccess) {
        free_tables(t);
        return cuda_fail(e, "uploading barcode tables");
    }
    for (int pass = 0; pass < passes; pass++) t->plan[pass] = plan_pass(t->P, pass);
    cfg->per_device[device] = t;
    *out = t;
    return BDX_OK;
}

// ---------------------------------------------------------------------------
// streams
// ---------------------------------------------------------------------------
void bdx_stream_drop_graphs(bdx_stream *s)
{
    for (Slot &sl : s->slot)
        if (sl.graph) {
            cudaGraphExecDestroy(sl.graph);
            sl.graph = nullptr;
            sl.graph_n = -1;
        }
}

static void free_scratch(Scratch &sc)
{
    cudaFree(sc.pass[0]);
    cudaFree(sc.pass[1]);
    cudaFree(sc.cand);
    cudaFree(sc.cand_cnt);
    cudaFree(sc.worklist);
    cudaFree(sc.n_work);
    cudaFree(sc.worklist2);
    cudaFree(sc.n_work2);
    cudaFree(sc.wl_win);
    cudaFree(sc.wl_full);
    cudaFree(sc.n_lit);
    sc = Scratch{};
}

static int ensure_scratch(bdx_stream *s, int64_t n)
{
    if (n <= s->sc_cap) return BDX_OK;
    // in-order on the compute stream: earlier kernels still own the old buffers
    CU(cudaStreamSynchronize(s->st_comp));
    bdx_stream_drop_graphs(s);      // captured launches hold the old scratch pointers
    free_scratch(s->sc);
    s->sc_cap = 0;
    const int64_t cap = n + n / 8 + 1024;
    CU(cudaMalloc(&s->sc.pass[0], cap * sizeof(PassOut)));
    CU(cudaMalloc(&s->sc.pass[1], cap * sizeof(PassOut)));
    CU(cudaMalloc(&s->sc.cand, cap * kCandMax * sizeof(uint16_t)));
    CU(cudaMalloc(&s->sc.cand_cnt, cap));
    CU(cudaMalloc(&s->sc.worklist, cap * sizeof(int)));
    CU(cudaMalloc(&s->sc.n_work, sizeof(int)));
    CU(cudaMalloc(&s->sc.worklist2, cap * sizeof(int)));
    CU(cudaMalloc(&s->sc.n_work2, sizeof(int)));
    CU(cudaMalloc(&s->sc.wl_win, cap * sizeof(int)));
    CU(cudaMalloc(&s->sc.wl_full, cap * sizeof(int)));
    CU(cudaMalloc(&s->sc.n_lit, 2 * sizeof(int)));
    s->sc_cap = cap;
    return BDX_OK;
}

// every buffer, event and graph of a slot: whatever stream_create_impl or ensure_input_buffers allocated
static void free_slot(Slot &sl)
{
    cudaFreeHost(sl.h_seq);
    cudaFreeHost(sl.h_off);
    cudaFreeHost(sl.h_res);
    cudaFreeHost(sl.h_det);
    cudaFree(sl.d_packed);
    cudaFreeHost(sl.h_packed);
    cudaFree(sl.d_win);
    cudaFree(sl.d_win_off);
    cudaFreeHost(sl.h_win_off);
    cudaFree(sl.d_seq);
    cudaFree(sl.d_off);
    cudaFree(sl.d_res);
    cudaFree(sl.d_det);
    if (sl.ev_h2d) cudaEventDestroy(sl.ev_h2d);
    if (sl.ev_kern) cudaEventDestroy(sl.ev_kern);
    if (sl.ev_done) cudaEventDestroy(sl.ev_done);
    if (sl.graph) cudaGraphExecDestroy(sl.graph);
}

extern "C" void bdx_stream_destroy(bdx_stream *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->st_comp) cudaStreamSynchronize(s->st_comp);
    if (s->st_copy) cudaStreamSynchronize(s->st_copy);
    if (s->st_d2h) cudaStreamSynchronize(s->st_d2h);
    for (Slot &sl : s->slot) free_slot(sl);
    free_scratch(s->sc);
    cudaFree(s->d_stats);
    cudaFree(s->d_ovf);
    cudaFree(s->d_n_ovf);
    cudaFree(s->d_counters);
    demux_state_destroy(s->demux);
    for (auto &pr : s->prof_events) {
        cudaEventDestroy(pr.e0);
        cudaEventDestroy(pr.e1);
    }
    if (s->st_copy) cudaStreamDestroy(s->st_copy);
    if (s->st_comp) cudaStreamDestroy(s->st_comp);
    if (s->st_d2h) cudaStreamDestroy(s->st_d2h);
    delete s;
}

static int stream_create_impl(bdx_stream *s)
{
    CU(cudaSetDevice(s->device));
    CU(cudaStreamCreateWithFlags(&s->st_copy, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&s->st_comp, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&s->st_d2h, cudaStreamNonBlocking));
    if (s->max_reads > 0) {
        for (Slot &sl : s->slot) {
            CU(cudaHostAlloc(&sl.h_res, (size_t)s->max_reads * sizeof(bdx_result), cudaHostAllocDefault));
            CU(cudaHostAlloc(&sl.h_det, (size_t)s->max_reads * 2 * sizeof(bdx_pass_detail), cudaHostAllocDefault));
            CU(cudaMalloc(&sl.d_seq, (size_t)std::max<int64_t>(s->max_bytes, 16) + 32));   // (+ slack: k_unpack4 stores 16-byte vectors)
            CU(cudaMalloc(&sl.d_off, ((size_t)s->max_reads + 1) * 4));
            CU(cudaMalloc(&sl.d_res, (size_t)s->max_reads * sizeof(bdx_result)));
            CU(cudaMalloc(&sl.d_det, (size_t)s->max_reads * 2 * sizeof(bdx_pass_detail)));
            CU(cudaEventCreateWithFlags(&sl.ev_h2d, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&sl.ev_kern, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
        }
        int rc = ensure_scratch(s, s->max_reads);
        if (rc) return rc;
    }
    CU(cudaMalloc(&s->d_counters, 12 * sizeof(unsigned long long)));
    CU(cudaMemset(s->d_counters, 0, 12 * sizeof(unsigned long long)));
    if (s->cfg->base.want_stats) {
        CU(cudaMalloc(&s->d_stats, (size_t)s->cfg->lay.total_len * 8));
        CU(cudaMemset(s->d_stats, 0, (size_t)s->cfg->lay.total_len * 8));
        CU(cudaMalloc(&s->d_ovf, (size_t)kStatsOvfCap * sizeof(bdx_stats_overflow)));
        s->ovf_cap = kStatsOvfCap;
        CU(cudaMalloc(&s->d_n_ovf, 2 * sizeof(unsigned int)));
        CU(cudaMemset(s->d_n_ovf, 0, 2 * sizeof(unsigned int)));
    }
    return BDX_OK;
}

extern "C" int bdx_stream_create(const bdx_config *cfg_c, int device, int32_t max_reads, int64_t max_bytes,
                                 bdx_stream **out)
{
    if (!cfg_c || !out || max_reads < 0 || max_bytes < 0) return fail(BDX_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (max_bytes > 0x7FFFFFF0ll) return fail(BDX_ERR_TOO_LARGE, "max_bytes must stay below 2^31 (int32 offsets)");
    bdx_config *cfg = const_cast<bdx_config *>(cfg_c);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(BDX_ERR_CUDA, "no CUDA device available (libbdx has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return fail(BDX_ERR_INVALID, "device index out of range");
    DeviceTables *tab = nullptr;
    int rc = get_tables(cfg, device, &tab);
    if (rc) return rc;
    bdx_stream *s = new (std::nothrow) bdx_stream();
    if (!s) return fail(BDX_ERR_NOMEM, "out of memory");
    s->cfg = cfg;
    s->tab = tab;
    s->device = device;
    s->max_reads = max_reads;
    s->max_bytes = max_bytes;
    s->details = cfg->base.want_stats != 0;
    rc = stream_create_impl(s);
    if (rc) {
        std::string keep = g_err;
        bdx_stream_destroy(s);
        g_err = keep;
        return rc;
    }
    *out = s;
    return BDX_OK;
}

extern "C" int bdx_stream_enable_details(bdx_stream *s, int on)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    if (s->in_flight) return fail(BDX_ERR_STATE, "batches in flight");
    s->details = on != 0;
    return BDX_OK;
}

// Enqueue the classification kernels for n reads resident on the device.
int bdx_enqueue_classify(bdx_stream *s, const uint8_t *d_seq, const int32_t *d_off, int32_t n,
                            bdx_result *d_res, bdx_pass_detail *d_det)
{
    if (n == 0) return BDX_OK;
    int rc = ensure_scratch(s, n);
    if (rc) return rc;
    // every kernel launch goes through here: counted, and bracketed by CUDA events while profiling is on
    auto staged = [s](int kind, auto &&launch) -> int {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (s->profile) {
            CU(cudaEventCreate(&e0));
            CU(cudaEventCreate(&e1));
            CU(cudaEventRecord(e0, s->st_comp));
        }
        const cudaError_t e = launch();
        if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
        s->launches++;
        if (s->profile) {
            CU(cudaEventRecord(e1, s->st_comp));
            s->prof_events.push_back(ProfEvent{kind, e0, e1});
        }
        return BDX_OK;
    };
    const DevParams &P = s->tab->P;
    const Scratch &sc = s->sc;
    const int sm = s->tab->sm_count;
    unsigned long long *const ctr = s->d_counters;
    cudaStream_t st = s->st_comp;
    int *const wl[3] = {nullptr, sc.worklist, sc.worklist2}, *const n_wl[3] = {nullptr, sc.n_work, sc.n_work2};
    for (int pass = 0; pass < (P.is_dual ? 2 : 1); pass++) {
        const PassPlan &plan = s->tab->plan[pass];
        if (plan.clear_lit) CU(cudaMemsetAsync(sc.n_lit, 0, 2 * sizeof(int), st));   // k_literal's two read lists
        for (int i = 0; i < plan.n; i++) {
            const PlanStep &t = plan.step[i];
            int *const in = wl[t.in], *const n_in = n_wl[t.in], *const out = wl[t.out], *const n_out = n_wl[t.out];
            const int *const list[5] = {nullptr, nullptr, sc.wl_win, sc.wl_full, in};   // k_literal's read list by t.reads
            const int *const len[5] = {nullptr, nullptr, sc.n_lit, sc.n_lit + 1, n_in};
            if ((rc = staged(t.stage, [&]() -> cudaError_t {
                switch (t.kind) {
                case kStepHammingScan: return launch_hamming_scan(P, pass, d_seq, d_off, n, sc, sm, st);
                case kStepPrefilter: return launch_prefilter(P, pass, d_seq, d_off, n, sc, sm, ctr, st);
                case kStepSeed: return launch_seed(P, pass, t.level, d_seq, d_off, n, sc, in, n_in, out, n_out, sm, ctr, st);
                case kStepSeedVar: return launch_seed_var(P, pass, t.level, d_seq, d_off, n, sc, in, n_in, out, n_out, sm, ctr, st);
                case kStepSeedDeep: return launch_seed_deep(P, pass, d_seq, d_off, n, sc, in, n_in, out, n_out, sm, ctr, st);
                case kStepFilter: return launch_filter(P, pass, d_seq, d_off, n, sc, sm, ctr, in, n_in, st);
                case kStepMarkPending: return launch_mark_pending(P, pass, n, sc, in, n_in, st);
                case kStepLiteral: return launch_literal(P, pass, t.reads != kLitAll, d_seq, d_off, n, sc, st, list[t.reads], len[t.reads]);
                }
                return cudaErrorInvalidValue;
            }))) return rc;
        }
    }
    StatsDev sd{s->d_stats, s->cfg->lay, s->d_ovf, s->d_n_ovf, (unsigned int)std::min<int64_t>(s->ovf_cap, 0xFFFFFFFFll)};
    if ((rc = staged(kStFinalize, [&] { return launch_finalize(P, d_off, n, sc, d_res, d_det, sd, st); }))) return rc;
    return BDX_OK;
}

// The kernels of one staged batch.  Batches up to kGraphMaxReads reads replay a CUDA graph captured on the
// slot's second use with that size (the first use runs plainly and warms the per-kernel launch caches, so the
// capture holds stream operations only); anything else -- other sizes, profiling, a failed capture -- launches
// the kernels one by one.
constexpr int32_t kGraphMaxReads = 100000;

static int enqueue_batch(bdx_stream *s, Slot &sl)
{
    const bool graphs_off = (s->cfg->debug & BDX_DEBUG_NO_GRAPHS) != 0;
    const int32_t n = sl.n;
    bdx_pass_detail *det = s->details ? sl.d_det : nullptr;
    const bool eligible = !graphs_off && s->graphs_ok && !s->profile && n > 0 && n <= kGraphMaxReads;
    if (eligible && sl.graph && sl.graph_n == n && sl.graph_details == s->details) {
        CU(cudaGraphLaunch(sl.graph, s->st_comp));
        s->launches += sl.graph_launches;
        return BDX_OK;
    }
    if (eligible && sl.uses >= 1 && n == s->max_reads) {          // full-size chunks are the ones that repeat
        int rc = ensure_scratch(s, n);                            // allocation is not capturable
        if (rc) return rc;
        if (sl.graph) {
            cudaGraphExecDestroy(sl.graph);
            sl.graph = nullptr;
        }
        const int64_t l0 = s->launches;
        cudaGraph_t g = nullptr;
        bool ok = cudaStreamBeginCapture(s->st_comp, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
        if (ok) {
            rc = bdx_enqueue_classify(s, sl.d_seq, sl.d_off, n, sl.d_res, det);
            const cudaError_t ce = cudaStreamEndCapture(s->st_comp, &g);
            ok = rc == BDX_OK && ce == cudaSuccess && g != nullptr;
        }
        if (ok) ok = cudaGraphInstantiate(&sl.graph, g, 0) == cudaSuccess;
        if (g) cudaGraphDestroy(g);
        if (ok) {
            sl.graph_n = n;
            sl.graph_details = s->details;
            sl.graph_launches = (int)(s->launches - l0);
            s->launches = l0;
            CU(cudaGraphLaunch(sl.graph, s->st_comp));
            s->launches += sl.graph_launches;
            return BDX_OK;
        }
        // capture failed: clear the error state and never try again on this stream
        cudaGetLastError();
        s->launches = l0;
        sl.graph = nullptr;
        s->graphs_ok = false;
    }
    sl.uses++;
    return bdx_enqueue_classify(s, sl.d_seq, sl.d_off, n, sl.d_res, det);
}

// ---- host batches: every bdx_submit* form and bdx_acquire / bdx_commit ----
// A batch as the caller hands it over: seq holds the reads' bytes, or -- packed -- their 4-bit codes (packed.cu);
// windowed, only the bytes (or codes) of the reads' search windows, at offsets win_off (windows.cu).  off: the
// offsets of the full reads.  pinned: the buffers are page-locked and go to the device as they are; otherwise the
// batch is first copied into the slot's pinned staging.
struct BatchInput {
    const uint8_t *seq;
    const int32_t *off;
    const int32_t *win_off;
    bool windows, packed, pinned;
};

// bytes of the batch's input stream, the one that travels to the device
static size_t sent_bytes(const BatchInput &in, int32_t n)
{
    if (!n) return 0;
    const size_t b = (size_t)(in.windows ? in.win_off[n] : in.off[n]);
    return in.packed ? (b + 1) / 2 : b;
}

static int launch_slot(bdx_stream *s, Slot &sl, const BatchInput &in)
{
    const int32_t n = sl.n;
    const size_t bytes = n ? (size_t)in.off[n] : 0, sent = sent_bytes(in, n);
    uint8_t *const d_in = in.packed ? sl.d_packed : in.windows ? sl.d_win : sl.d_seq;
    if (n) {
        CU(cudaMemcpyAsync(sl.d_off, in.off, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, s->st_copy));
        if (in.windows) CU(cudaMemcpyAsync(sl.d_win_off, in.win_off, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, s->st_copy));
        if (sent) CU(cudaMemcpyAsync(d_in, in.seq, sent, cudaMemcpyHostToDevice, s->st_copy));
    }
    CU(cudaEventRecord(sl.ev_h2d, s->st_copy));
    CU(cudaStreamWaitEvent(s->st_comp, sl.ev_h2d, 0));
    if (in.windows && bytes) {
        CU(launch_expand_windows(d_in, in.packed, sl.d_win_off, sl.d_off, sl.d_seq, n, (long long)bytes, s->tab->P,
                                 s->cfg->rep_of, s->tab->sm_count, s->st_comp));
        s->launches++;
    } else if (in.packed && bytes) {
        CU(launch_unpack4(sl.d_packed, sl.d_seq, sl.d_off, n, (long long)bytes, s->cfg->rep_of, s->tab->sm_count, s->st_comp));
        s->launches++;
    }
    int rc = enqueue_batch(s, sl);
    if (rc) return rc;
    CU(cudaEventRecord(sl.ev_kern, s->st_comp));
    CU(cudaStreamWaitEvent(s->st_d2h, sl.ev_kern, 0));
    if (n) {
        CU(cudaMemcpyAsync(sl.h_res, sl.d_res, (size_t)n * sizeof(bdx_result), cudaMemcpyDeviceToHost, s->st_d2h));
        if (s->details)
            CU(cudaMemcpyAsync(sl.h_det, sl.d_det, (size_t)n * 2 * sizeof(bdx_pass_detail),
                               cudaMemcpyDeviceToHost, s->st_d2h));
    }
    CU(cudaEventRecord(sl.ev_done, s->st_d2h));
    sl.busy = true;
    s->head = (s->head + 1) % BDX_MAX_IN_FLIGHT;
    s->in_flight++;
    return BDX_OK;
}

// The input buffers of every slot that a batch form needs beyond those each stream has, allocated lazily on the
// form's first batch: the device copy of packed codes or of window bytes (packed windows expand from d_packed) and
// the window offsets; staged (the caller's buffers are not pinned): the pinned host staging of each.
static int ensure_input_buffers(bdx_stream *s, bool packed, bool windows, bool staged)
{
    const size_t seq_cap = (size_t)std::max<int64_t>(s->max_bytes, 16), code_cap = seq_cap / 2 + 32;
    const size_t off_cap = ((size_t)s->max_reads + 1) * 4;
    for (Slot &sl : s->slot) {
        if (packed && !sl.d_packed) CU(cudaMalloc(&sl.d_packed, code_cap));
        if (windows && !packed && !sl.d_win) CU(cudaMalloc(&sl.d_win, seq_cap));
        if (windows && !sl.d_win_off) CU(cudaMalloc(&sl.d_win_off, off_cap));
        if (!staged) continue;
        if (packed && !sl.h_packed) CU(cudaHostAlloc(&sl.h_packed, code_cap, cudaHostAllocDefault));
        if (!packed && !sl.h_seq) CU(cudaHostAlloc(&sl.h_seq, seq_cap, cudaHostAllocDefault));
        if (!sl.h_off) CU(cudaHostAlloc(&sl.h_off, off_cap, cudaHostAllocDefault));
        if (windows && !sl.h_win_off) CU(cudaHostAlloc(&sl.h_win_off, off_cap, cudaHostAllocDefault));
    }
    return BDX_OK;
}

// Whether the stream can take a new batch now; `pending` is the refusal while a bdx_acquire awaits its bdx_commit.
static int check_stream(const bdx_stream *s, const char *pending)
{
    if (s->max_reads <= 0) return fail(BDX_ERR_STATE, "stream has no staging (max_reads = 0)");
    if (s->acquired) return fail(BDX_ERR_STATE, pending);
    if (s->in_flight >= BDX_MAX_IN_FLIGHT) return fail(BDX_ERR_STATE, "BDX_MAX_IN_FLIGHT batches already in flight; call bdx_fetch");
    return BDX_OK;
}

// Validates a host batch before anything is enqueued: sizes against the stream's staging, offsets non-decreasing
// (a decreasing pair would be a negative read length on the device).  One branch-free pass over the offsets also
// yields the longest read, which tells the DemuxStats overflow list how much room the batch can need.
static int check_batch(const bdx_stream *s, const int32_t *offsets, int32_t n, int32_t *max_len)
{
    if (n < 0) return fail(BDX_ERR_INVALID, "negative n_reads");
    if (n > s->max_reads) return fail(BDX_ERR_TOO_LARGE, "batch exceeds max_reads of the stream");
    if (n && offsets[0] != 0) return fail(BDX_ERR_INVALID, "offsets[0] must be 0");
    if (n && (offsets[n] < 0 || (int64_t)offsets[n] > s->max_bytes))
        return fail(BDX_ERR_TOO_LARGE, "batch exceeds max_bytes of the stream");
    int32_t min_len = 0;
    *max_len = 0;
    for (int32_t i = 0; i < n; i++) {
        const int32_t len = offsets[i + 1] - offsets[i];
        min_len = std::min(min_len, len);
        *max_len = std::max(*max_len, len);
    }
    if (min_len < 0) return fail(BDX_ERR_INVALID, "offsets must be non-decreasing");
    return BDX_OK;
}

// The device trusts win_off: every read's window length is checked against the rule here.
static int check_windows(const bdx_stream *s, const BatchInput &in, int32_t n)
{
    if (n && in.win_off[0] != 0) return fail(BDX_ERR_INVALID, "win_offsets[0] must be 0");
    int32_t last_n = -1, len = 0;
    for (int32_t i = 0; i < n; i++) {
        int sp[4];
        if (in.off[i + 1] - in.off[i] != last_n) len = read_windows(s->tab->P, last_n = in.off[i + 1] - in.off[i], sp);
        if (in.win_off[i + 1] - in.win_off[i] != len)
            return fail(BDX_ERR_INVALID, "win_offsets do not match the search windows of the read lengths (first bad read: " +
                                         std::to_string(i) + ")");
    }
    if (n && in.win_off[n] > 0 && !in.seq) return fail(BDX_ERR_INVALID, "null argument");
    return BDX_OK;
}

// A batch from its validation on (bdx_commit starts here): checks, then DemuxStats overflow room -- so a refused
// batch leaves the stream as it was -- then the form's buffers, the copy into pinned staging and the launch.
static int stage_batch(bdx_stream *s, const BatchInput &in, int32_t n, uint64_t tag)
{
    int32_t max_len = 0;
    int rc = check_batch(s, in.off, n, &max_len);
    if (!rc && in.windows) rc = check_windows(s, in, n);
    if (!rc) rc = bdx_stats_reserve_overflow(s, n, max_len);
    if (rc) return rc;
    s->acquired = false;            // a committed bdx_acquire: its staging now holds this batch
    CU(cudaSetDevice(s->device));
    if ((rc = ensure_input_buffers(s, in.packed, in.windows, !in.pinned))) return rc;
    Slot &sl = s->slot[s->head];
    sl.n = n;
    sl.tag = tag;
    if (in.pinned) return launch_slot(s, sl, in);
    uint8_t *const h_in = in.packed ? sl.h_packed : sl.h_seq;
    if (n) {
        memcpy(sl.h_off, in.off, ((size_t)n + 1) * 4);
        if (in.windows) memcpy(sl.h_win_off, in.win_off, ((size_t)n + 1) * 4);
        if (const size_t b = sent_bytes(in, n)) memcpy(h_in, in.seq, b);
    }
    return launch_slot(s, sl, {h_in, sl.h_off, sl.h_win_off, in.windows, in.packed, true});
}

static const char kNoPackedInput[] = "more than 15 distinct barcode bytes: no 4-bit packed input for this config";

static int submit_batch(bdx_stream *s, const BatchInput &in, int32_t n, uint64_t tag)
{
    if (!s || (n > 0 && (!in.off || (in.windows ? !in.win_off : !in.seq)))) return fail(BDX_ERR_INVALID, "null argument");
    if (in.packed && !s->cfg->n_codes) return fail(BDX_ERR_INVALID, kNoPackedInput);
    const int rc = check_stream(s, "bdx_acquire pending; call bdx_commit");
    return rc ? rc : stage_batch(s, in, n, tag);
}

extern "C" int bdx_submit(bdx_stream *s, const uint8_t *seq, const int32_t *offsets, int32_t n, uint64_t tag)
{
    return submit_batch(s, {seq, offsets, nullptr, false, false, false}, n, tag);
}

extern "C" int bdx_submit_pinned(bdx_stream *s, const uint8_t *seq, const int32_t *offsets, int32_t n,
                                 uint64_t tag)
{
    return submit_batch(s, {seq, offsets, nullptr, false, false, true}, n, tag);
}

// ---- 4-bit packed input ----
void bdx_pack4_bytes(const uint8_t code[256], const uint8_t *in, int64_t n, uint8_t *out);   // pack.cpp

extern "C" int bdx_config_code_table(const bdx_config *cfg, uint8_t table[256])
{
    if (!cfg || !table) return fail(BDX_ERR_INVALID, "null argument");
    if (!cfg->n_codes) return fail(BDX_ERR_INVALID, kNoPackedInput);
    memcpy(table, cfg->code_of, 256);
    return cfg->n_codes;
}

extern "C" int bdx_config_describe(const bdx_config *cfg, int pass, char *buf, int len)
{
    if (!cfg || pass < 0 || pass > 1 || len < 0 || (len > 0 && !buf)) return fail(BDX_ERR_INVALID, "bad argument");
    std::string text;
    if (cfg->base.set[pass].n_bc)
        text = bdx_describe_set(cfg->set[pass], cfg->base.set[pass]) + "plan: steps=" +
               plan_text(plan_pass(host_params(*cfg, kSm100SmemOptin), pass)) + "\n";
    if (len > 0) {
        const size_t k = std::min(text.size(), (size_t)len - 1);
        memcpy(buf, text.data(), k);
        buf[k] = 0;
    }
    return (int)text.size();
}

extern "C" int bdx_pack_reads4(const bdx_config *cfg, const uint8_t *seq, int64_t n_bytes, uint8_t *packed)
{
    if (!cfg || n_bytes < 0 || (n_bytes > 0 && (!seq || !packed))) return fail(BDX_ERR_INVALID, "bad argument");
    if (!cfg->n_codes) return fail(BDX_ERR_INVALID, kNoPackedInput);
    bdx_pack4_bytes(cfg->code_of, seq, n_bytes, packed);
    return BDX_OK;
}

extern "C" int bdx_submit_packed4(bdx_stream *s, const uint8_t *packed, const int32_t *offsets, int32_t n, uint64_t tag)
{
    return submit_batch(s, {packed, offsets, nullptr, false, true, false}, n, tag);
}

extern "C" int bdx_submit_packed4_pinned(bdx_stream *s, const uint8_t *packed, const int32_t *offsets, int32_t n, uint64_t tag)
{
    return submit_batch(s, {packed, offsets, nullptr, false, true, true}, n, tag);
}

// ---- search-window input (windows.cu) ----
extern "C" int bdx_window_spans(const bdx_config *cfg, int32_t read_len, int32_t spans[4])
{
    if (!cfg || !spans || read_len < 0) return fail(BDX_ERR_INVALID, "bad argument");
    const DevParams P = host_params(*cfg, kSm100SmemOptin);
    int sp[4];
    const int len = read_windows(P, read_len, sp);
    for (int k = 0; k < 4; k++) spans[k] = sp[k];
    return len;
}

extern "C" int bdx_window_reads(const bdx_config *cfg, const uint8_t *seq, const int32_t *offsets, int32_t n,
                                uint8_t *win, int32_t *win_off)
{
    if (!cfg || n < 0 || (n > 0 && (!offsets || !win_off || (win && !seq)))) return fail(BDX_ERR_INVALID, "bad argument");
    if (n == 0) {
        if (win_off) win_off[0] = 0;
        return BDX_OK;
    }
    if (offsets[0] != 0) return fail(BDX_ERR_INVALID, "offsets[0] must be 0");
    for (int32_t i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i]) return fail(BDX_ERR_INVALID, "offsets must be non-decreasing");
    const DevParams P = host_params(*cfg, kSm100SmemOptin);
    int32_t w = 0, last_n = -1, len = 0;
    int sp[4] = {};
    win_off[0] = 0;
    for (int32_t i = 0; i < n; i++) {
        if (offsets[i + 1] - offsets[i] != last_n)       // the spans follow from the length: runs of equal lengths
            len = read_windows(P, last_n = offsets[i + 1] - offsets[i], sp);
        if (win) {
            for (int k = 0; k < 4; k += 2)               // column c of read i is seq[offsets[i] + c - 1]
                if (sp[k + 1] >= sp[k]) {
                    memcpy(win + w, seq + offsets[i] + sp[k] - 1, (size_t)(sp[k + 1] - sp[k] + 1));
                    w += sp[k + 1] - sp[k] + 1;
                }
        } else {
            w += len;
        }
        win_off[i + 1] = w;
    }
    return BDX_OK;
}

extern "C" int bdx_submit_windows(bdx_stream *s, const uint8_t *win, const int32_t *win_offsets, const int32_t *offsets,
                                  int32_t n_reads, int packed4, uint64_t tag)
{
    return submit_batch(s, {win, offsets, win_offsets, true, packed4 != 0, false}, n_reads, tag);
}

extern "C" int bdx_submit_windows_pinned(bdx_stream *s, const uint8_t *win, const int32_t *win_offsets,
                                         const int32_t *offsets, int32_t n_reads, int packed4, uint64_t tag)
{
    return submit_batch(s, {win, offsets, win_offsets, true, packed4 != 0, true}, n_reads, tag);
}

extern "C" int bdx_acquire(bdx_stream *s, uint8_t **seq, int32_t **offsets)
{
    if (!s || !seq || !offsets) return fail(BDX_ERR_INVALID, "null argument");
    int rc = check_stream(s, "already acquired");
    if (rc) return rc;
    CU(cudaSetDevice(s->device));
    if ((rc = ensure_input_buffers(s, false, false, true))) return rc;
    Slot &sl = s->slot[s->head];
    *seq = sl.h_seq;
    *offsets = sl.h_off;
    s->acquired = true;
    return BDX_OK;
}

extern "C" int bdx_commit(bdx_stream *s, int32_t n, uint64_t tag)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    if (!s->acquired) return fail(BDX_ERR_STATE, "bdx_commit without bdx_acquire");
    const Slot &sl = s->slot[s->head];
    return stage_batch(s, {sl.h_seq, sl.h_off, nullptr, false, false, true}, n, tag);
}

// Waits for the oldest batch in flight and takes it off the ring; its results stay in the slot's pinned staging
// until a later submit reuses the slot.
static int pop_oldest(bdx_stream *s, uint64_t *tag, int32_t *n_reads, Slot *&out)
{
    Slot &sl = s->slot[s->tail];
    CU(cudaEventSynchronize(sl.ev_done));
    if (tag) *tag = sl.tag;
    if (n_reads) *n_reads = sl.n;
    sl.busy = false;
    s->tail = (s->tail + 1) % BDX_MAX_IN_FLIGHT;
    s->in_flight--;
    out = &sl;
    return BDX_OK;
}

extern "C" int bdx_fetch(bdx_stream *s, uint64_t *tag, int32_t *n_reads, bdx_result *results,
                         bdx_pass_detail *details)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    if (s->in_flight == 0) return fail(BDX_ERR_STATE, "nothing in flight");
    if (details && !s->details) return fail(BDX_ERR_STATE, "details not enabled on this stream");
    Slot *sl = nullptr;
    if (int rc = pop_oldest(s, tag, n_reads, sl)) return rc;
    if (results && sl->n) memcpy(results, sl->h_res, (size_t)sl->n * sizeof(bdx_result));
    if (details && sl->n) memcpy(details, sl->h_det, (size_t)sl->n * 2 * sizeof(bdx_pass_detail));
    return BDX_OK;
}

// zero-copy retrieval: pointers into the pinned result staging of the oldest batch,
// valid until the next bdx_submit / bdx_commit that reuses the slot
extern "C" int bdx_fetch_view(bdx_stream *s, uint64_t *tag, int32_t *n_reads, const bdx_result **results,
                              const bdx_pass_detail **details)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    if (s->in_flight == 0) return fail(BDX_ERR_STATE, "nothing in flight");
    Slot *sl = nullptr;
    if (int rc = pop_oldest(s, tag, n_reads, sl)) return rc;
    if (results) *results = sl->h_res;
    if (details) *details = s->details ? sl->h_det : nullptr;
    return BDX_OK;
}

extern "C" int bdx_classify(bdx_stream *s, const uint8_t *seq, const int32_t *offsets, int32_t n,
                            bdx_result *results, bdx_pass_detail *details)
{
    if (s && s->in_flight) return fail(BDX_ERR_STATE, "batches in flight");
    int rc = bdx_submit(s, seq, offsets, n, 0);
    if (rc) return rc;
    return bdx_fetch(s, nullptr, nullptr, results, details);
}

extern "C" int bdx_classify_device(bdx_stream *s, const uint8_t *d_seq, const int32_t *d_off, int32_t n,
                                   bdx_result *d_res, bdx_pass_detail *d_det)
{
    if (!s || n < 0 || (n > 0 && (!d_seq || !d_off || !d_res))) return fail(BDX_ERR_INVALID, "bad argument");
    CU(cudaSetDevice(s->device));
    const int rc = bdx_stats_reserve_overflow(s, n, -1);      // read lengths are known on the device only
    if (rc) return rc;
    return bdx_enqueue_classify(s, d_seq, d_off, n, d_res, d_det);
}

extern "C" int bdx_stream_sync(bdx_stream *s)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->st_comp));
    return BDX_OK;
}

extern "C" int bdx_stream_profile(bdx_stream *s, int on)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    s->profile = on != 0;
    return BDX_OK;
}

extern "C" int bdx_stream_profile_read_stages(bdx_stream *s, double ms[BDX_PROFILE_STAGES], int32_t n_launches[BDX_PROFILE_STAGES])
{
    if (!s || !ms || !n_launches) return fail(BDX_ERR_INVALID, "null argument");
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->st_comp));
    for (int k = 0; k < BDX_PROFILE_STAGES; k++) {
        ms[k] = 0.0;
        n_launches[k] = 0;
    }
    for (auto &pr : s->prof_events) {
        float t = 0.f;
        CU(cudaEventElapsedTime(&t, pr.e0, pr.e1));
        ms[pr.kind] += t;
        n_launches[pr.kind]++;
        cudaEventDestroy(pr.e0);
        cudaEventDestroy(pr.e1);
    }
    s->prof_events.clear();
    return BDX_OK;
}

extern "C" int bdx_stream_profile_read(bdx_stream *s, double *filter_ms, int32_t *n_launches)
{
    if (!s || !filter_ms || !n_launches) return fail(BDX_ERR_INVALID, "null argument");
    double ms[BDX_PROFILE_STAGES];
    int32_t nl[BDX_PROFILE_STAGES];
    const int rc = bdx_stream_profile_read_stages(s, ms, nl);
    if (rc) return rc;
    *filter_ms = ms[kStFilter];
    *n_launches = nl[kStFilter];
    return BDX_OK;
}

// the 12 counters of bdx_stream::d_counters once the compute stream has drained; reset: zero them afterwards
static int read_counters(bdx_stream *s, unsigned long long (&h)[12], int reset)
{
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->st_comp));
    CU(cudaMemcpy(h, s->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
    if (reset) CU(cudaMemset(s->d_counters, 0, sizeof(h)));
    return BDX_OK;
}

extern "C" int bdx_stream_path_counters(bdx_stream *s, int64_t *prefilter_reads, int64_t *seed_reads,
                                        int64_t *automaton_reads, int reset)
{
    if (!s) return fail(BDX_ERR_INVALID, "null stream");
    unsigned long long h[12];
    if (int rc = read_counters(s, h, reset)) return rc;
    if (prefilter_reads) *prefilter_reads = (int64_t)h[0];
    if (seed_reads) *seed_reads = (int64_t)h[2];
    if (automaton_reads) *automaton_reads = (int64_t)h[1];
    return BDX_OK;
}

extern "C" int bdx_stream_work_counters(bdx_stream *s, int64_t out[12], int reset)
{
    if (!s || !out) return fail(BDX_ERR_INVALID, "null argument");
    unsigned long long h[12];
    if (int rc = read_counters(s, h, reset)) return rc;
    out[0] = (int64_t)h[0];
    out[1] = (int64_t)h[2];
    out[2] = (int64_t)h[1];
    out[3] = (int64_t)h[3];
    out[4] = (int64_t)h[4];
    for (int k = 5; k < 9; k++) out[k] = (int64_t)h[k];
    out[9] = out[10] = out[11] = 0;
    return BDX_OK;
}

extern "C" void *bdx_stream_cuda_stream(bdx_stream *s) { return s ? (void *)s->st_comp : nullptr; }
extern "C" int64_t bdx_stream_launch_count(const bdx_stream *s) { return s ? s->launches : 0; }

// ---------------------------------------------------------------------------
// device FASTQ block demultiplexer (demux.cu)
// ---------------------------------------------------------------------------
extern "C" int bdx_demux_block(bdx_stream *s, const uint8_t *fq1, int64_t len1, const uint8_t *fq2, int64_t len2,
                               int final_block, int mode, bdx_demux_out *out)
{
    if (!s || !out) return fail(BDX_ERR_INVALID, "null argument");
    if ((mode & 3) > BDX_DEMUX_BOTH || (mode & ~(3 | BDX_DEMUX_DEVICE_IO))) return fail(BDX_ERR_INVALID, "unknown demux mode");
    if (s->in_flight) return fail(BDX_ERR_STATE, "batches in flight");
    CU(cudaSetDevice(s->device));
    if (!s->demux && !(s->demux = demux_state_create())) return fail(BDX_ERR_NOMEM, "out of memory");
    std::string err;
    const int rc = demux_run(
        s->demux, s->tab->P, s->st_comp,
        [s](const uint8_t *d_seq, const int *d_off, int n, bdx_result *d_res) {
            const int rc2 = bdx_stats_reserve_overflow(s, n, -1);
            if (rc2) return rc2;
            return bdx_enqueue_classify(s, d_seq, d_off, n, d_res, nullptr);
        },
        fq1, len1, fq2, len2, final_block, mode, &s->launches, out, err);
    if (rc && !err.empty()) g_err = err;
    return rc;
}

extern "C" int bdx_demux_stage_ms(const bdx_stream *s, float ms[8])
{
    if (!s || !ms) return fail(BDX_ERR_INVALID, "null argument");
    if (!s->demux) return fail(BDX_ERR_STATE, "no bdx_demux_block call yet");
    memcpy(ms, demux_stage_ms(s->demux), 8 * sizeof(float));
    return BDX_OK;
}

// ---------------------------------------------------------------------------
// utilities
// ---------------------------------------------------------------------------
extern "C" int bdx_synth_reads_device(bdx_stream *s, const bdx_synth_spec *spec, int32_t n, uint8_t *d_seq,
                                      int32_t *d_off)
{
    if (!s || !spec || n < 0 || !d_seq || !d_off) return fail(BDX_ERR_INVALID, "bad argument");
    if (spec->read_len <= 0 || (int64_t)spec->read_len * n > 0x7FFFFFF0ll)
        return fail(BDX_ERR_TOO_LARGE, "n_reads * read_len must stay below 2^31");
    if (spec->start_lo < 1 || spec->start_hi < spec->start_lo || spec->end_hi < spec->end_lo)
        return fail(BDX_ERR_INVALID, "bad plant range");
    CU(cudaSetDevice(s->device));
    CU(launch_synth(s->tab->P, *spec, n, d_seq, d_off, s->st_comp));
    s->launches++;
    return BDX_OK;
}

extern "C" int bdx_int_alu_peak(int device, double *ops_per_second)
{
    if (!ops_per_second) return fail(BDX_ERR_INVALID, "null argument");
    cudaError_t e = run_int_alu_peak(device, ops_per_second);
    if (e != cudaSuccess) return cuda_fail(e, "int alu peak microbenchmark");
    return BDX_OK;
}

extern "C" void *bdx_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void bdx_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}
