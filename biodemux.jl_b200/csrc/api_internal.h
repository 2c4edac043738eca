// api_internal.h -- host-side state behind the C ABI (include/bdx.h), shared by the translation units that
// implement it: tables.cu (barcode tables), bdx_api.cu (configs, streams, batches), pool.cu (multi-GPU
// dispatcher), stats.cu (DemuxStats counters).  Not installed.
#pragma once

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "bdx_internal.h"
#include "demux.h"

using namespace bdx;

// ---- errors: every C-ABI call returns a bdx_status; the text goes to the calling thread's bdx_last_error() ----
int bdx_fail(int code, const std::string &msg);
int bdx_cuda_fail(cudaError_t e, const char *what);
std::string &bdx_error_text();
#define CU(call)                                                  \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return bdx_cuda_fail(e__, #call); \
    } while (0)

// ---- configuration ----
// The host vectors of one barcode set's tables (tables.cu), each uploaded per device into the DevSet pointer that
// get_tables (bdx_api.cu) pairs it with.  The set's scalars -- sizes, seed lengths, depths, which stages exist -- are
// kept only in its DevSet, bdx_config::base.set[s].  A level that is not built has empty vectors.
struct HostSet {
    int min_m = 0;                       // shortest barcode
    std::vector<uint8_t> bytes, class_of, bc_cls;
    std::vector<int> off, norm, filt_allowed, allowed0;
    std::vector<uint32_t> peq;
    std::vector<uint32_t> pf_bitmap, pf_keys, pf_vals;   // perfect-occurrence prefilter
    struct HostSeedLevel {
        std::vector<uint32_t> bstart, entries, ekeys, bitmap;
    };
    HostSeedLevel sd[2], sdd[2];         // k_seed levels (seed.cu), k_seed_deep tables (seed_deep.cu)
    struct HostSeedVar {
        std::vector<uint16_t> bstart;
        std::vector<uint32_t> entries;
        std::vector<uint8_t> kdepth;
    };
    HostSeedVar sv[2];                   // k_seed_var levels (seed_var.cu)
    std::vector<uint16_t> hp_bstart, hp_entries;   // k_hamming_scan (hamming.cu)
    std::vector<uint2> hp_bcw;
};

// ---- the kernel sequence of a pass (plan.cu) ----
enum { kStepHammingScan, kStepPrefilter, kStepSeed, kStepSeedVar, kStepSeedDeep, kStepFilter, kStepMarkPending,
       kStepLiteral };
enum { kWlNone, kWlWork, kWlWork2 };   // no worklist (every read of the batch), Scratch::worklist, Scratch::worklist2
// k_literal's reads: all of them over every barcode, those with candidates, Scratch::wl_win, ::wl_full, a worklist
enum { kLitAll, kLitCand, kLitWin, kLitFull, kLitRest };
// one launch: kernel (kStep*), k_seed / k_seed_var level, the worklists (kWl*) it takes its reads from and appends the
// reads it leaves open to, k_literal's reads (kLit*; kLitRest: those of worklist `in`), profiling stage (kSt*)
struct PlanStep {
    uint8_t kind, level, in, out, reads, stage;
};
struct PassPlan {
    bool clear_lit = false;   // zero the lengths of k_literal's two read lists before the first step
    int n = 0;
    PlanStep step[8];
};
// What runs for `pass` of a config, from its parameters alone: the table sizes in P already reflect the device's
// shared-memory limit (bdx_api.cu).  Made once per config and device; bdx_enqueue_classify walks it.
PassPlan plan_pass(const DevParams &P, int pass);
std::string plan_text(const PassPlan &plan);   // "k_prefilter,k_seed@1,...": the steps for bdx_config_describe

struct DeviceTables {
    DevParams P;
    PassPlan plan[2];
    std::vector<void *> allocs;
    int sm_count = 0;
};

struct bdx_config {
    uint32_t debug = 0;  // BDX_DEBUG_* (bdx_config_create_debug); 0 in production
    // 4-bit packed input (packed.cu): byte -> code over the barcode bytes of both sets, code -> representative byte
    int n_codes = 0;     // codes incl. 0; 0 = more than 15 distinct barcode bytes, packed input unavailable
    uint8_t code_of[256] = {};
    uint8_t rep_of[16] = {};
    DevParams base{};  // every scalar of the config and its sets; device pointers unset
    HostSet set[2];
    bdx_stats_layout lay{};
    std::mutex mu;
    std::map<int, DeviceTables *> per_device;
};

// Validates one barcode set and builds its tables (tables.cu): the scalars into D, the vectors into hs.
// debug: BDX_DEBUG_* switches.
int bdx_build_set(const bdx_params &p, const bdx_barcode_set &in, HostSet &hs, DevSet &D, uint32_t debug,
                  const char *name);
std::string bdx_describe_set(const HostSet &hs, const DevSet &D);   // tables.cu: text for bdx_config_describe

// ---- streams ----
struct Slot {
    uint8_t *h_seq = nullptr;
    int32_t *h_off = nullptr;
    bdx_result *h_res = nullptr;
    bdx_pass_detail *h_det = nullptr;
    uint8_t *d_packed = nullptr;  // 4-bit packed input of the batch (allocated on first packed submit)
    uint8_t *h_packed = nullptr;  // its pinned staging (bdx_submit_packed4 only)
    // search-window input (windows.cu), allocated on the first windowed submit: the window bytes (packed windows
    // use d_packed / h_packed, byte windows use h_seq as host staging) and the window stream's offsets
    uint8_t *d_win = nullptr;
    int32_t *d_win_off = nullptr;
    int32_t *h_win_off = nullptr;
    uint8_t *d_seq = nullptr;
    int32_t *d_off = nullptr;
    bdx_result *d_res = nullptr;
    bdx_pass_detail *d_det = nullptr;
    cudaEvent_t ev_h2d = nullptr, ev_kern = nullptr, ev_done = nullptr;
    int32_t n = 0;
    uint64_t tag = 0;
    bool busy = false;
    // the kernel sequence of a batch of graph_n reads on this slot's buffers, captured as a CUDA graph: small
    // batches (the reference's 4000-read chunks) are bound by launch gaps, not by the kernels
    cudaGraphExec_t graph = nullptr;
    int32_t graph_n = -1;         // batch size the graph was captured for
    bool graph_details = false;
    int graph_launches = 0;       // kernel launches it holds
    int uses = 0;                 // plain runs of this slot so far (the first warms the launch caches)
};

// stage of a profiled kernel launch (bdx_stream_profile_read_stages)
enum { kStPrefilter = 0, kStSeed = 1, kStSeedDeep = 2, kStFilter = 3, kStLiteral = 4, kStHamming = 5, kStFinalize = 6,
       kStOther = 7 };
struct ProfEvent {
    int kind;
    cudaEvent_t e0, e1;
};

struct bdx_stream {
    bdx_config *cfg = nullptr;
    DeviceTables *tab = nullptr;
    int device = 0;
    int32_t max_reads = 0;
    int64_t max_bytes = 0;
    bool details = false;
    cudaStream_t st_copy = nullptr, st_comp = nullptr, st_d2h = nullptr;
    Slot slot[BDX_MAX_IN_FLIGHT];
    bool host_staging = false;  // pinned h_seq / h_off are allocated on first use
    int head = 0;      // next slot to submit into
    int tail = 0;      // oldest in-flight slot
    int in_flight = 0;
    bool acquired = false;
    Scratch sc{};
    int64_t sc_cap = 0;
    unsigned long long *d_stats = nullptr;
    bdx_stats_overflow *d_ovf = nullptr;       // exact records of passes outside the pos / len histograms
    unsigned int *d_n_ovf = nullptr;           // [2] appended, lost
    int64_t ovf_cap = 0;                       // records d_ovf holds
    int64_t ovf_bound = 0;                     // most records the batches enqueued since the last drain can append
    std::vector<bdx_stats_overflow> h_ovf;     // records drained to the host so far
    unsigned long long *d_counters = nullptr;  // [0] reads resolved by the perfect-occurrence prefilter,
                                               // [1] reads that ran the bit-parallel automaton
    int64_t launches = 0;
    // optional per-kernel timing of the dominant (filter) kernel, for roofline reporting
    bool profile = false;
    bool graphs_ok = true;                     // cleared when a capture fails: plain launches from then on
    std::vector<ProfEvent> prof_events;
    DemuxState *demux = nullptr;               // device FASTQ block demultiplexer (demux.cu), created on first use
};

// DemuxStats overflow list (stats.cu): make room for a batch of n_reads reads whose longest read has max_len bases
// (-1 = unknown) BEFORE its kernels are enqueued -- drains the device list to the host and grows it as needed, so
// that no record is ever dropped -- and move the device list to the host.
int bdx_stats_reserve_overflow(bdx_stream *s, int64_t n_reads, int64_t max_len);
int bdx_stats_drain_overflow(bdx_stream *s);
// the slots' captured CUDA graphs hold device pointers: drop them when a buffer they use is re-allocated
void bdx_stream_drop_graphs(bdx_stream *s);

// Enqueue the classification kernels for n device-resident reads on the stream's compute CUDA stream (bdx_api.cu).
int bdx_enqueue_classify(bdx_stream *s, const uint8_t *d_seq, const int32_t *d_off, int32_t n, bdx_result *d_res,
                         bdx_pass_detail *d_det);
