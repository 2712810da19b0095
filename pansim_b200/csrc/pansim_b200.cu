// pansim_b200.cu -- context management and the C ABI of include/pansim_b200.h.
// All device work is in the kernels of *.cuh; this file owns memory, streams,
// launch configuration and error mapping. There is no CPU fallback.
#include "../../include/pansim_b200.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <limits>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "acc_step.cuh"
#include "comm.hpp"
#include "common.cuh"
#include "core_hr.cuh"
#include "core_mut.cuh"
#include "distance.cuh"
#include "diversity.cuh"
#include "gene_ld.cuh"
#include "genealogy.cuh"
#include "ld.cuh"
#include "nj.cuh"
#include "pack.cuh"
#include "pangenome.cuh"
#include "parsimony.cuh"
#include "replay.cuh"
#include "select.cuh"
#include "vcf.cuh"
#include "fasta.cuh"

using namespace pansim;

namespace {

std::string g_create_error;

struct HostPoissonTable {
    std::vector<uint32_t> thr;
    uint32_t size = 1, nsub = 0, kmax = 0;
    uint32_t *d_thr = nullptr;
    double mean_per_draw = 0.0;
};

// thresholds T[j] = round(CDF(j) * 2^32) of Poisson(mean / nsub), see common.cuh
void build_poisson_table(double mean, HostPoissonTable &t)
{
    t.thr.clear();
    if (!(mean > 0.0)) {
        t.nsub = 0; t.size = 1; t.kmax = 0; t.thr.assign(1, 0xFFFFFFFFu);
        return;
    }
    t.nsub = (uint32_t)std::ceil(mean / 64.0);
    if (t.nsub < 1) t.nsub = 1;
    const long double m = (long double)mean / (long double)t.nsub;
    t.mean_per_draw = (double)m;
    long double p = expl(-m), cdf = p;
    for (uint32_t j = 0; j < POISSON_TABLE_MAX - 1; j++) {
        const long double scaled = cdf * 4294967296.0L;
        if (scaled >= 4294967295.5L) { t.thr.push_back(0xFFFFFFFFu); break; }
        t.thr.push_back((uint32_t)llroundl(scaled));
        p *= m / (long double)(j + 1);
        cdf += p;
    }
    if (t.thr.back() != 0xFFFFFFFFu) t.thr.push_back(0xFFFFFFFFu);
    t.kmax = (uint32_t)t.thr.size() - 1;
    uint32_t size = 1;
    while (size < t.thr.size() + 1) size <<= 1;
    t.size = size;
    t.thr.resize(size, 0xFFFFFFFFu);
}

// core_mut.cuh image: [CM_GUIDE u16 guide entries][size thresholds]; entry = 2*k0 + many,
// many = the bin holds two or more thresholds (poisson_fast finishes with a scan)
std::vector<uint32_t> poisson_fast_image(const HostPoissonTable &t)
{
    std::vector<uint32_t> img(CM_GUIDE_WORDS + t.size, 0u);
    for (uint32_t b = 0; b < CM_GUIDE; b++) {
        const uint32_t lo = b << CM_GUIDE_SHIFT;
        const uint32_t hi = lo | ((1u << CM_GUIDE_SHIFT) - 1u);
        uint32_t k0 = 0, k1 = 0;
        while (k0 < t.kmax && t.thr[k0] <= lo) k0++;
        k1 = k0;
        while (k1 < t.kmax && t.thr[k1] <= hi) k1++;
        const uint32_t entry = 2u * k0 + (k1 > k0 + 1u ? 1u : 0u);
        img[b >> 1] |= entry << (16u * (b & 1u));
    }
    for (uint32_t j = 0; j < t.size; j++) img[CM_GUIDE_WORDS + j] = t.thr[j];
    return img;
}

struct EventPool {
    std::vector<cudaEvent_t> ev;
    size_t used = 0;
    cudaEvent_t get()
    {
        if (used == ev.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ev.push_back(e);
        }
        return ev[used++];
    }
    void reset() { used = 0; }
    void destroy()
    {
        for (auto e : ev) cudaEventDestroy(e);
        ev.clear();
        used = 0;
    }
};

enum TimeGroup { TG_SELECT = 0, TG_ACC, TG_CORE, TG_CORE_HR, TG_PAIR_CORE, TG_PAIR_ACC,
                 TG_D_INTER, TG_D_AVG, TG_D_SEL, TG_D_FLIP, TG_D_GAIN, TG_D_HGT, TG_COUNT };   // TG_D_*: PANSIM_FINE_TIMING=1 (debug)

}  // namespace

struct pansim_ctx {
    pansim_config cfg;
    std::string err;
    cudaStream_t stream = nullptr;        // accessory / selection chain, copies, distances
    cudaStream_t stream_core = nullptr;   // core step (runs concurrently with the chain above)
    cudaStream_t stream_aux = nullptr;    // fitness sum, concurrent with the intersection counts of the competition term
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_parents[3] = {nullptr, nullptr, nullptr};    // parents[i] written
    cudaEvent_t ev_core_done[3] = {nullptr, nullptr, nullptr};  // core step that read parents[i] finished
    bool core_done_valid[3] = {false, false, false};
    cudaEvent_t ev_core_last = nullptr;   // the most recently launched core step finished (independent of the parents rotation)
    bool core_unjoined = false;           // a core step is in flight on stream_core that `stream` has not been ordered after
    uint32_t *d_parents_buf[3] = {nullptr, nullptr, nullptr};
    uint32_t *h_parents = nullptr;        // pinned [N + 1]: parents + status word read back by pansim_sample_indices
    uint32_t *h_parents_up[3] = {nullptr, nullptr, nullptr};   // pinned staging of host-supplied parents (one per rotating buffer)
    cudaEvent_t ev_h2d[3] = {nullptr, nullptr, nullptr};        // the upload out of h_parents_up[i] has completed
    bool h2d_valid[3] = {false, false, false};
    double *h_avg = nullptr;              // pinned [N]: staging of avg_pairwise_dists in both directions
    int *h_err = nullptr;                 // pinned [2]: read-back of d_err
    int parents_idx = 0;
    int sm_count = 0;

    uint32_t N = 0, G = 0;
    uint64_t L = 0, site_begin = 0, site_end = 0, Ll = 0;
    uint32_t n_regions = 0, region0 = 0;
    uint64_t core_stride = 0;
    uint32_t acc_stride_words = 0, acc_words = 0;

    uint8_t *core[2] = {nullptr, nullptr};
    // recombination (core_hr.cuh): per-item slots filled by the collect step, drained by the apply step
    uint16_t *d_hr_slots = nullptr, *d_hr_counts = nullptr;
    uint32_t hr_slot_cap = 0;
    unsigned long long *d_hr_ovf = nullptr;
    uint32_t *d_hr_ovf_count = nullptr;  // two counters, used alternately
    uint32_t hr_ovf_cap = 0;
    int hr_parity = 0;
    // deferred recombination (core_mut.cuh): the current core buffer holds the pre-recombination rows of
    // generation hr_pending_gen; the next core step applies the events while it gathers, a reader of the
    // state materialises them first (core_materialize)
    bool hr_pending = false;
    uint32_t hr_pending_gen = 0;
    bool hr_defer = true;                // PANSIM_HR_DEFER=0: recombination as two launches right after every core step
    size_t hr_smem = 0;
    uint32_t *acc[2] = {nullptr, nullptr};
    int core_cur = 0, acc_cur = 0;
    bool has_core = false, has_acc = false;

    uint32_t *d_parents = nullptr;
    double *d_lw = nullptr, *d_logfit = nullptr, *d_avgdist = nullptr;
    uint32_t *d_lethal = nullptr;         // bit g: ln(1 + s_g) = -inf (s_g = -1)
    // PANSIM_FITNESS_MODE: 1 = two warps per row (28 us, but ~500 CTAs resident beside the core kernel),
    // 2 = one lane per row (30 us, 8 CTAs), 0 = by entry point: two warps per row where the host waits on
    // the chain, one lane per row in the device-resident batch (the core kernel keeps its SM slots:
    // 154 against 175-189 us per generation at cfg2). All three give the same bits.
    int fitness_mode = 0;
    int32_t *d_num_genes = nullptr;
    int32_t *d_inter_diag = nullptr;      // gene counts as the diagonal of the intersection matrix (select.cuh K2a)
    bool fitness_join_pending = false;    // a fitness kernel is running on stream_aux that `stream` has not been ordered after
    double *d_tmp_a = nullptr, *d_tmp_b = nullptr, *d_weights = nullptr, *d_cum = nullptr;
    int *d_err = nullptr;                // [0] upload / selection errors, [1] recombination list overflow
    uint32_t *d_inter = nullptr;
    double *d_rowInvK = nullptr;
    uint32_t *d_gain_thr = nullptr;      // scratch (gene counts)
    uint32_t *d_gain_planes = nullptr;   // [gene words][32] bit-planes of the HGT gain thresholds
    bool avgdist_valid = false;
    bool fitness_valid = false;   // d_logfit / d_num_genes match the current accessory state
    bool neutral = true;          // every selection coefficient is 0 (ln(1 + s_j) = +0.0 for all genes)
    bool umma_bits_ready = false;     // the intersection kernel's dynamic shared-memory limit is raised
    double *d_rcp = nullptr;          // RN(1 / b), b = 0 .. G + core_genes; only when G + core_genes <= AVG_RCP_MAX
    bool fitness_blocked = false; // large shapes: blocked (fixed-association) fitness sum instead of the sequential chain

    HostPoissonTable tab_mut, tab_hr;    // per 256-site block (SNPs), per 8192-site region (HR)
    uint32_t hr_k0 = 0;                  // 32-threshold window of tab_hr that is tried first (core_mut.cuh)
    uint8_t *d_core_img = nullptr;       // constant image of the core kernel (core_mut.cuh)
    uint32_t flip_thr[2] = {0, 0};
    double flip_p[2] = {0, 0};
    double hgt_scale[2] = {0, 0};
    double p_mut_site = 0, p_hr_site = 0;

    // pair plan (row-stationary groups), cached while the pair list is unchanged
    std::vector<uint32_t> plan_r1, plan_r2;
    PairGroup *d_groups = nullptr;
    uint32_t *d_partner = nullptr, *d_orig = nullptr;
    size_t plan_groups = 0, plan_cap_groups = 0, plan_cap_pairs = 0;
    TileBatch *d_batches = nullptr;
    uint16_t *d_tile_slots = nullptr;
    uint32_t *d_tile_orig = nullptr;
    size_t plan_batches = 0, plan_cap_batches = 0, plan_cap_tile_pairs = 0;
    // plane form of the core rows for the distance kernels (distance.cuh), made by a pre-pass when the
    // state has changed since the last one; TMA descriptor of it for the tile kernel
    uint8_t *d_planes = nullptr;
    uint64_t core_version = 1, planes_version = 0;     // bumped whenever the current core buffer changes
    CUtensorMap planes_tmap;
    bool planes_tmap_ok = false;
    uint32_t *d_work_counter = nullptr;
    bool use_tiles2 = true;              // PANSIM_TILES2=0: row-stationary groups only
    // pair buffers
    uint32_t *d_r1 = nullptr, *d_r2 = nullptr, *d_cd = nullptr, *d_in = nullptr, *d_un = nullptr;
    size_t pair_cap = 0;
    bool pairs_on_device = false;        // d_r1 / d_r2 hold plan_r1 / plan_r2
    uint32_t *d_cnt2[3] = {nullptr, nullptr, nullptr};   // second set of count vectors (per-generation statistics batch)
    size_t cnt2_cap = 0;
    double *d_stats = nullptr, *h_stats = nullptr;       // per-generation statistics (4 doubles each), device / pinned
    size_t stats_cap = 0;
    // the stream the distance pass runs on: c->stream, except inside the --print_dist batch where the pass of
    // generation g runs on stream_pairs beside the selection chain and the core step of generation g+1
    cudaStream_t ps = nullptr, stream_pairs = nullptr;
    cudaEvent_t ev_acc_done = nullptr, ev_mat = nullptr;
    bool ev_pairs_valid[2] = {false, false};
    cudaStream_t stream_stats2[2] = {nullptr, nullptr};   // statistics kernels of consecutive generations run side by side
    cudaEvent_t ev_pairs[2] = {nullptr, nullptr}, ev_stats[2] = {nullptr, nullptr};
    bool ev_stats_valid[2] = {false, false};
    // diversity reductions (diversity.cuh): packed copy of the clonal row pansim_set_initial started from (the
    // ancestral allele of every site, for the SFS), per-call / per-generation results and the SFS bins
    uint32_t *d_anc = nullptr;
    bool has_anc = false;
    unsigned long long *d_div = nullptr, *h_div = nullptr;   // [n][4]: segregating, multiallelic, pair_diff_sum, -
    size_t div_cap = 0;
    unsigned long long *d_sfs = nullptr, *h_sfs = nullptr;   // [N + 1]

    // column shards of one alignment: NCCL communicator over the shards (comm.hpp). With a communicator the
    // pair-count entry points return whole-alignment core counts (summed over the shards on the device).
    ncclComm_t comm = nullptr;
    int comm_size = 1, comm_rank = 0;
    bool comm_owned = false;             // created by pansim_comm_init_rank (a pansim_group owns its communicators itself)

    // replay staging
    void *d_replay = nullptr;
    size_t replay_cap = 0;
    unsigned long long *d_hkeys = nullptr;
    uint32_t *d_hvals = nullptr;
    size_t hash_cap = 0;

    // text export (CSV, VCF): two device + two pinned host chunks (double buffering), completion events
    char *d_txt[2] = {nullptr, nullptr}, *h_txt[2] = {nullptr, nullptr};
    cudaEvent_t ev_txt[2] = {nullptr, nullptr};
    size_t txt_cap = 0;
    // VCF export (vcf.cuh): per-site allele counts (shared with the FASTA export), line descriptors and offsets,
    // scan blocks, chunk bounds
    uint4 *d_vcf_counts = nullptr;
    uint8_t *d_vcf_desc = nullptr;
    unsigned long long *d_vcf_off = nullptr, *d_vcf_block = nullptr, *d_vcf_bounds = nullptr;
    uint32_t *d_vcf_nchunks = nullptr;
    // FASTA export (fasta.cuh), SNP mode: polymorphic sites per scan block (+ total), constant-site letters, the
    // column list; pinned read-back of the column count and the constant-site letters
    unsigned long long *d_fa_block = nullptr, *d_fa_const = nullptr, *h_fa = nullptr;
    uint32_t *d_fa_cols = nullptr;
    // core LD (ld.cuh): allele counts, used-site ranks, the compacted used sites (position, derived count, 1 / (a (n - a)))
    // and their site-major derived bit rows. `ld` holds the context's own used sites followed by the halo copied from
    // the next shard; `ld_halo` is the halo this context makes of its first sites when it is the next of another one.
    struct LdBuf {
        uint4 *counts = nullptr;
        unsigned long long *block = nullptr;
        uint32_t *rank = nullptr, *pos = nullptr, *a = nullptr, *x = nullptr;
        double *inv = nullptr;
        size_t site_cap = 0, used_cap = 0, x_cap = 0;
    } ld, ld_halo;
    unsigned long long *d_ld_tiles = nullptr, *d_ld_bins = nullptr;   // tile-pair offsets [I tiles + 1], bins [n][4]
    size_t ld_tiles_cap = 0, ld_bins_cap = 0;
    unsigned long long *h_ld = nullptr, *h_ld_bins = nullptr;         // pinned: own / halo used sites, tile pairs; bins
    size_t h_ld_bins_cap = 0;
    cudaEvent_t ev_ld = nullptr;                                       // the halo of this context is ready
    // accessory-gene LD (gene_ld.cuh): presence counts and ranks of the G genes, the compacted used genes (presence
    // count, group, 1 / (a (n - a))), their gene-major presence bit rows, and the outputs (class totals, histogram,
    // used genes of group 1), mirrored in pinned host memory
    struct GeneLdBuf {
        uint32_t *counts = nullptr, *rank = nullptr, *a = nullptr, *grp = nullptr, *x = nullptr;
        double *inv = nullptr;
        unsigned long long *block = nullptr, *out = nullptr, *h_out = nullptr;
        size_t x_cap = 0, out_cap = 0;
    } gl;
    // pangenome accumulation (pangenome.cuh): the orders, the per-step deltas (also the swap indices of an order draw
    // that does not fit in shared memory), the chunk summaries and the four curves, sized for perm_cap orders; the
    // gene frequency spectrum
    struct GeneAccBuf {
        uint32_t *orders = nullptr, *delta = nullptr, *summary = nullptr, *curves = nullptr;
        size_t perm_cap = 0, summary_cap = 0;
        unsigned long long *spectrum = nullptr;
        int walk_slots = 0;          // resident walk CTAs of the device (per SM x SMs), queried on first use
        int order_smem_max = 0;      // shared memory a CTA can opt in to (the order draw's limit), queried on first use
    } ga;
    // clonal genealogy (genealogy.cuh): a ring of the last gen_cap parent vectors, each copied on stream_gen behind
    // ev_parents[i]; next_parents_buffer waits on ev_gen_done[i] before buffer i is rewritten. The trace and the
    // TMRCA walk run on stream_gen too, so they follow every copy enqueued before them.
    cudaStream_t stream_gen = nullptr;
    cudaEvent_t ev_gen_done[3] = {nullptr, nullptr, nullptr};
    bool gen_done_valid[3] = {false, false, false};
    uint32_t *d_gen_ring = nullptr;      // [gen_cap][N]
    uint32_t *d_gen_scratch = nullptr;   // trace scratch and node table, gen_scratch_words(N) words
    uint32_t gen_cap = 0;                // 0: recording off
    uint64_t gen_total = 0;              // vectors appended since the last reset
    uint64_t gen_epoch = 1, gen_traced = 0;   // bumped by every append and reset / the record the node table is of
    uint32_t gen_nodes = 0, gen_lineages = 0;
    uint32_t *d_gen_pairs = nullptr;     // TMRCA: r1, r2, result
    size_t gen_pair_cap = 0;
    // staging for upload/download
    uint8_t *d_stage = nullptr;
    size_t stage_cap = 0;

    // event dump
    bool dump_enabled = false;
    uint32_t dump_cap = 0;
    uint32_t *d_dump_counters = nullptr;
    uint32_t *d_mut_row = nullptr, *d_mut_site = nullptr, *d_mut_seq = nullptr;
    uint8_t *d_mut_allele = nullptr;
    uint32_t *d_hr_rec = nullptr, *d_hr_locus = nullptr, *d_hr_donor = nullptr, *d_hr_seq = nullptr;
    uint8_t *d_hr_value = nullptr;
    uint32_t *d_dump_flip = nullptr, *d_dump_gain = nullptr;

    // timing
    bool timing_enabled = true;
    int use_pdl = 1;                     // PANSIM_PDL: 0 = never, 1 = host-driven entry points only (default), 2 = always
    // Dependents that wait inside an SM slot take that slot from the core kernel: worth it when the host
    // waits on the chain every generation (step_with_parents / sample_indices / average_distance), not in
    // the device-resident batch of run_generations, which is bound by the core kernel (measured: -21 us of
    // chain per generation either way, +3 % core kernel time in the batch).
    bool pdl_now = false;
    bool fine_timing = false;            // PANSIM_FINE_TIMING=1: per-kernel spans of the selection chain, printed by pansim_get_timing
    EventPool pool;
    struct Span { cudaEvent_t a, b; int group; };
    std::vector<Span> spans;
    cudaEvent_t t_begin = nullptr, t_end = nullptr;
    uint32_t launches = 0;

    // CUDA graphs of the selection chain (competition, fitness, parent draw, accessory step) of ONE generation
    // for the device-resident batches: six phases (three parents buffers x two accessory buffers), one
    // executable graph each. The core kernel stays an ordinary launch on its own low-priority stream.
    bool use_graph = true;               // PANSIM_GRAPH=0: every kernel of the chain is launched on its own
    bool graph_spans = true;             // PANSIM_GRAPH_SPANS=0: no event-record nodes (kernel-group timing) inside the graphs
    bool chain_graph_now = false;        // set by the batch entry points
    bool capturing = false;
    const uint32_t *gen_dev_now = nullptr;   // while capturing: kernels take the generation as args.gen + *gen_dev
    uint32_t *d_gen_base = nullptr;
    uint32_t gen_base_host = 0xFFFFFFFFu;    // value d_gen_base will hold when the work enqueued so far has run
    struct GraphKey { int parents_idx, acc_cur, fitness_mode; bool competition, timing, neutral, fitness_valid, fitness_blocked; };
    struct GraphEntry {
        GraphKey key{};
        cudaGraphExec_t exec = nullptr;
        EventPool pool;                  // events referenced by the graph's record nodes (never recycled)
        std::vector<Span> spans;
        uint32_t kernels = 0;            // kernel launches captured
        uint32_t used = 0;               // launches in the current timed call (scales the spans in pansim_get_timing)
        int acc_cur_after = 0;           // host-side state the captured calls leave behind
        bool fitness_valid_after = false;
    };
    std::vector<GraphEntry *> graphs;
    GraphEntry *cap = nullptr;           // entry being captured

    uint32_t core_grid = 0, core_items_per_warp = 1;
    uint32_t core_items_batch = 0;        // items per warp in the device-resident batch (0 = same as core_items_per_warp)
    size_t core_smem = 0;
    int core_occupancy = 0;
};

namespace {

#define FAIL(ctx, code, ...)                                 \
    do {                                                     \
        char _b[512];                                        \
        snprintf(_b, sizeof _b, __VA_ARGS__);                \
        (ctx)->err = _b;                                     \
        return (code);                                       \
    } while (0)

#define CU(ctx, call)                                                                            \
    do {                                                                                         \
        cudaError_t _e = (call);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            FAIL(ctx, PANSIM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e),   \
                 __FILE__, __LINE__);                                                            \
    } while (0)

#define LAUNCH_CHECK(ctx)                                                                        \
    do {                                                                                         \
        (ctx)->launches++;                                                                       \
        cudaError_t _e = cudaGetLastError();                                                     \
        if (_e != cudaSuccess)                                                                   \
            FAIL(ctx, PANSIM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), \
                 __FILE__, __LINE__);                                                            \
    } while (0)

inline uint32_t div_up64(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

struct ScopedSpan {
    pansim_ctx *c;
    int group;
    cudaStream_t st;
    cudaEvent_t a = nullptr;
    bool on = false;
    ScopedSpan(pansim_ctx *ctx, int g, cudaStream_t stream = nullptr) : c(ctx), group(g), st(stream ? stream : ctx->stream)
    {
        on = c->timing_enabled && !(c->capturing && !c->graph_spans);
        if (on) {
            if (c->capturing) {         // an event-record NODE of the graph: it holds the time of the last replay
                a = c->cap->pool.get();
                cudaEventRecordWithFlags(a, st, cudaEventRecordExternal);
            } else {
                a = c->pool.get();
                cudaEventRecord(a, st);
            }
        }
    }
    ~ScopedSpan()
    {
        if (on) {
            if (c->capturing) {
                cudaEvent_t b = c->cap->pool.get();
                cudaEventRecordWithFlags(b, st, cudaEventRecordExternal);
                c->cap->spans.push_back({a, b, group});
            } else {
                cudaEvent_t b = c->pool.get();
                cudaEventRecord(b, st);
                c->spans.push_back({a, b, group});
            }
        }
    }
};

// Launch `kernel` as a programmatic dependent of the kernel enqueued just before it on `st`
// (common.cuh: pdl_wait / pdl_launch_dependents). With c->use_pdl off it is an ordinary launch.
template <typename... KArgs, typename... Args>
void launch_dependent(pansim_ctx *c, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = (c->use_pdl == 2 || (c->use_pdl == 1 && c->pdl_now)) ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, args...);
}

// debug-only sub-span (PANSIM_FINE_TIMING=1)
struct FineSpan {
    pansim_ctx *c; int group; cudaEvent_t a = nullptr;
    FineSpan(pansim_ctx *ctx, int g) : c(ctx), group(g)
    {
        if (c->fine_timing && c->timing_enabled) { a = c->pool.get(); cudaEventRecord(a, c->stream); }
    }
    ~FineSpan()
    {
        if (a) { cudaEvent_t b = c->pool.get(); cudaEventRecord(b, c->stream); c->spans.push_back({a, b, group}); }
    }
};

void timing_begin(pansim_ctx *c)
{
    c->launches = 0;
    c->spans.clear();
    c->pool.reset();
    for (auto *e : c->graphs) e->used = 0;
    if (c->timing_enabled) {
        c->t_begin = c->pool.get();
        cudaEventRecord(c->t_begin, c->stream);
    }
}

void timing_end(pansim_ctx *c)
{
    if (c->timing_enabled) {
        c->t_end = c->pool.get();
        cudaEventRecord(c->t_end, c->stream);
    }
}

int ensure_stage(pansim_ctx *c, size_t bytes)
{
    if (bytes <= c->stage_cap) return 0;
    if (c->d_stage) cudaFree(c->d_stage);
    c->d_stage = nullptr;
    c->stage_cap = 0;
    CU(c, cudaMalloc(&c->d_stage, bytes));
    c->stage_cap = bytes;
    return 0;
}

// d_err[0]: input / selection errors (meaning given by the caller). d_err[1]: the recombination
// overflow list (sized 12 sigma above its mean) was full, i.e. events were dropped. Both are read
// back together wherever a call synchronises anyway.
int flags_enqueue_readback(pansim_ctx *c)
{
    CU(c, cudaMemcpyAsync(c->h_err, c->d_err, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

// after the stream has been synchronised behind flags_enqueue_readback
int flags_inspect(pansim_ctx *c, int code, const char *what)
{
    const int f0 = c->h_err[0], f1 = c->h_err[1];
    if (f0 || f1) cudaMemsetAsync(c->d_err, 0, 2 * sizeof(int), c->stream);
    if (f1) FAIL(c, PANSIM_ERR_STATE, "recombination overflow list full: events were dropped in an earlier generation");
    if (f0) FAIL(c, code, "%s", what);
    return 0;
}

int check_hr_flag(pansim_ctx *c)
{
    if (!c->d_hr_slots) return 0;
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    const int f1 = c->h_err[1];
    if (f1) {
        cudaMemsetAsync(c->d_err + 1, 0, sizeof(int), c->stream);
        FAIL(c, PANSIM_ERR_STATE, "recombination overflow list full: events were dropped in an earlier generation");
    }
    return 0;
}

int check_device_flag(pansim_ctx *c, int code, const char *what)
{
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return flags_inspect(c, code, what);
}

#define NCK(ctx, call)                                                                            \
    do {                                                                                          \
        ncclResult_t _r = (call);                                                                 \
        if (_r != ncclSuccess)                                                                    \
            FAIL(ctx, PANSIM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, nccl_api().GetErrorString(_r), __FILE__, __LINE__); \
    } while (0)

// sum of the per-pair partial core counts over the column shards, in place, on c->stream (C2 of SURVEY.md 2)
int comm_allreduce_counts(pansim_ctx *c, uint32_t *d_counts, size_t n)
{
    if (!c->comm || c->comm_size < 2 || !d_counts || !n) return 0;
    NCK(c, nccl_api().AllReduce(d_counts, d_counts, n, ncclUint32, ncclSum, c->comm, c->ps));
    c->launches++;
    timing_end(c);          // the collective belongs to the pass it completes (total_ms of pansim_get_timing)
    return 0;
}

// ---- kernel group launchers (asynchronous on ctx->stream) -----------------

// order `stream` after the fitness kernel that launch_competition started on the aux stream
int join_fitness(pansim_ctx *c)
{
    if (!c->fitness_join_pending) return 0;
    CU(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    c->fitness_join_pending = false;
    return 0;
}

int launch_fitness(pansim_ctx *c, cudaStream_t st = nullptr)
{
    if (c->fitness_valid) return 0;
    if (int rc = join_fitness(c)) return rc;        // an earlier one still writes the same outputs
    if (!st) st = c->stream;
    const uint32_t *acc = c->acc[c->acc_cur];
    if (c->neutral)          // every ln(1 + s_j) is +0.0: the sum is +0.0, only the row popcounts are needed
        fitness_count_kernel<<<div_up64(c->N, FIT_WARPS), FIT_WARPS * 32, 0, st>>>(acc, c->N, c->G, c->acc_stride_words,
                                                                              c->d_logfit, c->d_num_genes);
    else if (c->fitness_blocked)
        fitness_blocked_kernel<<<div_up64(c->N, FIT_WARPS), FIT_WARPS * 32, 0, st>>>(acc, c->N, c->G, c->acc_stride_words,
                                                                                c->d_lw, c->d_logfit, c->d_num_genes);
    else if (c->fitness_mode == 1 || (c->fitness_mode == 0 && c->pdl_now))
        fitness_kernel<<<div_up64(c->N, FIT_ROWS), FIT_ROWS * 64, 0, st>>>(acc, c->N, c->G, c->acc_stride_words,
                                                                      c->d_lw, c->d_logfit, c->d_num_genes);
    else
        fitness_lane_kernel<<<div_up64(c->N, FITL_THREADS), FITL_THREADS, 0, st>>>(acc, c->N, c->G, c->acc_stride_words,
                                                                              c->d_lw, c->d_lethal, c->d_logfit, c->d_num_genes);
    LAUNCH_CHECK(c);
    c->fitness_valid = true;
    return 0;
}

// the intersection matrix, the intersection kernel's shared-memory limit, and the reciprocal table of the mean-distance
// kernel when the shape allows it
int ensure_competition_buffers(pansim_ctx *c)
{
    if (!c->d_inter) CU(c, cudaMalloc(&c->d_inter, (size_t)c->N * c->N * sizeof(uint32_t)));
    if (!c->umma_bits_ready) {
        CU(c, cudaFuncSetAttribute(acc_inter_umma_bits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UbCfg<128>::smem_bytes()));
        c->umma_bits_ready = true;
    }
    if (!c->d_rcp && (uint64_t)c->G + c->cfg.core_genes <= AVG_RCP_MAX) {
        const size_t n = (size_t)c->G + c->cfg.core_genes + 1;
        std::vector<double> h(n);
        for (size_t b = 0; b < n; b++) h[b] = 1.0 / (double)b;            // IEEE division: correctly rounded; b = 0 -> inf
        CU(c, cudaMalloc(&c->d_rcp, n * sizeof(double)));
        CU(c, cudaMemcpy(c->d_rcp, h.data(), n * sizeof(double), cudaMemcpyHostToDevice));
    }
    return 0;
}

int launch_competition(pansim_ctx *c)
{
    if (c->N < 2) FAIL(c, PANSIM_ERR_INVALID, "average_distance needs pop_size >= 2");
    if (!c->capturing)
        if (int rc = ensure_competition_buffers(c)) return rc;
    // the fitness sum runs on the aux stream beside the intersection counts AND the distance kernel (which
    // takes the gene counts from the diagonal of the intersection matrix); whoever needs log-fitness or
    // d_num_genes joins it (join_fitness)
    std::unique_ptr<FineSpan> fs(new FineSpan(c, TG_D_INTER));
    if (!c->fitness_valid) {
        CU(c, cudaEventRecord(c->ev_fork, c->stream));
        CU(c, cudaStreamWaitEvent(c->stream_aux, c->ev_fork, 0));
        if (launch_fitness(c, c->stream_aux)) return PANSIM_ERR_CUDA;
        CU(c, cudaEventRecord(c->ev_join, c->stream_aux));
        c->fitness_join_pending = true;
    }
    const uint32_t nb = div_up64(c->N, UM_TILE);
    acc_inter_umma_bits_kernel<<<nb * (nb + 1) / 2, UB_THREADS, UbCfg<128>::smem_bytes(), c->stream>>>(
        c->acc[c->acc_cur], c->N, c->acc_stride_words, (uint32_t)div_up64(std::max<uint64_t>(c->G, 1), 128), c->d_inter, c->d_inter_diag);
    LAUNCH_CHECK(c);
    fs.reset();
    FineSpan fs2(c, TG_D_AVG);
    if (c->d_rcp)          // the reciprocal table exists iff G + core_genes <= AVG_RCP_MAX
        avg_distance_pipe_kernel<<<div_up64(c->N, AVG_WARPS), AVG_WARPS * 32, 0, c->stream>>>(c->d_inter, c->d_inter_diag, c->N,
                                                                             c->cfg.core_genes, c->d_rcp, c->d_avgdist);
    else
        avg_distance_kernel<<<div_up64(c->N, AVG_WARPS), AVG_WARPS * 32, 0, c->stream>>>(c->d_inter, c->d_inter_diag, c->N,
                                                                        c->cfg.core_genes, c->d_avgdist);
    LAUNCH_CHECK(c);
    c->avgdist_valid = true;
    return 0;
}

int launch_select(pansim_ctx *c, uint32_t gen, bool use_avgdist)
{
    if (launch_fitness(c)) return PANSIM_ERR_CUDA;
    if (int rc = join_fitness(c)) return rc;
    SelectArgs a;
    a.logfit = c->d_logfit;
    a.num_genes = c->d_num_genes;
    a.avgdist = use_avgdist ? c->d_avgdist : nullptr;
    a.n_rows = c->N;
    a.n_genes = c->G;
    a.avg_gene_num = c->cfg.avg_gene_num;
    a.no_control_genome_size = c->cfg.no_control_genome_size;
    a.log_penalty = std::log(c->cfg.genome_size_penalty);
    a.competition_strength = c->cfg.competition_strength;
    a.key = make_uint2((uint32_t)c->cfg.seed, (uint32_t)(c->cfg.seed >> 32));
    a.gen = gen;
    a.gen_dev = c->gen_dev_now;
    a.tmp_a = c->d_tmp_a;
    a.tmp_b = c->d_tmp_b;
    a.weights = c->d_weights;
    a.cumulative = c->d_cum;
    a.parents = c->d_parents;
    a.err_flag = c->d_err;
    {
        FineSpan fs(c, TG_D_SEL);
        if (c->N <= SEL_SMALL_MAX)
            launch_dependent(c, select_parents_small_kernel, dim3(1), dim3(SEL_THREADS), 0, c->stream, a);
        else if (c->N <= 4096)
            launch_dependent(c, select_parents_kernel<SEL_THREADS>, dim3(1), dim3(SEL_THREADS), 0, c->stream, a);
        else
            launch_dependent(c, select_parents_kernel<1024>, dim3(1), dim3(1024), 0, c->stream, a);
    }
    LAUNCH_CHECK(c);
    return 0;
}

void fill_acc_args(pansim_ctx *c, AccArgs &a, uint32_t gen)
{
    memset(&a, 0, sizeof a);
    a.old_state = c->acc[c->acc_cur];
    a.new_state = c->acc[c->acc_cur ^ 1];
    a.parents = c->d_parents;
    a.n_rows = c->N;
    a.n_genes = c->G;
    a.stride_words = c->acc_stride_words;
    a.key = make_uint2((uint32_t)c->cfg.seed, (uint32_t)(c->cfg.seed >> 32));
    a.rk = philox_key_schedule(a.key);
    a.gen = gen;
    a.gen_dev = c->gen_dev_now;
    if (c->cfg.n_compartments > 0) { a.lo0 = c->cfg.comp_lo[0]; a.hi0 = c->cfg.comp_hi[0]; }
    if (c->cfg.n_compartments > 1) { a.lo1 = c->cfg.comp_lo[1]; a.hi1 = c->cfg.comp_hi[1]; }
    a.flip_thr0 = c->flip_thr[0]; a.flip_thr1 = c->flip_thr[1];
    a.hgt_scale0 = c->hgt_scale[0]; a.hgt_scale1 = c->hgt_scale[1];
    a.rowInvK = c->d_rowInvK;
    a.gain_planes = c->d_gain_planes;
    a.dump_flip = c->d_dump_flip;
    a.dump_gain = c->d_dump_gain;
}

int launch_acc_step(pansim_ctx *c, uint32_t gen)
{
    if (c->G == 0) return 0;
    if (int rc = join_fitness(c)) return rc;        // it reads the accessory buffers this step recycles
    AccArgs a;
    fill_acc_args(c, a, gen);
    const uint32_t rows_per_cta = 8;
    {
        FineSpan fs(c, TG_D_FLIP);
        if (c->dump_enabled)
            acc_gather_flip_kernel<true><<<div_up64(c->N, rows_per_cta), 256, 0, c->stream>>>(a);
        else
            acc_gather_flip_kernel<false><<<div_up64(c->N, rows_per_cta), 256, 0, c->stream>>>(a);
    }
    LAUNCH_CHECK(c);
    const bool hgt = (a.hgt_scale0 > 0.0 || a.hgt_scale1 > 0.0);
    if (hgt) {
        {
            FineSpan fs(c, TG_D_GAIN);
            launch_dependent(c, acc_gain_threshold_kernel, dim3(c->acc_words), dim3(GAIN_WARPS * 32), 0, c->stream, a);
        }
        LAUNCH_CHECK(c);
        const uint64_t total = (uint64_t)c->N * c->acc_stride_words;
        {
            FineSpan fs(c, TG_D_HGT);
            if (c->dump_enabled)
                launch_dependent(c, acc_hgt_apply_kernel<true>, dim3(div_up64(total, 256)), dim3(256), 0, c->stream, a);
            else
                launch_dependent(c, acc_hgt_apply_kernel<false>, dim3(div_up64(total, 256)), dim3(256), 0, c->stream, a);
        }
        LAUNCH_CHECK(c);
    } else if (c->dump_enabled) {
        CU(c, cudaMemsetAsync(c->d_dump_gain, 0, (size_t)c->N * c->acc_stride_words * 4, c->stream));
    }
    c->acc_cur ^= 1;
    c->fitness_valid = false;
    return 0;
}

void fill_core_args(pansim_ctx *c, CoreMutArgs &a, uint32_t gen)
{
    memset(&a, 0, sizeof a);
    a.old_state = c->core[c->core_cur];
    a.new_state = c->core[c->core_cur ^ 1];
    a.parents = c->d_parents;
    a.n_rows = c->N;
    a.n_regions = c->n_regions;
    a.row_stride = c->core_stride;
    a.region0 = c->region0;
    a.items_per_warp = (!c->pdl_now && c->core_items_batch) ? c->core_items_batch : c->core_items_per_warp;
    a.site_limit = c->site_end;
    a.last_greg = (uint32_t)((c->site_end - 1) / REGION_SITES);
    a.lim_last = (uint32_t)(c->site_end - (uint64_t)a.last_greg * REGION_SITES);
    a.key = make_uint2((uint32_t)c->cfg.seed, (uint32_t)(c->cfg.seed >> 32));
    a.rk = philox_key_schedule(a.key);
    a.gen = gen;
    a.gen_dev = c->gen_dev_now;
    a.const_img = c->d_core_img; a.mut_size = c->tab_mut.size; a.mut_nsub = c->tab_mut.nsub; a.mut_kmax = c->tab_mut.kmax;
    a.hr_size = c->tab_hr.size;
    a.hr_lemire_t = c->N > 1 ? (uint32_t)((1ull << 32) % (c->N - 1)) : 0u; a.hr_kmax = c->tab_hr.kmax; a.hr_gen = c->hr_pending_gen;
    a.hr_nsub = c->hr_pending ? c->tab_hr.nsub : 0u;
    a.hr_k0 = c->hr_k0;
    a.dump_counters = c->d_dump_counters;
    a.dump_cap = c->dump_cap;
    a.d_mut_row = c->d_mut_row; a.d_mut_site = c->d_mut_site; a.d_mut_seq = c->d_mut_seq; a.d_mut_allele = c->d_mut_allele;
}

void fill_hr_args(pansim_ctx *c, HrArgs &h, uint32_t gen, uint8_t *state)
{
    memset(&h, 0, sizeof h);
    h.state = reinterpret_cast<uint32_t *>(state);
    h.n_rows = c->N;
    h.n_regions = c->n_regions;
    h.lemire_t = c->N > 1 ? (uint32_t)((1ull << 32) % (c->N - 1)) : 0u;
    h.region0 = c->region0;
    h.row_stride_words = c->core_stride / 4;
    h.site_limit = c->site_end;
    h.key = make_uint2((uint32_t)c->cfg.seed, (uint32_t)(c->cfg.seed >> 32));
    h.gen = gen;
    h.tab = c->tab_hr.d_thr; h.tab_words = c->tab_hr.size; h.nsub = c->tab_hr.nsub; h.kmax = c->tab_hr.kmax;
    h.slots = c->d_hr_slots;
    h.counts = c->d_hr_counts;
    h.slot_cap = c->hr_slot_cap;
    h.ovf = c->d_hr_ovf;
    h.ovf_count = c->d_hr_ovf_count + c->hr_parity;
    h.ovf_count_other = c->d_hr_ovf_count + (c->hr_parity ^ 1);
    h.ovf_cap = c->hr_ovf_cap;
    h.err_flag = c->d_err + 1;
    h.dump_counters = c->d_dump_counters;
    h.dump_cap = c->dump_cap;
    h.d_hr_rec = c->d_hr_rec; h.d_hr_locus = c->d_hr_locus; h.d_hr_donor = c->d_hr_donor; h.d_hr_seq = c->d_hr_seq;
    h.d_hr_value = c->d_hr_value;
}

// homologous recombination of generation `gen` on the rows the gather + SNP pass wrote into `state`,
// as two launches (core_hr.cuh)
int launch_core_hr(pansim_ctx *c, uint32_t gen, uint8_t *state, cudaStream_t st)
{
    HrArgs h;
    fill_hr_args(c, h, gen, state);
    const uint64_t qn = (c->N + HR_ROWS_PER_TASK - 1) / HR_ROWS_PER_TASK;
    const uint32_t grid = div_up64((uint64_t)c->n_regions * qn, HR_WARPS);
    if (c->dump_enabled)
        hr_collect_kernel<true><<<grid, HR_WARPS * 32, c->hr_smem, st>>>(h);
    else
        hr_collect_kernel<false><<<grid, HR_WARPS * 32, c->hr_smem, st>>>(h);
    LAUNCH_CHECK(c);
    hr_apply_kernel<<<div_up64((uint64_t)c->N * c->n_regions, HR_WARPS * HR_APPLY_ITEMS), HR_WARPS * 32, 0, st>>>(h);
    LAUNCH_CHECK(c);
    c->hr_parity ^= 1;
    c->core_version++;
    return 0;
}

// Order `stream` after the core step that is still in flight on stream_core (if any). The
// generate-mode entry points return without waiting for the core kernel, so that the selection
// chain of the next generation overlaps it; whoever touches the core buffers on `stream` joins first.
int ensure_core_joined(pansim_ctx *c)
{
    if (!c->core_unjoined) return 0;
    // ev_core_last, not ev_core_done[parents_idx]: sample_indices / next_generation rotate the parents
    // buffers without launching a core step, so the indexed event may belong to an older step
    CU(c, cudaStreamWaitEvent(c->stream, c->ev_core_last, 0));
    c->core_unjoined = false;
    return 0;
}

// Apply the pending recombination events to the current core buffer (deferred mode, core_mut.cuh).
// Every reader of the core state other than the generate-mode core step calls this first.
int core_materialize(pansim_ctx *c, cudaStream_t st)
{
    if (st == c->stream)
        if (int rc = ensure_core_joined(c)) return rc;
    if (st == c->stream_pairs && c->core_unjoined) CU(c, cudaStreamWaitEvent(st, c->ev_core_last, 0));   // c->stream stays unjoined
    if (!c->hr_pending) return 0;
    ScopedSpan sp(c, TG_CORE_HR, st);
    if (int rc = launch_core_hr(c, c->hr_pending_gen, c->core[c->core_cur], st)) return rc;
    c->hr_pending = false;
    return 0;
}

int launch_core_step(pansim_ctx *c, uint32_t gen, bool rng, cudaStream_t st)
{
    if (c->Ll == 0) return 0;
    if (st == c->stream)
        if (int rc = ensure_core_joined(c)) return rc;
    const bool hr = rng && c->tab_hr.nsub;
    const bool defer = c->hr_defer && !c->dump_enabled;
    // replay / plain gather, the event dump and the non-deferred mode work on materialised rows
    if (!rng || !defer)
        if (int rc = core_materialize(c, st)) return rc;
    CoreMutArgs a;
    fill_core_args(c, a, gen);
    const uint64_t per_cta = (uint64_t)CM_WARPS * a.items_per_warp;
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, ((uint64_t)c->N * c->n_regions + per_cta - 1) / per_cta);
    if (!rng || (!a.mut_nsub && !a.hr_nsub))
        core_mut_kernel<false, false><<<grid, CM_THREADS, c->core_smem, st>>>(a);
    else if (c->dump_enabled)
        core_mut_kernel<true, true><<<grid, CM_THREADS, c->core_smem, st>>>(a);
    else
        core_mut_kernel<true, false><<<grid, CM_THREADS, c->core_smem, st>>>(a);
    LAUNCH_CHECK(c);
    c->core_cur ^= 1;
    c->core_version++;
    c->hr_pending = false;
    if (hr) {
        if (defer) {
            c->hr_pending = true;
            c->hr_pending_gen = gen;
        } else {
            ScopedSpan sp(c, TG_CORE_HR, st);
            if (int rc = launch_core_hr(c, gen, c->core[c->core_cur], st)) return rc;
        }
    }
    return 0;
}

int require_state(pansim_ctx *c)
{
    if (!c->has_core || !c->has_acc) FAIL(c, PANSIM_ERR_STATE, "state not initialised: call pansim_set_initial or pansim_upload_*");
    return 0;
}

// Rotate to the next parents buffer. The buffer was last read by the core step
// issued three generations ago (and by the genealogy copy of that generation): the
// selection chain must not overwrite it before that kernel has finished.
int next_parents_buffer(pansim_ctx *c)
{
    c->parents_idx = (c->parents_idx + 1) % 3;
    const int i = c->parents_idx;
    if (c->core_done_valid[i]) CU(c, cudaStreamWaitEvent(c->stream, c->ev_core_done[i], 0));
    if (c->gen_done_valid[i]) CU(c, cudaStreamWaitEvent(c->stream, c->ev_gen_done[i], 0));
    c->d_parents = c->d_parents_buf[i];
    return 0;
}

// With genealogy recording on: append the current parents vector (ev_parents[i] recorded behind it) to the ring,
// one device-to-device copy on stream_gen into the slot the host already knows
int genealogy_record(pansim_ctx *c)
{
    if (!c->gen_cap) return 0;
    const int i = c->parents_idx;
    CU(c, cudaStreamWaitEvent(c->stream_gen, c->ev_parents[i], 0));
    uint32_t *dst = c->d_gen_ring + (size_t)(c->gen_total % c->gen_cap) * c->N;
    CU(c, cudaMemcpyAsync(dst, c->d_parents, (size_t)c->N * 4, cudaMemcpyDeviceToDevice, c->stream_gen));
    CU(c, cudaEventRecord(c->ev_gen_done[i], c->stream_gen));
    c->gen_done_valid[i] = true;
    c->gen_total++;
    c->gen_epoch++;
    return 0;
}

// the state was replaced: the record starts again (T = 0)
void genealogy_reset(pansim_ctx *c)
{
    c->gen_total = 0;
    c->gen_epoch++;
}

// accessory step on the chain stream, fused core step on the core stream; both
// read the current parents buffer, which must have been produced on c->stream.
// the core step of generation `gen` on the core stream, behind the parents of the current slot
int launch_core_part(pansim_ctx *c, uint32_t gen)
{
    const int i = c->parents_idx;
    CU(c, cudaEventRecord(c->ev_parents[i], c->stream));
    CU(c, cudaStreamWaitEvent(c->stream_core, c->ev_parents[i], 0));
    if (int rc = genealogy_record(c)) return rc;
    {
        ScopedSpan s(c, TG_CORE, c->stream_core);
        if (int rc = launch_core_step(c, gen, true, c->stream_core)) return rc;
    }
    CU(c, cudaEventRecord(c->ev_core_done[i], c->stream_core));
    CU(c, cudaEventRecord(c->ev_core_last, c->stream_core));
    c->core_done_valid[i] = true;
    c->core_unjoined = true;
    return 0;
}

int launch_population_steps(pansim_ctx *c, uint32_t gen)
{
    if (int rc = launch_core_part(c, gen)) return rc;
    {
        ScopedSpan s(c, TG_ACC);
        if (int rc = launch_acc_step(c, gen)) return rc;
    }
    return 0;
}

// after a batch of generations: later work on c->stream must see the core state
int join_core_stream(pansim_ctx *c) { return ensure_core_joined(c); }

// the selection chain of one generation: competition (if any) -> fitness -> parents
int launch_chain_select(pansim_ctx *c, uint32_t gen)
{
    ScopedSpan s(c, TG_SELECT);
    bool use_avg = false;
    if (c->cfg.competition_strength > 0.0) {          // main.rs:438-440
        if (int rc = launch_competition(c)) return rc;
        use_avg = true;
    }
    return launch_select(c, gen, use_avg);
}

__global__ void gen_base_add_kernel(uint32_t *gen_base, uint32_t n) { *gen_base += n; }

// Selection chain + accessory step of generation `gen` as one graph launch on c->stream. The graph of the
// current phase (parents slot, accessory buffer, ...) is captured on first use from the very calls the
// launch-by-launch path makes; the fitness kernel's side stream enters the capture through its fork event
// and is joined before the parent draw. Generation numbers inside are relative to the device word
// d_gen_base, which the last node advances by one, so a phase's graph serves every generation of that phase.
int chain_graph_step(pansim_ctx *c, uint32_t gen)
{
    if (!c->d_gen_base) {
        CU(c, cudaMalloc(&c->d_gen_base, sizeof(uint32_t)));
        CU(c, cudaMemsetAsync(c->d_gen_base, 0xFF, sizeof(uint32_t), c->stream));
    }
    if (int rc = join_fitness(c)) return rc;                    // nothing uncaptured may be waited for inside a capture
    if (c->cfg.competition_strength > 0.0)
        if (int rc = ensure_competition_buffers(c)) return rc;          // allocations are not capturable
    pansim_ctx::GraphKey key;
    memset(&key, 0, sizeof key);
    key.parents_idx = c->parents_idx; key.acc_cur = c->acc_cur; key.fitness_mode = c->fitness_mode;
    key.competition = c->cfg.competition_strength > 0.0; key.timing = c->timing_enabled && c->graph_spans; key.neutral = c->neutral;
    key.fitness_valid = c->fitness_valid; key.fitness_blocked = c->fitness_blocked;
    pansim_ctx::GraphEntry *ge = nullptr;
    for (auto *e : c->graphs)
        if (memcmp(&e->key, &key, sizeof key) == 0) ge = e;
    // the generation the graph's kernels add their relative 0 to
    if (c->gen_base_host != gen) {
        CU(c, cudaMemcpyAsync(c->d_gen_base, &gen, sizeof gen, cudaMemcpyHostToDevice, c->stream));      // pageable source: staged before the call returns
        c->gen_base_host = gen;
    }
    if (!ge) {
        ge = new pansim_ctx::GraphEntry();
        ge->key = key;
        const uint32_t launches0 = c->launches;
        CU(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        c->capturing = true;
        c->cap = ge;
        c->gen_dev_now = c->d_gen_base;
        int rc = launch_chain_select(c, 0u);
        if (!rc) {
            ScopedSpan s(c, TG_ACC);
            rc = launch_acc_step(c, 0u);
        }
        if (!rc) rc = join_fitness(c);
        if (!rc) {
            gen_base_add_kernel<<<1, 1, 0, c->stream>>>(c->d_gen_base, 1u);
            if (cudaGetLastError() != cudaSuccess) rc = PANSIM_ERR_CUDA;
        }
        c->capturing = false;
        c->cap = nullptr;
        c->gen_dev_now = nullptr;
        ge->kernels = c->launches - launches0 + 1u;
        c->launches = launches0;
        ge->acc_cur_after = c->acc_cur;
        ge->fitness_valid_after = c->fitness_valid;
        cudaGraph_t graph = nullptr;
        const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
        c->fitness_join_pending = false;                        // ev_join is a captured event now
        cudaError_t ei = cudaSuccess;
        if (!rc && e == cudaSuccess && graph) ei = cudaGraphInstantiate(&ge->exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (rc || e != cudaSuccess || ei != cudaSuccess || !ge->exec) {
            cudaGetLastError();
            ge->pool.destroy();
            delete ge;
            if (rc) return rc;
            FAIL(c, PANSIM_ERR_CUDA, "CUDA graph capture of the selection chain failed: %s", cudaGetErrorString(e != cudaSuccess ? e : ei));
        }
        c->graphs.push_back(ge);
    } else {
        // what the captured calls do to the host-side state
        c->acc_cur = ge->acc_cur_after;
        c->fitness_valid = ge->fitness_valid_after;
        c->avgdist_valid = key.competition;
    }
    CU(c, cudaGraphLaunch(ge->exec, c->stream));
    c->launches += ge->kernels;
    ge->used++;
    c->gen_base_host = gen + 1u;
    return 0;
}

int step_device(pansim_ctx *c, uint32_t gen)
{
    if (int rc = next_parents_buffer(c)) return rc;
    if (c->chain_graph_now && !c->capturing) {
        if (int rc = chain_graph_step(c, gen)) return rc;       // parents + accessory step of this generation
        if (int rc = launch_core_part(c, gen)) return rc;
    } else {
        if (int rc = launch_chain_select(c, gen)) return rc;
        if (int rc = launch_population_steps(c, gen)) return rc;
    }
    c->avgdist_valid = false;
    return 0;
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

void pansim_config_init(pansim_config *cfg)
{
    memset(cfg, 0, sizeof(*cfg));
    cfg->struct_size = (uint32_t)sizeof(*cfg);
    cfg->genome_size_penalty = 0.99;
}

const char *pansim_version(void) { return "pansim_b200 0.1 (sm_100a)"; }

const char *pansim_last_error(const pansim_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

double pansim_core_distance(uint32_t core_diff, uint64_t core_size)
{
    return (double)core_diff / (double)core_size;                 // population.rs:822
}

double pansim_acc_distance(uint32_t inter, uint32_t uni, uint32_t core_genes)
{
    return 1.0 - (((double)inter + (double)core_genes) / ((double)uni + (double)core_genes));   // :828-830
}

void pansim_destroy(pansim_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->cfg.device);
    if (c->comm && c->comm_owned) {
        if (c->stream) cudaStreamSynchronize(c->stream);
        nccl_api().CommDestroy(c->comm);
    }
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->stream_core) cudaStreamSynchronize(c->stream_core);
    if (c->stream_aux) cudaStreamSynchronize(c->stream_aux);
    void *ptrs[] = {c->core[0], c->core[1], c->d_hr_slots, c->d_hr_counts, c->d_hr_ovf, c->d_hr_ovf_count, c->d_core_img, c->acc[0], c->acc[1], c->d_parents_buf[0], c->d_parents_buf[1], c->d_parents_buf[2], c->d_lw, c->d_lethal, c->d_logfit, c->d_avgdist,
                    c->d_num_genes, c->d_inter_diag, c->d_tmp_a, c->d_tmp_b, c->d_weights, c->d_cum, c->d_err, c->d_inter, c->d_rcp, c->d_rowInvK, c->d_gain_planes,
                    c->d_gain_thr, c->tab_mut.d_thr, c->tab_hr.d_thr, c->d_r1, c->d_r2, c->d_cd, c->d_in, c->d_un,
                    c->d_planes, c->d_work_counter, c->d_replay, c->d_hkeys, c->d_hvals, c->d_stage, c->d_groups, c->d_partner, c->d_orig, c->d_batches, c->d_tile_slots, c->d_tile_orig, c->d_dump_counters, c->d_mut_row, c->d_mut_site,
                    c->d_mut_seq, c->d_mut_allele, c->d_hr_rec, c->d_hr_locus, c->d_hr_donor, c->d_hr_seq,
                    c->d_hr_value, c->d_dump_flip, c->d_dump_gain, c->d_anc, c->d_div, c->d_sfs,
                    c->d_vcf_counts, c->d_vcf_desc, c->d_vcf_off, c->d_vcf_block, c->d_vcf_bounds, c->d_vcf_nchunks,
                    c->d_fa_block, c->d_fa_const, c->d_fa_cols};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (auto *b : {&c->ld, &c->ld_halo}) {
        void *lp[] = {b->counts, b->block, b->rank, b->pos, b->a, b->x, b->inv};
        for (void *p : lp)
            if (p) cudaFree(p);
    }
    if (c->d_ld_tiles) cudaFree(c->d_ld_tiles);
    if (c->d_ld_bins) cudaFree(c->d_ld_bins);
    if (c->h_ld) cudaFreeHost(c->h_ld);
    if (c->h_fa) cudaFreeHost(c->h_fa);
    if (c->h_ld_bins) cudaFreeHost(c->h_ld_bins);
    if (c->ev_ld) cudaEventDestroy(c->ev_ld);
    {
        void *gp[] = {c->gl.counts, c->gl.rank, c->gl.a, c->gl.grp, c->gl.x, c->gl.inv, c->gl.block, c->gl.out};
        for (void *p : gp)
            if (p) cudaFree(p);
        if (c->gl.h_out) cudaFreeHost(c->gl.h_out);
        for (void *p : {(void *)c->ga.orders, (void *)c->ga.delta, (void *)c->ga.summary, (void *)c->ga.curves, (void *)c->ga.spectrum})
            if (p) cudaFree(p);
    }
    if (c->stream_gen) { cudaStreamSynchronize(c->stream_gen); cudaStreamDestroy(c->stream_gen); }
    for (auto e : c->ev_gen_done) if (e) cudaEventDestroy(e);
    for (void *p : {(void *)c->d_gen_ring, (void *)c->d_gen_scratch, (void *)c->d_gen_pairs}) if (p) cudaFree(p);
    for (auto *e : c->graphs) {
        if (e->exec) cudaGraphExecDestroy(e->exec);
        e->pool.destroy();
        delete e;
    }
    if (c->d_gen_base) cudaFree(c->d_gen_base);
    if (c->h_parents) cudaFreeHost(c->h_parents);
    for (int i = 0; i < 3; i++) {
        if (c->h_parents_up[i]) cudaFreeHost(c->h_parents_up[i]);
        if (c->ev_h2d[i]) cudaEventDestroy(c->ev_h2d[i]);
    }
    if (c->h_avg) cudaFreeHost(c->h_avg);
    for (int b = 0; b < 2; b++) {
        if (c->h_txt[b]) cudaFreeHost(c->h_txt[b]);
        if (c->d_txt[b]) cudaFree(c->d_txt[b]);
        if (c->ev_txt[b]) cudaEventDestroy(c->ev_txt[b]);
    }
    if (c->h_stats) cudaFreeHost(c->h_stats);
    if (c->d_stats) cudaFree(c->d_stats);
    if (c->h_div) cudaFreeHost(c->h_div);
    if (c->h_sfs) cudaFreeHost(c->h_sfs);
    for (auto q : c->d_cnt2) if (q) cudaFree(q);
    for (int i = 0; i < 2; i++) {
        if (c->ev_pairs[i]) cudaEventDestroy(c->ev_pairs[i]);
        if (c->ev_stats[i]) cudaEventDestroy(c->ev_stats[i]);
    }
    for (auto st : c->stream_stats2) if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    if (c->stream_pairs) { cudaStreamSynchronize(c->stream_pairs); cudaStreamDestroy(c->stream_pairs); }
    if (c->ev_acc_done) cudaEventDestroy(c->ev_acc_done);
    if (c->ev_mat) cudaEventDestroy(c->ev_mat);
    if (c->h_err) cudaFreeHost(c->h_err);
    c->pool.destroy();
    for (int i = 0; i < 3; i++) {
        if (c->ev_parents[i]) cudaEventDestroy(c->ev_parents[i]);
        if (c->ev_core_done[i]) cudaEventDestroy(c->ev_core_done[i]);
    }
    if (c->ev_core_last) cudaEventDestroy(c->ev_core_last);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->stream_aux) cudaStreamDestroy(c->stream_aux);
    if (c->stream_core) cudaStreamDestroy(c->stream_core);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int pansim_create(const pansim_config *cfg, pansim_ctx **out)
{
    if (!cfg || !out) { g_create_error = "null argument"; return PANSIM_ERR_INVALID; }
    *out = nullptr;
    if (cfg->struct_size != sizeof(pansim_config)) { g_create_error = "pansim_config.struct_size mismatch"; return PANSIM_ERR_INVALID; }
    pansim_ctx *c = new pansim_ctx();
    c->cfg = *cfg;
    auto fail = [&](int code) { g_create_error = c->err; pansim_destroy(c); return code; };
    auto body = [&]() -> int {
        if (cfg->pop_size < 1) FAIL(c, PANSIM_ERR_INVALID, "pop_size must be >= 1");
        if (cfg->core_size < 1) FAIL(c, PANSIM_ERR_INVALID, "core_size must be >= 1");
        if (cfg->core_size > 0xFFFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "core_size above 2^32-1 is not supported");
        if (cfg->n_compartments > 2) FAIL(c, PANSIM_ERR_INVALID, "at most two gene compartments (main.rs:341-367)");
        c->N = cfg->pop_size;
        c->G = cfg->pan_size;
        c->L = cfg->core_size;
        c->site_begin = cfg->site_begin;
        c->site_end = cfg->site_end;
        if (c->site_begin == 0 && c->site_end == 0) c->site_end = c->L;
        if (c->site_end > c->L || c->site_begin > c->site_end) FAIL(c, PANSIM_ERR_INVALID, "bad column shard [%llu,%llu)", (unsigned long long)c->site_begin, (unsigned long long)c->site_end);
        if (c->site_begin % PANSIM_SITE_ALIGN && c->site_begin != c->site_end) FAIL(c, PANSIM_ERR_INVALID, "site_begin must be a multiple of %u", PANSIM_SITE_ALIGN);
        if (c->site_end != c->L && c->site_end % PANSIM_SITE_ALIGN && c->site_begin != c->site_end) FAIL(c, PANSIM_ERR_INVALID, "site_end must be core_size or a multiple of %u", PANSIM_SITE_ALIGN);
        c->Ll = c->site_end - c->site_begin;
        c->region0 = (uint32_t)(c->site_begin / REGION_SITES);
        c->n_regions = (uint32_t)((c->Ll + REGION_SITES - 1) / REGION_SITES);
        c->core_stride = (uint64_t)c->n_regions * REGION_BYTES;
        if ((uint64_t)c->N * c->n_regions >= 0x7FFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "pop_size x regions exceeds 2^31");
        c->acc_words = (c->G + 31) / 32;
        c->acc_stride_words = ((c->acc_words + 3) / 4) * 4;
        if (c->acc_stride_words == 0) c->acc_stride_words = 4;
        for (uint32_t k = 0; k < cfg->n_compartments; k++)
            if (cfg->comp_lo[k] > cfg->comp_hi[k] || cfg->comp_hi[k] > c->G) FAIL(c, PANSIM_ERR_INVALID, "compartment %u out of range", k);
        if ((cfg->hr_mean > 0.0 || cfg->hgt_mean[0] > 0.0 || cfg->hgt_mean[1] > 0.0) && c->N < 2)
            FAIL(c, PANSIM_ERR_INVALID, "recombination needs pop_size >= 2 (Uniform::new(0, nrows-1), population.rs:584)");
        if (cfg->core_mut_mean < 0 || cfg->hr_mean < 0) FAIL(c, PANSIM_ERR_INVALID, "negative event mean");
        if (!(cfg->genome_size_penalty > 0.0)) FAIL(c, PANSIM_ERR_INVALID, "genome_size_penalty must be > 0");

        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) FAIL(c, PANSIM_ERR_CUDA, "no CUDA device: libpansim_b200 has no CPU fallback");
        if (cfg->device < 0 || cfg->device >= ndev) FAIL(c, PANSIM_ERR_INVALID, "device %d out of range (0..%d)", cfg->device, ndev - 1);
        CU(c, cudaSetDevice(cfg->device));
        cudaDeviceProp prop;
        CU(c, cudaGetDeviceProperties(&prop, cfg->device));
        if (prop.major < 10) FAIL(c, PANSIM_ERR_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
        c->sm_count = prop.multiProcessorCount;
        {
            // the accessory/selection chain is latency-critical and tiny: give it priority over the core step
            int lo = 0, hi = 0;
            CU(c, cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CU(c, cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, hi));
            CU(c, cudaStreamCreateWithPriority(&c->stream_core, cudaStreamNonBlocking, lo));
            CU(c, cudaStreamCreateWithPriority(&c->stream_aux, cudaStreamNonBlocking, hi));
            c->ps = c->stream;
            CU(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
            CU(c, cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        }
        CU(c, cudaEventCreateWithFlags(&c->ev_core_last, cudaEventDisableTiming));
        for (int i = 0; i < 3; i++) {
            CU(c, cudaEventCreateWithFlags(&c->ev_parents[i], cudaEventDisableTiming));
            CU(c, cudaEventCreateWithFlags(&c->ev_core_done[i], cudaEventDisableTiming));
        }

        // per-cell rates (SURVEY.md 8a rows M, R)
        const double rate_mut = cfg->core_mut_mean / (double)c->L;
        const double rate_hr = cfg->hr_mean / (double)c->L;
        c->p_mut_site = -std::expm1(-rate_mut);
        c->p_hr_site = -std::expm1(-rate_hr);
        build_poisson_table(rate_mut * BLOCK_SITES, c->tab_mut);
        build_poisson_table(rate_hr * REGION_SITES, c->tab_hr);
        if (c->tab_hr.size < 32) { c->tab_hr.size = 32; c->tab_hr.thr.resize(32, 0xFFFFFFFFu); }      // whole warps of thresholds (core_hr.cuh)
        {
            // window of 32 thresholds around the median of the count distribution
            uint32_t med = 0;
            while (med < c->tab_hr.kmax && c->tab_hr.thr[med] < 0x80000000u) med++;
            c->hr_k0 = med > 16u ? med - 16u : 0u;
            if (c->hr_k0 + 32u > c->tab_hr.size) c->hr_k0 = c->tab_hr.size - 32u;
        }
        if ((double)c->tab_hr.nsub * c->tab_hr.kmax > 1.5e7) FAIL(c, PANSIM_ERR_INVALID, "recombination rate too high (more than ~1e7 events per 8192-site region)");
        {
            // constant image of the core kernel: allele-digit table, SNP count table, recombination thresholds
            const uint32_t hr_size = c->tab_hr.nsub ? c->tab_hr.size : 0u;
            std::vector<uint8_t> img(core_mut_const_bytes(c->tab_mut.size, hr_size), 0);
            uint32_t *lut = reinterpret_cast<uint32_t *>(img.data());
            for (uint32_t v = 0; v < CM_LUT_ENTRIES; v++) {
                // entry v = base-3 digits of v; word j = allele code (digit j) + 1 in all 16 cells: {C,G,T} (population.rs:531)
                uint32_t t = v;
                for (int j = 0; j < 4; j++) { lut[v * 4 + j] = (t % 3u + 1u) * 0x55555555u; t /= 3u; }
            }
            const std::vector<uint32_t> mimg = poisson_fast_image(c->tab_mut);
            memcpy(img.data() + CM_LUT_BYTES, mimg.data(), mimg.size() * 4);
            if (hr_size) memcpy(img.data() + CM_LUT_BYTES + mimg.size() * 4, c->tab_hr.thr.data(), (size_t)hr_size * 4);
            CU(c, cudaMalloc(&c->d_core_img, img.size()));
            CU(c, cudaMemcpy(c->d_core_img, img.data(), img.size(), cudaMemcpyHostToDevice));
        }
        {
            CU(c, cudaMalloc(&c->tab_hr.d_thr, c->tab_hr.thr.size() * sizeof(uint32_t)));      // thresholds only (core_hr.cuh)
            CU(c, cudaMemcpy(c->tab_hr.d_thr, c->tab_hr.thr.data(), c->tab_hr.thr.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        }
        for (uint32_t k = 0; k < cfg->n_compartments; k++) {
            const double sites = (double)(cfg->comp_hi[k] - cfg->comp_lo[k]);
            if (sites > 0 && cfg->acc_mut_mean[k] > 0) {
                const double rate = cfg->acc_mut_mean[k] / sites;            // per gene per row
                const double p = -0.5 * std::expm1(-2.0 * rate);
                c->flip_p[k] = p;
                const double t = std::rint(p * 4294967296.0);
                c->flip_thr[k] = t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
            }
            if (cfg->hgt_mean[k] > 0) c->hgt_scale[k] = cfg->hgt_mean[k] / (double)(c->N - 1);
        }

        const size_t core_bytes = (size_t)c->N * c->core_stride;
        const size_t acc_bytes = (size_t)c->N * c->acc_stride_words * 4;
        for (int b = 0; b < 2; b++) {
            if (core_bytes) {
                if (cudaMalloc(&c->core[b], core_bytes) != cudaSuccess) FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (packed core) failed", core_bytes);
                CU(c, cudaMemset(c->core[b], 0, core_bytes));
            }
            CU(c, cudaMalloc(&c->acc[b], acc_bytes));
            CU(c, cudaMemset(c->acc[b], 0, acc_bytes));
        }
        // the bit-exact sequential fitness chain is kept up to 2^25 accessory cells (cfg1-3: 4e6)
        c->fitness_blocked = (uint64_t)c->N * c->G > (1ull << 25);
        if (const char *e = getenv("PANSIM_FITNESS_BLOCKED")) c->fitness_blocked = atoi(e) != 0;
        if (const char *e = getenv("PANSIM_TILES2")) c->use_tiles2 = atoi(e) != 0;
        if (const char *e = getenv("PANSIM_GRAPH")) c->use_graph = atoi(e) != 0;
        if (const char *e = getenv("PANSIM_GRAPH_SPANS")) c->graph_spans = atoi(e) != 0;
        if (const char *e = getenv("PANSIM_FINE_TIMING")) c->fine_timing = atoi(e) != 0;
        if (const char *e = getenv("PANSIM_PDL")) c->use_pdl = atoi(e);
        if (c->tab_hr.nsub && core_bytes) {
            // recombination slots: per (region, row) item room for mean + 6 sigma changed cells (a multiple of 32,
            // 32 when the mean is small); the rare item that needs more spills to the overflow list
            const double m_item = rate_hr * REGION_SITES;
            uint32_t cap = 32;
            if (m_item > 24.0) cap = 32u * (uint32_t)std::ceil((m_item + 6.0 * std::sqrt(m_item)) / 32.0);
            if (cap > 8192) cap = 8192;                               // a region has 8192 cells
            c->hr_slot_cap = cap;
            const size_t items = (size_t)c->N * c->n_regions;
            if (cudaMalloc(&c->d_hr_slots, items * cap * 2) != cudaSuccess) FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (recombination slots) failed", items * cap * 2);
            CU(c, cudaMalloc(&c->d_hr_counts, items * 2));
            CU(c, cudaMemset(c->d_hr_counts, 0, items * 2));
            const double mean = rate_hr * (double)c->Ll * (double)c->N;
            c->hr_ovf_cap = (uint32_t)std::min(4.0e8, 65536.0 + 0.02 * mean);
            CU(c, cudaMalloc(&c->d_hr_ovf, (size_t)c->hr_ovf_cap * 8));
            CU(c, cudaMalloc(&c->d_hr_ovf_count, 2 * sizeof(uint32_t)));
            CU(c, cudaMemset(c->d_hr_ovf_count, 0, 2 * sizeof(uint32_t)));
            c->hr_smem = hr_collect_smem_bytes(c->tab_hr.size);
        }
        const size_t n = c->N;
        for (int i = 0; i < 3; i++) CU(c, cudaMalloc(&c->d_parents_buf[i], (n + 1) * 4));   // + status word (select.cuh)
        CU(c, cudaMallocHost(&c->h_parents, (n + 1) * 4));
        for (int i = 0; i < 3; i++) {
            CU(c, cudaMallocHost(&c->h_parents_up[i], n * 4));
            CU(c, cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming));
        }
        CU(c, cudaMallocHost(&c->h_avg, n * 8));
        CU(c, cudaMallocHost(&c->h_err, 2 * sizeof(int)));
        c->h_err[0] = c->h_err[1] = 0;
        c->d_parents = c->d_parents_buf[0];
        CU(c, cudaMalloc(&c->d_lw, (size_t)(c->G ? c->G : 1) * 8));
        CU(c, cudaMemset(c->d_lw, 0, (size_t)(c->G ? c->G : 1) * 8));
        CU(c, cudaMalloc(&c->d_lethal, (size_t)(c->acc_words ? c->acc_words : 1) * 4));
        CU(c, cudaMemset(c->d_lethal, 0, (size_t)(c->acc_words ? c->acc_words : 1) * 4));
        if (const char *e = getenv("PANSIM_FITNESS_MODE")) c->fitness_mode = atoi(e);
        CU(c, cudaMalloc(&c->d_logfit, n * 8));
        CU(c, cudaMalloc(&c->d_avgdist, n * 8));
        CU(c, cudaMalloc(&c->d_num_genes, n * 4));
        CU(c, cudaMalloc(&c->d_inter_diag, n * 4));
        CU(c, cudaMalloc(&c->d_tmp_a, n * 8));
        CU(c, cudaMalloc(&c->d_tmp_b, n * 8));
        CU(c, cudaMalloc(&c->d_weights, n * 8));
        CU(c, cudaMalloc(&c->d_cum, n * 8));
        CU(c, cudaMalloc(&c->d_err, 2 * sizeof(int)));
        CU(c, cudaMemset(c->d_err, 0, 2 * sizeof(int)));
        CU(c, cudaMalloc(&c->d_rowInvK, 2 * n * 8));
        CU(c, cudaMalloc(&c->d_gain_thr, (size_t)(c->G ? c->G : 1) * 4));
        // one 32-word plane block per word of the row STRIDE: acc_hgt_apply_kernel runs over the padded rows
        CU(c, cudaMalloc(&c->d_gain_planes, (size_t)c->acc_stride_words * 32 * 4));
        CU(c, cudaMemset(c->d_gain_planes, 0, (size_t)c->acc_stride_words * 32 * 4));
        CU(c, cudaMalloc(&c->d_dump_counters, 2 * sizeof(uint32_t)));
        CU(c, cudaMemset(c->d_dump_counters, 0, 2 * sizeof(uint32_t)));

        // launch shape of the core kernel
        c->core_smem = core_mut_smem_bytes(c->tab_mut.size, c->tab_hr.nsub ? c->tab_hr.size : 0u);
        {
            // at most CM_RESIDENT_CTAS core CTAs per SM: the registers and shared memory they leave free hold
            // the selection chain's CTAs while the core kernel runs (core_mut.cuh)
            const size_t fit = prop.sharedMemPerMultiprocessor / (CM_RESIDENT_CTAS + 1) + 1;
            if (fit > prop.reservedSharedMemPerBlock)
                c->core_smem = std::max(c->core_smem, std::min(fit - prop.reservedSharedMemPerBlock, prop.sharedMemPerBlockOptin));
        }
        if (const char *e = getenv("PANSIM_CORE_SMEM_PAD_KB")) c->core_smem += (size_t)std::max(0, atoi(e)) * 1024;   // experiment: cap the CTAs per SM
        if (const char *e = getenv("PANSIM_HR_DEFER")) c->hr_defer = atoi(e) != 0;
        CU(c, cudaFuncSetAttribute(core_mut_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->core_smem));
        CU(c, cudaFuncSetAttribute(core_mut_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->core_smem));
        CU(c, cudaFuncSetAttribute(core_mut_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->core_smem));
        int occ = 0;
        CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, core_mut_kernel<true, false>, CM_THREADS, c->core_smem));
        if (occ < 1) FAIL(c, PANSIM_ERR_CUDA, "core_mut_kernel does not fit on an SM (smem %zu)", c->core_smem);
        c->core_occupancy = occ;
        const uint64_t items = (uint64_t)c->N * c->n_regions;
        // short-lived CTAs (3 items per warp) where the selection chain is on the critical path; longer ones
        // (up to 12) once the core step has hundreds of items per resident warp and the chain hides under it
        c->core_items_per_warp = (uint32_t)std::min<uint64_t>(12, std::max<uint64_t>(3, items / ((uint64_t)c->sm_count * occ * CM_WARPS * 40)));
        if (const char *e = getenv("PANSIM_CORE_CTAS_PER_SM")) {
            // long-lived CTAs: a grid of (CTAs per SM) x (SM count), each warp takes its share of the items
            const uint64_t ctas = (uint64_t)std::max(1, atoi(e)) * c->sm_count;
            c->core_items_per_warp = (uint32_t)std::max<uint64_t>(1, (items + ctas * CM_WARPS - 1) / (ctas * CM_WARPS));
        }
        if (const char *e = getenv("PANSIM_CORE_ITEMS_PER_WARP")) c->core_items_per_warp = (uint32_t)std::max(1, atoi(e));
        // Items per warp in the device-resident batch. Short-lived CTAs turn SM slots over often, so the chain
        // (select + accessory step) of the NEXT generation finds room sooner; longer ones pay the per-warp
        // prologue less often. Measured at cfg2 with the two-stage kernel at 4 resident CTAs (us per
        // generation): 4 items 146.9-147.4, 5 items 143.8-144.3, 6 items 152.6-153.0.
        c->core_items_batch = std::max(c->core_items_per_warp, 5u);
        if (const char *e = getenv("PANSIM_CORE_ITEMS_BATCH")) c->core_items_batch = (uint32_t)std::max(0, atoi(e));
        const uint64_t per_cta = (uint64_t)CM_WARPS * c->core_items_per_warp;
        c->core_grid = (uint32_t)std::max<uint64_t>(1, (items + per_cta - 1) / per_cta);
        if (c->tab_hr.nsub && core_bytes && c->hr_smem > 48 * 1024) {
            CU(c, cudaFuncSetAttribute(hr_collect_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->hr_smem));
            CU(c, cudaFuncSetAttribute(hr_collect_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->hr_smem));
        }
        return 0;
    };
    int rc = body();
    if (rc) return fail(rc);
    *out = c;
    return PANSIM_OK;
}

int pansim_get_info(pansim_ctx *c, pansim_info *o)
{
    if (!c || !o) return PANSIM_ERR_INVALID;
    memset(o, 0, sizeof *o);
    o->core_row_stride_bytes = c->core_stride;
    o->acc_row_stride_bytes = (uint64_t)c->acc_stride_words * 4;
    o->local_sites = c->Ll;
    o->core_state_bytes = (uint64_t)c->N * c->core_stride;
    o->algorithmic_bytes_per_generation = 2ull * c->N * ((c->Ll + 3) / 4) + 2ull * c->N * ((c->G + 7) / 8);
    o->algorithmic_bytes_per_pair = 2ull * ((c->Ll + 3) / 4) + 2ull * ((c->G + 7) / 8);
    o->sm_count = (uint32_t)c->sm_count;
    o->core_step_grid = c->core_grid;
    o->core_step_block = CM_THREADS;
    o->core_step_smem = (uint32_t)c->core_smem;
    return 0;
}

int pansim_get_rates(pansim_ctx *c, double *out)
{
    if (!c || !out) return PANSIM_ERR_INVALID;
    out[0] = c->p_mut_site; out[1] = c->p_hr_site; out[2] = c->flip_p[0]; out[3] = c->flip_p[1];
    return 0;
}

int pansim_set_timing(pansim_ctx *c, int enabled)
{
    if (!c) return PANSIM_ERR_INVALID;
    c->timing_enabled = enabled != 0;
    return 0;
}

int pansim_get_timing(pansim_ctx *c, pansim_timing *o)
{
    if (!c || !o) return PANSIM_ERR_INVALID;
    memset(o, 0, sizeof *o);
    o->launches = c->launches;
    CU(c, cudaSetDevice(c->cfg.device));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaStreamSynchronize(c->stream_core));
    if (!c->timing_enabled || !c->t_begin || !c->t_end) return 0;
    CU(c, cudaEventElapsedTime(&o->total_ms, c->t_begin, c->t_end));
    float g[TG_COUNT] = {0};
    for (auto &s : c->spans) {
        float ms = 0;
        CU(c, cudaEventElapsedTime(&ms, s.a, s.b));
        g[s.group] += ms;
    }
    for (auto *e : c->graphs)       // the record nodes of a graph hold the times of its LAST launch: scaled to its launches in this call
        if (e->used)
            for (auto &s : e->spans) {
                float ms = 0;
                if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) g[s.group] += ms * (float)e->used;
                else cudaGetLastError();
            }
    if (c->fine_timing)
        fprintf(stderr, "[pansim fine timing, ms over the batch] inter(+fitness join) %.4f avg %.4f select %.4f flip %.4f gain %.4f hgt %.4f | groups: select %.4f acc %.4f core %.4f\n",
                g[TG_D_INTER], g[TG_D_AVG], g[TG_D_SEL], g[TG_D_FLIP], g[TG_D_GAIN], g[TG_D_HGT], g[TG_SELECT], g[TG_ACC], g[TG_CORE]);
    o->select_ms = g[TG_SELECT]; o->acc_step_ms = g[TG_ACC]; o->core_step_ms = g[TG_CORE];
    o->core_hr_ms = g[TG_CORE_HR];
    o->pair_core_ms = g[TG_PAIR_CORE]; o->pair_acc_ms = g[TG_PAIR_ACC];
    return 0;
}

// ---- state ----------------------------------------------------------------
int pansim_upload_core(pansim_ctx *c, const uint8_t *bytes)
{
    if (!c || !bytes) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->Ll == 0) { c->has_core = true; genealogy_reset(c); return 0; }
    // stage at most ~256 MiB of host bytes at a time
    uint32_t rows_per = (uint32_t)std::max<uint64_t>(1, (256ull << 20) / c->Ll);
    if (rows_per > c->N) rows_per = c->N;
    if (int rc = ensure_stage(c, (size_t)rows_per * c->Ll)) return rc;
    if (int rc = ensure_core_joined(c)) return rc;
    uint8_t *dst = c->core[c->core_cur];
    c->hr_pending = false;                       // the state is replaced
    c->core_version++;
    genealogy_reset(c);
    for (uint32_t r0 = 0; r0 < c->N; r0 += rows_per) {
        const uint32_t nr = std::min(rows_per, c->N - r0);
        CU(c, cudaMemcpyAsync(c->d_stage, bytes + (size_t)r0 * c->Ll, (size_t)nr * c->Ll, cudaMemcpyHostToDevice, c->stream));
        const uint64_t words = (uint64_t)nr * (c->core_stride / 4);
        pack_core_kernel<<<div_up64(words, 256), 256, 0, c->stream>>>(c->d_stage, c->Ll, r0, nr, dst, c->core_stride, c->d_err);
        LAUNCH_CHECK(c);
    }
    if (int rc = check_device_flag(c, PANSIM_ERR_INVALID, "core matrix holds a byte that is not one-hot {1,2,4,8}")) return rc;
    c->has_core = true;
    return 0;
}

int pansim_upload_acc(pansim_ctx *c, const uint8_t *bytes)
{
    if (!c || (!bytes && c->G)) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = join_fitness(c)) return rc;
    genealogy_reset(c);
    if (c->G) {
        if (int rc = ensure_stage(c, (size_t)c->N * c->G)) return rc;
        CU(c, cudaMemcpyAsync(c->d_stage, bytes, (size_t)c->N * c->G, cudaMemcpyHostToDevice, c->stream));
        const uint64_t words = (uint64_t)c->N * c->acc_stride_words;
        pack_acc_kernel<<<div_up64(words, 256), 256, 0, c->stream>>>(c->d_stage, c->G, c->N, c->acc[c->acc_cur], c->acc_stride_words, c->d_err);
        LAUNCH_CHECK(c);
        if (int rc = check_device_flag(c, PANSIM_ERR_INVALID, "accessory matrix holds a byte that is not 0/1")) return rc;
    }
    c->has_acc = true;
    c->avgdist_valid = false;
    c->fitness_valid = false;
    return 0;
}

int pansim_set_initial(pansim_ctx *c, const uint8_t *core_row, const uint8_t *acc_row)
{
    if (!c || !core_row || (!acc_row && c->G)) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    genealogy_reset(c);
    if (c->Ll) {
        if (int rc = ensure_stage(c, (size_t)c->Ll)) return rc;
        CU(c, cudaMemcpyAsync(c->d_stage, core_row + c->site_begin, c->Ll, cudaMemcpyHostToDevice, c->stream));
        if (int rc = ensure_core_joined(c)) return rc;
        uint8_t *dst = c->core[c->core_cur];
        c->hr_pending = false;                   // the state is replaced
        c->core_version++;
        pack_core_kernel<<<div_up64(c->core_stride / 4, 256), 256, 0, c->stream>>>(c->d_stage, c->Ll, 0, 1, dst, c->core_stride, c->d_err);
        LAUNCH_CHECK(c);
        // the clonal row is the ancestral row of the SFS (pansim_core_diversity); uploads leave it alone
        if (!c->d_anc) CU(c, cudaMalloc(&c->d_anc, c->core_stride));
        CU(c, cudaMemcpyAsync(c->d_anc, dst, c->core_stride, cudaMemcpyDeviceToDevice, c->stream));
        if (c->N > 1) {
            const uint64_t vecs = (uint64_t)(c->N - 1) * (c->core_stride / 16);
            replicate_row_kernel<<<div_up64(vecs, 256), 256, 0, c->stream>>>(dst, c->core_stride, c->N);
            LAUNCH_CHECK(c);
        }
        if (int rc = check_device_flag(c, PANSIM_ERR_INVALID, "core row holds a byte that is not one-hot {1,2,4,8}")) return rc;
    }
    c->has_core = true;
    c->has_anc = true;
    if (c->G) {
        std::vector<uint8_t> full((size_t)c->N * c->G);
        for (uint32_t r = 0; r < c->N; r++) memcpy(full.data() + (size_t)r * c->G, acc_row, c->G);
        return pansim_upload_acc(c, full.data());
    }
    c->has_acc = true;
    return 0;
}

int pansim_download_core(pansim_ctx *c, uint8_t *out)
{
    if (!c || !out) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->Ll == 0) return 0;
    if (int rc = core_materialize(c, c->stream)) return rc;
    if (int rc = check_hr_flag(c)) return rc;
    uint32_t rows_per = (uint32_t)std::max<uint64_t>(1, (256ull << 20) / c->Ll);
    if (rows_per > c->N) rows_per = c->N;
    if (int rc = ensure_stage(c, (size_t)rows_per * c->Ll)) return rc;
    const uint64_t wpr = (c->Ll + 15) / 16;
    for (uint32_t r0 = 0; r0 < c->N; r0 += rows_per) {
        const uint32_t nr = std::min(rows_per, c->N - r0);
        unpack_core_kernel<<<div_up64((uint64_t)nr * wpr, 256), 256, 0, c->stream>>>(c->core[c->core_cur], c->core_stride, c->Ll, r0, nr, c->d_stage);
        LAUNCH_CHECK(c);
        CU(c, cudaMemcpyAsync(out + (size_t)r0 * c->Ll, c->d_stage, (size_t)nr * c->Ll, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return 0;
}

// the two device and two pinned host chunks of the text exports, each at least `bytes`
static int ensure_txt_staging(pansim_ctx *c, size_t bytes, const char *what)
{
    if (bytes <= c->txt_cap) return 0;
    for (int b = 0; b < 2; b++) {
        if (c->h_txt[b]) cudaFreeHost(c->h_txt[b]);
        if (c->d_txt[b]) cudaFree(c->d_txt[b]);
        c->h_txt[b] = nullptr; c->d_txt[b] = nullptr;
    }
    c->txt_cap = 0;
    for (int b = 0; b < 2; b++) {
        if (cudaMallocHost(&c->h_txt[b], bytes) != cudaSuccess || cudaMalloc(&c->d_txt[b], bytes) != cudaSuccess)
            FAIL(c, PANSIM_ERR_NOMEM, "staging buffers of %zu bytes for the %s export failed", bytes, what);
        if (!c->ev_txt[b]) CU(c, cudaEventCreateWithFlags(&c->ev_txt[b], cudaEventDisableTiming));
    }
    c->txt_cap = bytes;
    return 0;
}

// Text expanded on the GPU chunk by chunk and streamed out through two pinned host buffers: while chunk k
// is handed to `sink` (copied into the caller's buffer, or written to a file), the kernel and the
// device-to-host copy of chunk k+1 are in flight. expand(k, dst, &bytes) enqueues the kernel of chunk k on
// c->stream, which writes `bytes` (at most cap) bytes at dst; sink(chunk_ptr, bytes) returns 0 to go on.
extern "C++" {
template <typename Expand, typename Sink>
static int stream_text_chunks(pansim_ctx *c, size_t n_chunks, size_t cap, const char *what, Expand &&expand, Sink &&sink)
{
    if (n_chunks == 0) return 0;
    if (int rc = ensure_txt_staging(c, cap, what)) return rc;
    size_t bytes[2] = {0, 0};
    auto enqueue = [&](size_t k, int b) -> int {
        if (int rc = expand(k, c->d_txt[b], &bytes[b])) return rc;
        CU(c, cudaMemcpyAsync(c->h_txt[b], c->d_txt[b], bytes[b], cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaEventRecord(c->ev_txt[b], c->stream));
        return 0;
    };
    int b = 0;
    if (int rc = enqueue(0, 0)) return rc;
    for (size_t k = 0; k < n_chunks; k++, b ^= 1) {
        if (k + 1 < n_chunks)
            if (int rc = enqueue(k + 1, b ^ 1)) return rc;                 // next chunk in flight while this one is consumed
        CU(c, cudaEventSynchronize(c->ev_txt[b]));
        if (sink(c->h_txt[b], bytes[b])) FAIL(c, PANSIM_ERR_INVALID, "%s export: the sink failed (short write?)", what);
    }
    return 0;
}

// `A,C,G,T\n` rows of _core_genome.csv (population.rs:877-879), a chunk of rows per kernel
template <typename Sink>
static int export_core_csv_stream(pansim_ctx *c, uint32_t row_begin, uint32_t row_end, Sink &&sink)
{
    if (row_begin > row_end || row_end > c->N) FAIL(c, PANSIM_ERR_INVALID, "rows [%u, %u) out of range", row_begin, row_end);
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->Ll == 0 || row_begin == row_end) return 0;
    if (int rc = core_materialize(c, c->stream)) return rc;
    if (int rc = check_hr_flag(c)) return rc;
    const size_t row_bytes = 2 * (size_t)c->Ll;
    const size_t chunk_target = 32ull << 20;
    const uint32_t rows_per = (uint32_t)std::max<size_t>(1, chunk_target / row_bytes);
    const size_t chunk_bytes = (size_t)std::min<uint32_t>(rows_per, row_end - row_begin) * row_bytes;
    const size_t n_chunks = (row_end - row_begin + (size_t)rows_per - 1) / rows_per;
    const uint64_t wpr = (c->Ll + 15) / 16;
    return stream_text_chunks(c, n_chunks, chunk_bytes, "CSV", [&](size_t k, char *dst, size_t *bytes) -> int {
        const uint32_t r0 = row_begin + (uint32_t)k * rows_per;
        const uint32_t nr = std::min(rows_per, row_end - r0);
        export_core_csv_kernel<<<div_up64((uint64_t)nr * wpr, 256), 256, 0, c->stream>>>(c->core[c->core_cur], c->core_stride, c->Ll, r0, nr, dst);
        LAUNCH_CHECK(c);
        *bytes = (size_t)nr * row_bytes;
        return 0;
    }, sink);
}
}  // extern "C++"

int pansim_export_core_csv(pansim_ctx *c, uint32_t row_begin, uint32_t row_end, char *out)
{
    if (!c || !out) return PANSIM_ERR_INVALID;
    char *dst = out;
    return export_core_csv_stream(c, row_begin, row_end, [&](const char *p, size_t n) { memcpy(dst, p, n); dst += n; return 0; });
}

// _core_genome.csv of population.rs:865-882 written by the library itself: the pinned chunks go
// straight to the file, no second host copy. bytes_out (may be NULL) = bytes written.
int pansim_write_core_csv(pansim_ctx *c, const char *path, uint64_t *bytes_out)
{
    if (!c || !path) return PANSIM_ERR_INVALID;
    FILE *f = fopen(path, "wb");
    if (!f) FAIL(c, PANSIM_ERR_INVALID, "cannot create %s", path);
    uint64_t total = 0;
    const int rc = export_core_csv_stream(c, 0, c->N, [&](const char *p, size_t n) { total += n; return fwrite(p, 1, n, f) == n ? 0 : 1; });
    const int rc2 = fclose(f);
    if (bytes_out) *bytes_out = total;
    if (rc) return rc;
    if (rc2) FAIL(c, PANSIM_ERR_INVALID, "closing %s failed", path);
    return 0;
}

int pansim_download_acc(pansim_ctx *c, uint8_t *out)
{
    if (!c || (!out && c->G)) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->G == 0) return 0;
    if (int rc = ensure_stage(c, (size_t)c->N * c->G)) return rc;
    unpack_acc_kernel<<<div_up64((uint64_t)c->N * c->G, 256), 256, 0, c->stream>>>(c->acc[c->acc_cur], c->acc_stride_words, c->G, c->N, c->d_stage);
    LAUNCH_CHECK(c);
    CU(c, cudaMemcpyAsync(out, c->d_stage, (size_t)c->N * c->G, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int pansim_set_selection(pansim_ctx *c, const double *s)
{
    if (!c || (!s && c->G)) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->G == 0) return 0;
    if (int rc = join_fitness(c)) return rc;
    std::vector<double> lw(c->G);
    bool neutral = true;
    for (uint32_t j = 0; j < c->G; j++) {
        lw[j] = std::log(1.0 + s[j] * 1.0);                                   // population.rs:306 with x = 1
        if (!(lw[j] == 0.0) || std::signbit(lw[j])) neutral = false;
    }
    c->neutral = neutral;
    std::vector<uint32_t> lethal(c->acc_words ? c->acc_words : 1, 0u);
    for (uint32_t j = 0; j < c->G; j++)
        if (std::isinf(lw[j]) && lw[j] < 0) lethal[j >> 5] |= 1u << (j & 31);
    CU(c, cudaMemcpyAsync(c->d_lethal, lethal.data(), lethal.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(c->d_lw, lw.data(), (size_t)c->G * 8, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    c->fitness_valid = false;
    return 0;
}

// ---- operators ------------------------------------------------------------
int pansim_average_distance(pansim_ctx *c, double *out)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    c->pdl_now = true;
    timing_begin(c);
    {
        ScopedSpan s(c, TG_SELECT);
        if (int rc = launch_competition(c)) return rc;
    }
    timing_end(c);
    if (out) CU(c, cudaMemcpyAsync(c->h_avg, c->d_avgdist, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (out) memcpy(out, c->h_avg, (size_t)c->N * 8);
    return 0;
}

int pansim_sample_indices(pansim_ctx *c, uint32_t gen, const double *avg, uint32_t *parents_out)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    c->pdl_now = true;
    if (int rc = next_parents_buffer(c)) return rc;
    bool use_avg = false;
    if (avg) {
        memcpy(c->h_avg, avg, (size_t)c->N * 8);      // pinned staging: the copy is a plain DMA (the previous use of h_avg was synchronised)
        CU(c, cudaMemcpyAsync(c->d_avgdist, c->h_avg, (size_t)c->N * 8, cudaMemcpyHostToDevice, c->stream));
        use_avg = true;
    } else if (c->cfg.competition_strength > 0.0) {
        if (!c->avgdist_valid) FAIL(c, PANSIM_ERR_STATE, "competition_strength > 0: call pansim_average_distance first or pass avg_pairwise_dists");
        use_avg = true;
    }
    timing_begin(c);
    {
        ScopedSpan s(c, TG_SELECT);
        if (int rc = launch_select(c, gen, use_avg)) return rc;
    }
    timing_end(c);
    // one read-back, one synchronisation: the parents and the kernel's status word behind them
    CU(c, cudaMemcpyAsync(c->h_parents, c->d_parents, ((size_t)c->N + 1) * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (parents_out) memcpy(parents_out, c->h_parents, (size_t)c->N * 4);
    if (c->h_parents[c->N]) {
        cudaMemsetAsync(c->d_err, 0, sizeof(int), c->stream);
        FAIL(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
    }
    return 0;
}

// main.rs:435-443 as ONE call: average_distance (if competition_strength > 0) + sample_indices, both
// vectors read back behind a single synchronisation.
int pansim_select_parents(pansim_ctx *c, uint32_t gen, double *avg_out, uint32_t *parents_out)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    c->pdl_now = true;
    if (int rc = next_parents_buffer(c)) return rc;
    timing_begin(c);
    const bool use_avg = c->cfg.competition_strength > 0.0;          // main.rs:438-440
    {
        ScopedSpan s(c, TG_SELECT);
        if (use_avg)
            if (int rc = launch_competition(c)) return rc;
        if (int rc = launch_select(c, gen, use_avg)) return rc;
    }
    timing_end(c);
    if (avg_out && use_avg) CU(c, cudaMemcpyAsync(c->h_avg, c->d_avgdist, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(c->h_parents, c->d_parents, ((size_t)c->N + 1) * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (avg_out) {
        if (use_avg) memcpy(avg_out, c->h_avg, (size_t)c->N * 8);
        else for (uint32_t i = 0; i < c->N; i++) avg_out[i] = 1.0;    // main.rs:435
    }
    if (parents_out) memcpy(parents_out, c->h_parents, (size_t)c->N * 4);
    if (c->h_parents[c->N]) {
        cudaMemsetAsync(c->d_err, 0, sizeof(int), c->stream);
        FAIL(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
    }
    return 0;
}

int pansim_get_weights(pansim_ctx *c, double *weights, int32_t *num_genes, double *logfit)
{
    if (!c) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = join_fitness(c)) return rc;
    if (weights) CU(c, cudaMemcpyAsync(weights, c->d_weights, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    if (num_genes) CU(c, cudaMemcpyAsync(num_genes, c->d_num_genes, (size_t)c->N * 4, cudaMemcpyDeviceToHost, c->stream));
    if (logfit) CU(c, cudaMemcpyAsync(logfit, c->d_logfit, (size_t)c->N * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int pansim_get_parents(pansim_ctx *c, uint32_t *out)
{
    if (!c || !out) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    CU(c, cudaMemcpyAsync(out, c->d_parents, (size_t)c->N * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// The caller's vector is copied into the context's own pinned staging buffer of the current
// parents slot, so it is consumed when this returns whatever kind of host memory it lives in
// (a pageable source would make cudaMemcpyAsync host-synchronous, a pinned one would not).
static int upload_parents(pansim_ctx *c, const uint32_t *parents)
{
    const int i = c->parents_idx;
    if (c->h2d_valid[i]) CU(c, cudaEventSynchronize(c->ev_h2d[i]));      // the upload of three steps ago: long done
    uint32_t *stage = c->h_parents_up[i];
    uint32_t bad = 0xFFFFFFFFu;
    for (uint32_t k = 0; k < c->N; k++) {
        const uint32_t v = parents[k];
        stage[k] = v;
        if (v >= c->N && bad == 0xFFFFFFFFu) bad = k;
    }
    if (bad != 0xFFFFFFFFu) FAIL(c, PANSIM_ERR_INVALID, "parents[%u] = %u out of range", bad, parents[bad]);
    CU(c, cudaMemcpyAsync(c->d_parents, stage, (size_t)c->N * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaEventRecord(c->ev_h2d[i], c->stream));
    c->h2d_valid[i] = true;
    return 0;
}

int pansim_step_with_parents(pansim_ctx *c, uint32_t gen, const uint32_t *parents)
{
    if (!c || !parents) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    c->pdl_now = true;
    if (int rc = next_parents_buffer(c)) return rc;
    if (int rc = upload_parents(c, parents)) return rc;
    if (c->dump_enabled) CU(c, cudaMemsetAsync(c->d_dump_counters, 0, 2 * sizeof(uint32_t), c->stream));
    timing_begin(c);
    if (int rc = launch_population_steps(c, gen)) return rc;
    timing_end(c);
    c->avgdist_valid = false;
    // Returns with the step enqueued (the parents vector has been consumed: it was copied into the
    // context's pinned staging buffer). The core kernel keeps running beside the next
    // generation's selection chain; every call that reads or writes the core state joins it first.
    return 0;
}

int pansim_step(pansim_ctx *c, uint32_t gen) { return pansim_run_generations(c, gen, 1); }

#define PANSIM_WEIGHTS_MSG "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)"

// enqueue n generations (asynchronous); the caller synchronises and inspects the device flags.
// The selection chain of every generation is ONE graph launch (chain_graph_step), so the host issues
// about ten calls per generation instead of twenty-five: with eight ranks on one host that enqueue path,
// not the GPUs, was what limited the step.
static int run_generations_enqueue(pansim_ctx *c, uint32_t gen0, uint32_t n)
{
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->dump_enabled) CU(c, cudaMemsetAsync(c->d_dump_counters, 0, 2 * sizeof(uint32_t), c->stream));
    c->pdl_now = false;
    c->ps = c->stream;
    timing_begin(c);
    c->chain_graph_now = c->use_graph && !c->dump_enabled && !c->fine_timing && n >= 8;
    int rc = 0;
    for (uint32_t g = 0; g < n && !rc; g++) rc = step_device(c, gen0 + g);
    c->chain_graph_now = false;
    if (rc) return rc;
    if (int rc2 = join_core_stream(c)) return rc2;
    timing_end(c);
    return 0;
}

int pansim_run_generations(pansim_ctx *c, uint32_t gen0, uint32_t n)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = run_generations_enqueue(c, gen0, n)) return rc;
    return check_device_flag(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG);
}

int pansim_next_generation(pansim_ctx *c, const uint32_t *parents)
{
    if (!c || !parents) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = next_parents_buffer(c)) return rc;
    if (int rc = upload_parents(c, parents)) return rc;
    if (c->gen_cap) {
        CU(c, cudaEventRecord(c->ev_parents[c->parents_idx], c->stream));
        if (int rc = genealogy_record(c)) return rc;
    }
    timing_begin(c);
    if (int rc = join_fitness(c)) return rc;
    if (c->G) {
        const uint64_t total = (uint64_t)c->N * c->acc_stride_words;
        acc_gather_kernel<<<div_up64(total, 256), 256, 0, c->stream>>>(c->acc[c->acc_cur], c->acc[c->acc_cur ^ 1], c->d_parents, c->N, c->acc_stride_words);
        LAUNCH_CHECK(c);
        c->acc_cur ^= 1;
        c->fitness_valid = false;
    }
    if (int rc = launch_core_step(c, 0, false, c->stream)) return rc;
    timing_end(c);
    c->avgdist_valid = false;
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int pansim_step_replay(pansim_ctx *c, const pansim_events *ev)
{
    if (!c || !ev || !ev->parents) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    const size_t nm = ev->n_core_mut, nh = ev->n_hr, nf = ev->n_acc_flip, ng = ev->n_hgt;
    if (nm + nh >= 0xFFFFFFFEull) FAIL(c, PANSIM_ERR_INVALID, "too many core events for one replay step");
    for (size_t k = 0; k < nm; k++)
        if (ev->core_mut_row[k] >= c->N || ev->core_mut_site[k] >= c->L) FAIL(c, PANSIM_ERR_INVALID, "core mutation event %zu out of range", k);
    for (size_t k = 0; k < nh; k++)
        if (ev->hr_recipient[k] >= c->N || ev->hr_locus[k] >= c->L) FAIL(c, PANSIM_ERR_INVALID, "HR event %zu out of range", k);
    for (size_t k = 0; k < nf; k++)
        if (ev->acc_flip_row[k] >= c->N || ev->acc_flip_gene[k] >= c->G) FAIL(c, PANSIM_ERR_INVALID, "flip event %zu out of range", k);
    for (size_t k = 0; k < ng; k++)
        if (ev->hgt_recipient[k] >= c->N || ev->hgt_gene[k] >= c->G) FAIL(c, PANSIM_ERR_INVALID, "HGT event %zu out of range", k);

    // main.rs:445-447
    if (int rc = pansim_next_generation(c, ev->parents)) return rc;

    // stage all event arrays in one device buffer
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t need = al(nm * 4) * 2 + al(nm) + al(nh * 4) * 2 + al(nh) + al(nf * 4) * 2 + al(ng * 4) * 2 + 256;
    if (need > c->replay_cap) {
        if (c->d_replay) cudaFree(c->d_replay);
        c->d_replay = nullptr; c->replay_cap = 0;
        if (cudaMalloc(&c->d_replay, need) != cudaSuccess) FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc(%zu) for replay events failed", need);
        c->replay_cap = need;
    }
    uint8_t *base = (uint8_t *)c->d_replay;
    size_t off = 0;
    auto put = [&](const void *src, size_t bytes) -> void * {
        void *d = base + off;
        if (bytes) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, c->stream);
        off += al(bytes);
        return d;
    };
    CoreWriteList mut, hr;
    mut.row = (uint32_t *)put(ev->core_mut_row, nm * 4);
    mut.site = (uint32_t *)put(ev->core_mut_site, nm * 4);
    mut.value = (uint8_t *)put(ev->core_mut_allele, nm);
    mut.n = nm; mut.index_base = 0;
    hr.row = (uint32_t *)put(ev->hr_recipient, nh * 4);
    hr.site = (uint32_t *)put(ev->hr_locus, nh * 4);
    hr.value = (uint8_t *)put(ev->hr_value, nh);
    hr.n = nh; hr.index_base = (uint32_t)nm;
    uint32_t *f_row = (uint32_t *)put(ev->acc_flip_row, nf * 4);
    uint32_t *f_gene = (uint32_t *)put(ev->acc_flip_gene, nf * 4);
    uint32_t *g_row = (uint32_t *)put(ev->hgt_recipient, ng * 4);
    uint32_t *g_gene = (uint32_t *)put(ev->hgt_gene, ng * 4);
    CU(c, cudaGetLastError());

    // core: mutations then HR as one ordered write list (population.rs:537, :745)
    if (nm + nh > 0 && c->Ll) {
        size_t cap = 1024;
        while (cap < 2 * (nm + nh)) cap <<= 1;
        if (cap > c->hash_cap) {
            if (c->d_hkeys) cudaFree(c->d_hkeys);
            if (c->d_hvals) cudaFree(c->d_hvals);
            c->d_hkeys = nullptr; c->d_hvals = nullptr; c->hash_cap = 0;
            if (cudaMalloc(&c->d_hkeys, cap * 8) != cudaSuccess || cudaMalloc(&c->d_hvals, cap * 4) != cudaSuccess)
                FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for the replay hash table (%zu slots) failed", cap);
            c->hash_cap = cap;
        }
        cap = c->hash_cap;
        CU(c, cudaMemsetAsync(c->d_hkeys, 0, cap * 8, c->stream));
        CU(c, cudaMemsetAsync(c->d_hvals, 0, cap * 4, c->stream));
        uint8_t *state = c->core[c->core_cur];
        c->core_version++;
        for (CoreWriteList *l : {&mut, &hr}) {
            if (!l->n) continue;
            replay_insert_kernel<<<div_up64(l->n, 256), 256, 0, c->stream>>>(*l, c->site_begin, c->site_end, c->Ll, c->d_hkeys, c->d_hvals, cap - 1);
            LAUNCH_CHECK(c);
        }
        for (CoreWriteList *l : {&mut, &hr}) {
            if (!l->n) continue;
            replay_apply_kernel<<<div_up64(l->n, 256), 256, 0, c->stream>>>(*l, c->site_begin, c->site_end, c->Ll, c->d_hkeys, c->d_hvals, cap - 1, state, c->core_stride, c->d_err);
            LAUNCH_CHECK(c);
        }
    }
    // accessory: flips (population.rs:504-508) then HGT sets (:745 with value 1)
    c->fitness_valid = false;
    if (nf) {
        acc_apply_flips_kernel<<<div_up64(nf, 256), 256, 0, c->stream>>>(c->acc[c->acc_cur], f_row, f_gene, nf, c->acc_stride_words);
        LAUNCH_CHECK(c);
    }
    if (ng) {
        acc_apply_sets_kernel<<<div_up64(ng, 256), 256, 0, c->stream>>>(c->acc[c->acc_cur], g_row, g_gene, ng, c->acc_stride_words);
        LAUNCH_CHECK(c);
    }
    return check_device_flag(c, PANSIM_ERR_INVALID, "replay event carries an allele that is not one-hot {1,2,4,8}");
}

// ---- distances ------------------------------------------------------------
static int ensure_pairs(pansim_ctx *c, size_t n)
{
    if (n <= c->pair_cap) return 0;
    for (uint32_t **p : {&c->d_r1, &c->d_r2, &c->d_cd, &c->d_in, &c->d_un}) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    c->pair_cap = 0;
    c->pairs_on_device = false;
    for (uint32_t **p : {&c->d_r1, &c->d_r2, &c->d_cd, &c->d_in, &c->d_un})
        if (cudaMalloc(p, n * 4) != cudaSuccess) FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for %zu pairs failed", n);
    c->pair_cap = n;
    return 0;
}

// Plane form of the current core buffer (distance.cuh) and its TMA descriptor; the pre-pass runs only
// when the rows have changed since the last one.
static int ensure_planes(pansim_ctx *c)
{
    const size_t core_bytes = (size_t)c->N * c->core_stride;
    if (!c->d_planes) {
        if (cudaMalloc(&c->d_planes, core_bytes) != cudaSuccess) FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (bit planes for the distance pass) failed", core_bytes);
        CU(c, cudaMalloc(&c->d_work_counter, sizeof(uint32_t)));
        c->planes_version = 0;
        // 2-D tensor map over the plane rows: x = 32-bit words of a row, y = rows; box = 512 bytes x 64 rows
        c->planes_tmap_ok = false;
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn &&
            qres == cudaDriverEntryPointSuccess && c->N >= 1 && c->core_stride / 4 < (1ull << 32)) {
            typedef CUresult (*encode_t)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                         const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                         CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
            const cuuint64_t gdim[2] = {c->core_stride / 4, c->N};
            const cuuint64_t gstride[1] = {c->core_stride};
            const cuuint32_t box[2] = {T2_CHUNK_BYTES / 4, T2_BLOCK_ROWS};
            const cuuint32_t estr[2] = {1, 1};
            const CUresult r = reinterpret_cast<encode_t>(fn)(&c->planes_tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, c->d_planes, gdim, gstride, box,
                                                             estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            c->planes_tmap_ok = r == CUDA_SUCCESS;
        }
        cudaGetLastError();
        CU(c, cudaFuncSetAttribute(pair_tile2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile2_smem_bytes()));
    }
    if (c->planes_version != c->core_version) {
        const uint64_t n_vec4 = core_bytes / 16;
        const uint32_t grid = (uint32_t)std::min<uint64_t>((n_vec4 + 255) / 256, (uint64_t)c->sm_count * 32);
        core_planes_kernel<<<grid, 256, 0, c->ps>>>(reinterpret_cast<const uint4 *>(c->core[c->core_cur]),
                                                        reinterpret_cast<uint4 *>(c->d_planes), n_vec4);
        LAUNCH_CHECK(c);
        c->planes_version = c->core_version;
    }
    return 0;
}

// Build (or reuse) the plan for this pair list. Pairs are bucketed by the pair of 64-row blocks their
// endpoints fall in; a bucket with enough pairs is cut into batches for the TMA tile kernel (every staged
// row then serves several pairs), the rest goes to the row-stationary group kernel.
static int ensure_pair_plan(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P)
{
    if (c->plan_r1.size() == P && (c->plan_groups || c->plan_batches) &&
        memcmp(c->plan_r1.data(), r1, P * 4) == 0 && memcmp(c->plan_r2.data(), r2, P * 4) == 0)
        return 0;
    const uint32_t NB = (c->N + T2_BLOCK_ROWS - 1) / T2_BLOCK_ROWS;
    const size_t n_keys = (size_t)NB * NB;
    std::vector<uint32_t> key(P);
    std::vector<uint32_t> kcount;
    const bool use_tiles = c->use_tiles2 && n_keys <= (1u << 24);
    if (use_tiles) {
        kcount.assign(n_keys + 1, 0);
        for (size_t k = 0; k < P; k++) {
            const uint32_t bi = r1[k] / T2_BLOCK_ROWS, bj = r2[k] / T2_BLOCK_ROWS;
            key[k] = std::min(bi, bj) * NB + std::max(bi, bj);
            kcount[key[k] + 1]++;
        }
    }
    // a tile stages 64 or 128 rows per chunk: below this many pairs the rows are barely used and the
    // row-stationary kernel (9 row reads per 8 pairs) moves less
    const uint32_t dense_min = 96;
    std::vector<TileBatch> batches;
    std::vector<uint16_t> tslots;
    std::vector<uint32_t> torig;
    std::vector<uint8_t> is_dense(P, 0);
    if (use_tiles) {
        std::vector<uint32_t> kstart(kcount);
        for (size_t i = 0; i < n_keys; i++) kstart[i + 1] += kstart[i];
        std::vector<uint32_t> order(P), cur(kstart.begin(), kstart.end() - 1);
        for (size_t k = 0; k < P; k++) order[cur[key[k]]++] = (uint32_t)k;
        const uint32_t cols = (uint32_t)(c->core_stride / T2_CHUNK_BYTES);
        size_t n_dense_batches = 0;
        for (size_t kk = 0; kk < n_keys; kk++) {
            const uint32_t cnt = kstart[kk + 1] - kstart[kk];
            if (cnt >= dense_min) n_dense_batches += (cnt + T2_BATCH - 1) / T2_BATCH;
        }
        // Column ranges. (i) enough work items for ~8 per SM (the persistent CTAs balance themselves); (ii) the
        // rows of one range, N x range bytes, are what all concurrently running items read: at most ~40 MB so
        // that the range stays in L2 while its items run and DRAM sees every row once per pass (measured at
        // cfg1: 4 ranges of 75 MB -> 580 MB of DRAM reads, 8 ranges of 37 MB -> 306 MB = 1.02 x the rows; finer
        // ranges only add per-item prologues: 16 -> 1.56 ms, 32 -> 1.77 ms against 1.49 ms); (iii) ranges of at
        // least 16 chunks.
        uint32_t col_split = 1;
        while (n_dense_batches && n_dense_batches * col_split < (size_t)c->sm_count * 8 && cols / (col_split * 2) >= 32) col_split *= 2;
        const uint64_t slab_target = 40ull << 20;
        const uint32_t by_l2 = (uint32_t)std::min<uint64_t>(cols, ((uint64_t)c->N * c->core_stride + slab_target - 1) / slab_target);
        col_split = std::max(col_split, by_l2);
        if (cols / col_split < 16) col_split = std::max(1u, cols / 16);
        if (const char *e = getenv("PANSIM_TILE_COLSPLIT")) col_split = (uint32_t)std::max(1, std::min((int)cols, atoi(e)));
        struct Raw { uint32_t ba, bb, first, count; };
        std::vector<Raw> raw;
        for (size_t kk = 0; kk < n_keys; kk++) {
            const uint32_t cnt = kstart[kk + 1] - kstart[kk];
            if (cnt < dense_min) continue;
            const uint32_t ba = (uint32_t)(kk / NB), bb = (uint32_t)(kk % NB);
            // slots of each pair (0..63 block a, 64..127 block b), sorted by first slot: a warp keeps the
            // first row's piece in registers while it repeats. The distance is symmetric, so a pair whose
            // first endpoint lies in the later block is taken as (j, i).
            std::vector<std::pair<uint32_t, uint32_t>> v;      // (slot_a << 8 | slot_b, orig)
            v.reserve(cnt);
            for (uint32_t t = kstart[kk]; t < kstart[kk + 1]; t++) {
                const uint32_t k = order[t];
                is_dense[k] = 1;
                uint32_t i = r1[k], j = r2[k];
                if (i / T2_BLOCK_ROWS != ba) std::swap(i, j);
                const uint32_t sa = i % T2_BLOCK_ROWS, sb = (ba == bb ? 0u : (uint32_t)T2_BLOCK_ROWS) + j % T2_BLOCK_ROWS;
                v.push_back({(sa << 8) | sb, k});
            }
            std::sort(v.begin(), v.end());
            // equal batches (a bucket of 400 pairs becomes 2 x 200, not 384 + 16)
            const uint32_t nb = (cnt + T2_BATCH - 1) / T2_BATCH;
            for (uint32_t b = 0; b < nb; b++) {
                const uint32_t f = (uint32_t)((uint64_t)cnt * b / nb), e = (uint32_t)((uint64_t)cnt * (b + 1) / nb);
                raw.push_back({ba, bb, (uint32_t)tslots.size(), e - f});
                for (uint32_t t = f; t < e; t++) {
                    tslots.push_back((uint16_t)((v[t].first >> 8) | ((v[t].first & 0xFFu) << 8)));   // low byte = slot_a
                    torig.push_back(v[t].second);
                }
            }
        }
        // work items in column-range-major order: the items that run at the same time read the same
        // column range of all rows, so DRAM sees every row about once per pass
        for (uint32_t sp = 0; sp < col_split; sp++)
            for (const Raw &rw : raw) {
                TileBatch b;
                b.block_a = rw.ba; b.block_b = rw.bb; b.first = rw.first; b.count = rw.count;
                b.col_begin = (uint32_t)((uint64_t)cols * sp / col_split);
                b.col_end = (uint32_t)((uint64_t)cols * (sp + 1) / col_split);
                batches.push_back(b);
            }
    }
    // ---- sparse part: row-stationary groups (counting sort by first row) ----
    std::vector<uint32_t> start(c->N + 1, 0);
    for (size_t k = 0; k < P; k++) if (!is_dense[k]) start[r1[k] + 1]++;
    for (uint32_t i = 0; i < c->N; i++) start[i + 1] += start[i];
    const size_t n_sparse = start[c->N];
    std::vector<uint32_t> partner(n_sparse), orig(n_sparse), cursor(start.begin(), start.end() - 1);
    for (size_t k = 0; k < P; k++) {
        if (is_dense[k]) continue;
        const uint32_t pos = cursor[r1[k]]++;
        partner[pos] = r2[k];
        orig[pos] = (uint32_t)k;
    }
    std::vector<PairGroup> groups;
    for (uint32_t i = 0; i < c->N; i++)
        for (uint32_t f = start[i]; f < start[i + 1]; f += PAIR_GROUP)
            groups.push_back(PairGroup{i, f, std::min<uint32_t>(PAIR_GROUP, start[i + 1] - f)});

    auto grow = [&](void **ptr, size_t &cap, size_t need, size_t elem) -> int {
        if (need <= cap) return 0;
        if (*ptr) cudaFree(*ptr);
        *ptr = nullptr; cap = 0;
        if (cudaMalloc(ptr, need * elem) != cudaSuccess) return -1;
        cap = need;
        return 0;
    };
    size_t cap_tp2 = c->plan_cap_tile_pairs, cap_p2 = c->plan_cap_pairs;
    if (grow((void **)&c->d_groups, c->plan_cap_groups, groups.size(), sizeof(PairGroup)) ||
        grow((void **)&c->d_partner, c->plan_cap_pairs, n_sparse, 4) || grow((void **)&c->d_orig, cap_p2, n_sparse, 4) ||
        grow((void **)&c->d_batches, c->plan_cap_batches, batches.size(), sizeof(TileBatch)) ||
        grow((void **)&c->d_tile_slots, c->plan_cap_tile_pairs, tslots.size(), 2) ||
        grow((void **)&c->d_tile_orig, cap_tp2, torig.size(), 4))
        FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for the pair plan failed");
    auto up = [&](void *dst, const void *src, size_t bytes) { if (bytes) cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream); };
    up(c->d_groups, groups.data(), groups.size() * sizeof(PairGroup));
    up(c->d_partner, partner.data(), n_sparse * 4);
    up(c->d_orig, orig.data(), n_sparse * 4);
    up(c->d_batches, batches.data(), batches.size() * sizeof(TileBatch));
    up(c->d_tile_slots, tslots.data(), tslots.size() * 2);
    up(c->d_tile_orig, torig.data(), torig.size() * 4);
    CU(c, cudaStreamSynchronize(c->stream));      // the host vectors go out of scope
    CU(c, cudaGetLastError());
    c->plan_groups = groups.size();
    c->plan_batches = batches.size();
    c->plan_r1.assign(r1, r1 + P);
    c->plan_r2.assign(r2, r2 + P);
    return 0;
}

// core Hamming counts of the planned pairs (c->plan_batches / c->plan_groups) into d_cd[P];
// rows_active = number of distinct rows the plan touches (sizes the L2-resident column chunk)
static int launch_pair_core(pansim_ctx *c, uint32_t *d_cd, size_t P, uint32_t rows_active, bool clear)
{
    if (int rc = ensure_planes(c)) return rc;
    const uint32_t row_vec4 = (uint32_t)(c->core_stride / 16);
    // column chunk sized so that rows x chunk stays L2 resident
    uint64_t chunk_bytes = (48ull << 20) / std::max(1u, rows_active);
    chunk_bytes = (chunk_bytes / 4096) * 4096;
    // Below 32 KB per row the chunks no longer amortise the per-group work, and with that many rows the
    // L2-resident slab is gone anyway: stream long chunks from HBM instead (N = 10 000, L = 5 Mbp, 20 000
    // sampled pairs: 1.8e6 pairs/s with 4 KB chunks, 3.0e6 with 32 KB, 3.1e6 with >= 128 KB).
    if (chunk_bytes < 32768) chunk_bytes = 262144;
    if (chunk_bytes > c->core_stride) chunk_bytes = ((c->core_stride + 4095) / 4096) * 4096;
    uint32_t chunk_vec4 = (uint32_t)(chunk_bytes / 16);
    uint32_t n_chunks = (row_vec4 + chunk_vec4 - 1) / chunk_vec4;
    if (n_chunks > 65535) { n_chunks = 65535; chunk_vec4 = (row_vec4 + n_chunks - 1) / n_chunks; chunk_vec4 = ((chunk_vec4 + 255) / 256) * 256; n_chunks = (row_vec4 + chunk_vec4 - 1) / chunk_vec4; }
    if (clear) CU(c, cudaMemsetAsync(d_cd, 0, P * 4, c->ps));      // both kernels accumulate with integer atomics
    if (c->plan_batches) {
        if (!c->planes_tmap_ok) FAIL(c, PANSIM_ERR_CUDA, "no TMA descriptor for the plane rows (cuTensorMapEncodeTiled unavailable)");
        CU(c, cudaMemsetAsync(c->d_work_counter, 0, sizeof(uint32_t), c->ps));
        const uint32_t grid = (uint32_t)std::min<size_t>(c->plan_batches, (size_t)c->sm_count);
        pair_tile2_kernel<<<grid, T2_THREADS, tile2_smem_bytes(), c->ps>>>(
            c->planes_tmap, c->d_batches, (uint32_t)c->plan_batches, c->d_work_counter, c->d_tile_slots, c->d_tile_orig, d_cd);
        LAUNCH_CHECK(c);
    }
    if (c->plan_groups) {
        const uint32_t gx = (uint32_t)std::min<size_t>(c->plan_groups, 1u << 20);
        pair_planes_grouped_kernel<<<dim3(gx, n_chunks), PAIR_THREADS, 0, c->ps>>>(
            c->d_planes, c->core_stride, chunk_vec4, row_vec4, c->d_groups, (uint32_t)c->plan_groups,
            c->d_partner, c->d_orig, d_cd);
        LAUNCH_CHECK(c);
    }
    return 0;
}

// Validate the pair list, build (or reuse) its plan and put range1/range2 on the device. A list that
// equals the cached one (the pairs are fixed for a whole run, main.rs:413-427) has been validated and
// uploaded before: two memcmp and nothing else.
static int pair_prepare(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P)
{
    if (P > 0x7FFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "more than 2^31 pairs per call");
    if (c->pairs_on_device && c->plan_r1.size() == P && memcmp(c->plan_r1.data(), r1, P * 4) == 0 &&
        memcmp(c->plan_r2.data(), r2, P * 4) == 0)
        return 0;
    for (size_t k = 0; k < P; k++)
        if (r1[k] >= c->N || r2[k] >= c->N) FAIL(c, PANSIM_ERR_INVALID, "pair %zu out of range", k);
    c->pairs_on_device = false;
    if (c->Ll) {
        if (int rc = ensure_pair_plan(c, r1, r2, P)) return rc;
    } else {
        c->plan_r1.assign(r1, r1 + P);
        c->plan_r2.assign(r2, r2 + P);
    }
    CU(c, cudaMemcpyAsync(c->d_r1, c->plan_r1.data(), P * 4, cudaMemcpyHostToDevice, c->stream));   // from the context's copy:
    CU(c, cudaMemcpyAsync(c->d_r2, c->plan_r2.data(), P * 4, cudaMemcpyHostToDevice, c->stream));   // the caller's may go away
    CU(c, cudaStreamSynchronize(c->stream));
    c->pairs_on_device = true;
    return 0;
}

// the kernels of one distance pass over the prepared pairs (asynchronous on c->stream)
static int pair_launch(pansim_ctx *c, size_t P, uint32_t *d_cd, uint32_t *d_in, uint32_t *d_un)
{
    if (d_cd && c->Ll)
        if (int rc = core_materialize(c, c->ps)) return rc;     // recombination events still pending on the rows
    if (d_cd) {
        ScopedSpan s(c, TG_PAIR_CORE, c->ps);
        if (c->Ll == 0) {
            CU(c, cudaMemsetAsync(d_cd, 0, P * 4, c->ps));
        } else {
            if (int rc = launch_pair_core(c, d_cd, P, c->N, true)) return rc;
        }
    }
    if (d_in || d_un) {
        ScopedSpan s(c, TG_PAIR_ACC, c->ps);
        const uint32_t grid = (uint32_t)std::min<size_t>((P + 7) / 8, (size_t)c->sm_count * 16);
        pair_acc_kernel<<<grid ? grid : 1, 256, 0, c->ps>>>(c->acc[c->acc_cur], c->acc_stride_words, c->acc_words, c->d_r1, c->d_r2, (uint32_t)P, d_in, d_un);
        LAUNCH_CHECK(c);
    }
    return 0;
}

static int pair_counts_impl(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P, uint32_t *d_cd,
                            uint32_t *d_in, uint32_t *d_un)
{
    c->ps = c->stream;
    if (int rc = pair_prepare(c, r1, r2, P)) return rc;
    timing_begin(c);
    if (int rc = pair_launch(c, P, d_cd, d_in, d_un)) return rc;
    timing_end(c);
    return 0;
}

int pansim_pair_counts(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P, uint32_t *core_diff,
                       uint32_t *inter, uint32_t *uni)
{
    if (!c || (P && (!r1 || !r2))) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (P == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_pairs(c, P)) return rc;
    if (int rc = pair_counts_impl(c, r1, r2, P, core_diff ? c->d_cd : nullptr, (inter || uni) ? c->d_in : nullptr, (inter || uni) ? c->d_un : nullptr)) return rc;
    if (core_diff)
        if (int rc = comm_allreduce_counts(c, c->d_cd, P)) return rc;
    if (core_diff) CU(c, cudaMemcpyAsync(core_diff, c->d_cd, P * 4, cudaMemcpyDeviceToHost, c->stream));
    if (inter) CU(c, cudaMemcpyAsync(inter, c->d_in, P * 4, cudaMemcpyDeviceToHost, c->stream));
    if (uni) CU(c, cudaMemcpyAsync(uni, c->d_un, P * 4, cudaMemcpyDeviceToHost, c->stream));
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return flags_inspect(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
}

int pansim_pair_counts_device(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P, void *d_cd,
                              void *d_in, void *d_un)
{
    if (!c || (P && (!r1 || !r2))) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (P == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_pairs(c, P)) return rc;
    if (int rc = pair_counts_impl(c, r1, r2, P, (uint32_t *)d_cd, (uint32_t *)d_in, (uint32_t *)d_un)) return rc;
    if (int rc = comm_allreduce_counts(c, (uint32_t *)d_cd, P)) return rc;
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return flags_inspect(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
}

// ---- --print_dist statistics on the device (main.rs:502-519, population.rs:87-94) -------------
static int ensure_stats(pansim_ctx *c, size_t n_gen, size_t P, bool second_counts)
{
    if (!c->stream_stats2[0]) {
        int lo = 0, hi = 0;
        CU(c, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(c, cudaStreamCreateWithPriority(&c->stream_pairs, cudaStreamNonBlocking, lo));
        CU(c, cudaEventCreateWithFlags(&c->ev_acc_done, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&c->ev_mat, cudaEventDisableTiming));
        for (int i = 0; i < 2; i++) {
            CU(c, cudaStreamCreateWithPriority(&c->stream_stats2[i], cudaStreamNonBlocking, hi));
            CU(c, cudaEventCreateWithFlags(&c->ev_pairs[i], cudaEventDisableTiming));
            CU(c, cudaEventCreateWithFlags(&c->ev_stats[i], cudaEventDisableTiming));
        }
    }
    if (n_gen > c->stats_cap) {
        if (c->d_stats) cudaFree(c->d_stats);
        if (c->h_stats) cudaFreeHost(c->h_stats);
        c->d_stats = nullptr; c->h_stats = nullptr; c->stats_cap = 0;
        CU(c, cudaMalloc(&c->d_stats, n_gen * 4 * sizeof(double)));
        CU(c, cudaMallocHost(&c->h_stats, n_gen * 4 * sizeof(double)));
        c->stats_cap = n_gen;
    }
    if (second_counts && P > c->cnt2_cap) {
        for (auto &q : c->d_cnt2) { if (q) cudaFree(q); q = nullptr; }
        c->cnt2_cap = 0;
        for (auto &q : c->d_cnt2)
            if (cudaMalloc(&q, P * 4) != cudaSuccess) FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for %zu pairs failed", P);
        c->cnt2_cap = P;
    }
    return 0;
}

// statistics kernel of one pass on the statistics stream, behind the pass on c->stream
static int launch_pair_stats(pansim_ctx *c, int slot, size_t P, const uint32_t *d_cd, const uint32_t *d_in, const uint32_t *d_un,
                             double *d_out)
{
    CU(c, cudaEventRecord(c->ev_pairs[slot], c->ps));
    c->ev_pairs_valid[slot] = true;
    cudaStream_t st = c->stream_stats2[slot];
    CU(c, cudaStreamWaitEvent(st, c->ev_pairs[slot], 0));
    PairStatsArgs a;
    a.core_diff = d_cd; a.inter = d_in; a.uni = d_un;
    a.n_pairs = (uint32_t)P;
    a.core_size = (double)c->L;
    a.core_genes = (double)c->cfg.core_genes;
    a.out = d_out;
    pair_stats_kernel<<<1, STATS_THREADS, 0, st>>>(a);
    LAUNCH_CHECK(c);
    CU(c, cudaEventRecord(c->ev_stats[slot], st));
    c->ev_stats_valid[slot] = true;
    return 0;
}

static int require_whole_alignment(pansim_ctx *c, const char *what)
{
    if (c->Ll != c->L && !c->comm) FAIL(c, PANSIM_ERR_STATE, "%s on a column shard needs a communicator (pansim_comm_init_rank): core counts are partial", what);
    return 0;
}

// One generation of the --print_dist batch on one context. The generation step goes to its usual
// streams; the distance pass of this generation goes to stream_pairs, so it runs beside the selection
// chain and the core step of the NEXT generation instead of in front of them:
//   pass(g) starts after core step g and accessory step g; it first materialises the recombination
//   events of g in the current core buffer (core step g+1 waits for that and applies nothing itself);
//   accessory step g+2 recycles the buffer pass(g) reads, so generation g+2 waits for pass(g) -- which
//   is also the back-pressure that keeps the steps at most two generations ahead of the passes;
//   the count vectors alternate between two sets (the statistics kernel of g reads set g & 1).
static int stats_generation(pansim_ctx *c, uint32_t gen, int slot, size_t P, bool want_acc, uint32_t **cd_out, uint32_t **in_out,
                            uint32_t **un_out)
{
    c->pdl_now = false;
    c->ps = c->stream;
    if (c->ev_pairs_valid[slot]) CU(c, cudaStreamWaitEvent(c->stream, c->ev_pairs[slot], 0));          // pass(g-2) done
    c->chain_graph_now = c->use_graph && !c->dump_enabled && !c->fine_timing;
    const int rc_step = step_device(c, gen);
    c->chain_graph_now = false;
    if (rc_step) return rc_step;
    cudaStream_t sp = c->stream_pairs;
    CU(c, cudaEventRecord(c->ev_acc_done, c->stream));
    CU(c, cudaStreamWaitEvent(sp, c->ev_acc_done, 0));
    if (c->ev_stats_valid[slot]) CU(c, cudaStreamWaitEvent(sp, c->ev_stats[slot], 0));               // statistics(g-2) have read this set
    c->ps = sp;
    uint32_t *cd = slot ? c->d_cnt2[0] : c->d_cd, *in = slot ? c->d_cnt2[1] : c->d_in, *un = slot ? c->d_cnt2[2] : c->d_un;
    if (c->Ll) {
        if (int rc = core_materialize(c, sp)) { c->ps = c->stream; return rc; }
        CU(c, cudaEventRecord(c->ev_mat, sp));
        CU(c, cudaStreamWaitEvent(c->stream_core, c->ev_mat, 0));       // the next core step reads the materialised rows
    }
    const int rc = P ? pair_launch(c, P, cd, want_acc ? in : nullptr, want_acc ? un : nullptr) : 0;   // P = 0: diversity batch without pairs
    if (rc) { c->ps = c->stream; return rc; }
    *cd_out = cd; *in_out = in; *un_out = un;
    return 0;        // c->ps stays on stream_pairs: the caller's all-reduce and statistics launch follow the pass
}

// after the last generation: c->stream joins the core stream, the passes and the statistics
static int stats_batch_end(pansim_ctx *c)
{
    c->ps = c->stream;
    if (int rc = join_core_stream(c)) return rc;
    for (int i = 0; i < 2; i++) {
        if (c->ev_pairs_valid[i]) CU(c, cudaStreamWaitEvent(c->stream, c->ev_pairs[i], 0));
        if (c->ev_stats_valid[i]) CU(c, cudaStreamWaitEvent(c->stream, c->ev_stats[i], 0));
    }
    return 0;
}

int pansim_pair_stats(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P, double *out)
{
    if (!c || !out || !P || !r1 || !r2) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (int rc = require_whole_alignment(c, "pansim_pair_stats")) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_pairs(c, P)) return rc;
    if (int rc = ensure_stats(c, 1, P, false)) return rc;
    if (int rc = pair_counts_impl(c, r1, r2, P, c->d_cd, c->d_in, c->d_un)) return rc;
    if (int rc = comm_allreduce_counts(c, c->d_cd, P)) return rc;
    if (int rc = launch_pair_stats(c, 0, P, c->d_cd, c->d_in, c->d_un, c->d_stats)) return rc;
    CU(c, cudaMemcpyAsync(c->h_stats, c->d_stats, 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream_stats2[0]));
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaStreamSynchronize(c->stream_stats2[0]));
    memcpy(out, c->h_stats, 4 * sizeof(double));
    return flags_inspect(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
}

// n generations, each followed by the distance pass and its statistics, without returning to the
// host: the loop main.rs:429-519 runs with --print_dist. 32 bytes per generation leave the device.
int pansim_run_generations_stats(pansim_ctx *c, uint32_t gen0, uint32_t n, const uint32_t *r1, const uint32_t *r2, size_t P,
                                 double *stats_out)
{
    if (!c || !stats_out || !P || !r1 || !r2) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (int rc = require_whole_alignment(c, "pansim_run_generations_stats")) return rc;
    if (n == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_pairs(c, P)) return rc;
    if (int rc = ensure_stats(c, n, P, true)) return rc;
    if (int rc = pair_prepare(c, r1, r2, P)) return rc;
    if (c->dump_enabled) CU(c, cudaMemsetAsync(c->d_dump_counters, 0, 2 * sizeof(uint32_t), c->stream));
    timing_begin(c);
    for (uint32_t g = 0; g < n; g++) {
        uint32_t *cd = nullptr, *in = nullptr, *un = nullptr;
        if (int rc = stats_generation(c, gen0 + g, (int)(g & 1u), P, true, &cd, &in, &un)) return rc;
        if (int rc = comm_allreduce_counts(c, cd, P)) return rc;
        if (int rc = launch_pair_stats(c, (int)(g & 1u), P, cd, in, un, c->d_stats + (size_t)g * 4)) return rc;
    }
    if (int rc = stats_batch_end(c)) return rc;
    timing_end(c);
    CU(c, cudaMemcpyAsync(c->h_stats, c->d_stats, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (int rc = check_device_flag(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)")) return rc;
    memcpy(stats_out, c->h_stats, (size_t)n * 4 * sizeof(double));
    return 0;
}

// Exact all-pairs extension: every pair (i, j), i in [row_begin, row_end), i < j < N, in (i, j)
// order; pair list and plan generated on the device (distance.cuh).
static int pair_counts_rows_impl(pansim_ctx *c, uint32_t row_begin, uint32_t row_end, uint32_t *d_cd, uint32_t *d_in,
                                 uint32_t *d_un, size_t *n_out)
{
    if (row_begin > row_end || row_end > c->N) FAIL(c, PANSIM_ERR_INVALID, "row block [%u, %u) out of range", row_begin, row_end);
    c->ps = c->stream;
    const uint32_t nr = row_end - row_begin;
    std::vector<uint32_t> off(nr + 1, 0);
    uint64_t P = 0;
    for (uint32_t r = 0; r < nr; r++) {
        off[r] = (uint32_t)P;
        P += (uint64_t)c->N - 1u - (row_begin + r);
        if (P > 0x7FFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "more than 2^31 pairs in rows [%u, %u): use smaller row blocks", row_begin, row_end);
    }
    off[nr] = (uint32_t)P;
    *n_out = (size_t)P;
    if (P == 0) return 0;
    // Partner rows are walked in column blocks of the pair matrix: a launch touches the nr rows of the
    // block and at most jb partner rows, so a column chunk of those rows (>= 32 KB each) stays in L2
    // however large N is.
    const uint32_t jb = std::max(256u, 1536u > nr ? 1536u - nr : 0u);
    const uint32_t j_first = row_begin + 1u;
    const uint32_t n_jblocks = (c->N - j_first + jb - 1) / jb;
    std::vector<uint32_t> goff((size_t)n_jblocks * (nr + 1), 0);
    std::vector<uint32_t> n_groups(n_jblocks, 0);
    size_t max_groups = 0;
    for (uint32_t b = 0; b < n_jblocks; b++) {
        const uint32_t jb0 = j_first + b * jb, jb1 = std::min(c->N, jb0 + jb);
        uint32_t *go = goff.data() + (size_t)b * (nr + 1);
        uint64_t G = 0;
        for (uint32_t r = 0; r < nr; r++) {
            go[r] = (uint32_t)G;
            const uint32_t j_lo = std::max(row_begin + r + 1u, jb0);
            if (j_lo < jb1) G += (jb1 - j_lo + PAIR_GROUP - 1) / PAIR_GROUP;
        }
        go[nr] = (uint32_t)G;
        n_groups[b] = (uint32_t)G;
        max_groups = std::max(max_groups, (size_t)G);
    }
    if (int rc = ensure_pairs(c, (size_t)P)) return rc;
    auto grow = [&](void **ptr, size_t &cap, size_t need, size_t elem) -> int {
        if (need <= cap) return 0;
        if (*ptr) cudaFree(*ptr);
        *ptr = nullptr; cap = 0;
        if (cudaMalloc(ptr, need * elem) != cudaSuccess) return -1;
        cap = need;
        return 0;
    };
    size_t cap_p2 = c->plan_cap_pairs;
    if (grow((void **)&c->d_groups, c->plan_cap_groups, max_groups, sizeof(PairGroup)) ||
        grow((void **)&c->d_partner, c->plan_cap_pairs, (size_t)P, 4) || grow((void **)&c->d_orig, cap_p2, (size_t)P, 4))
        FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for the all-pairs plan failed");
    if (int rc = ensure_stage(c, ((size_t)(nr + 1) + goff.size()) * 4)) return rc;
    uint32_t *d_off = reinterpret_cast<uint32_t *>(c->d_stage), *d_goff = d_off + (nr + 1);
    CU(c, cudaMemcpyAsync(d_off, off.data(), (size_t)(nr + 1) * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(d_goff, goff.data(), goff.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));                 // the host vectors go out of scope
    c->plan_r1.clear(); c->plan_r2.clear();                  // the cached sampled-pair plan is gone
    c->pairs_on_device = false;
    c->plan_batches = 0;
    timing_begin(c);
    if (c->Ll)
        if (int rc = core_materialize(c, c->stream)) return rc;
    rows_pairs_kernel<<<div_up64(P, 256), 256, 0, c->stream>>>(d_off, nr, row_begin, (uint32_t)P, c->d_r1, c->d_r2, c->d_partner, c->d_orig);
    LAUNCH_CHECK(c);
    if (d_cd) {
        ScopedSpan s(c, TG_PAIR_CORE);
        CU(c, cudaMemsetAsync(d_cd, 0, (size_t)P * 4, c->stream));
        for (uint32_t b = 0; b < n_jblocks && c->Ll; b++) {
            if (!n_groups[b]) continue;
            const uint32_t jb0 = j_first + b * jb, jb1 = std::min(c->N, jb0 + jb);
            rows_groups_kernel<<<div_up64(n_groups[b], 256), 256, 0, c->stream>>>(d_off, d_goff + (size_t)b * (nr + 1), nr, row_begin,
                                                                                  jb0, jb1, n_groups[b], c->d_groups);
            LAUNCH_CHECK(c);
            c->plan_groups = n_groups[b];
            if (int rc = launch_pair_core(c, d_cd, (size_t)P, nr + (jb1 - jb0), false)) return rc;
        }
    }
    c->plan_groups = 0;                                      // the device plan is only valid for this call
    if (d_in || d_un) {
        ScopedSpan s(c, TG_PAIR_ACC);
        const uint32_t grid = (uint32_t)std::min<size_t>(((size_t)P + 7) / 8, (size_t)c->sm_count * 16);
        pair_acc_kernel<<<grid ? grid : 1, 256, 0, c->stream>>>(c->acc[c->acc_cur], c->acc_stride_words, c->acc_words, c->d_r1, c->d_r2, (uint32_t)P, d_in, d_un);
        LAUNCH_CHECK(c);
    }
    timing_end(c);
    return 0;
}

int pansim_pair_counts_rows(pansim_ctx *c, uint32_t row_begin, uint32_t row_end, uint32_t *core_diff, uint32_t *inter,
                            uint32_t *uni, size_t *n_pairs_out)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    // buffers must exist before their addresses are passed on: size them for this block first
    uint64_t P0 = 0;
    for (uint32_t i = row_begin; i < row_end && i < c->N; i++) P0 += (uint64_t)c->N - 1u - i;
    if (P0 > 0x7FFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "more than 2^31 pairs in rows [%u, %u): use smaller row blocks", row_begin, row_end);
    if (P0) if (int rc = ensure_pairs(c, (size_t)P0)) return rc;
    size_t P = 0;
    if (int rc = pair_counts_rows_impl(c, row_begin, row_end, core_diff ? c->d_cd : nullptr, (inter || uni) ? c->d_in : nullptr,
                                       (inter || uni) ? c->d_un : nullptr, &P)) return rc;
    if (n_pairs_out) *n_pairs_out = P;
    if (P == 0) return 0;
    if (core_diff)
        if (int rc = comm_allreduce_counts(c, c->d_cd, P)) return rc;
    if (core_diff) CU(c, cudaMemcpyAsync(core_diff, c->d_cd, P * 4, cudaMemcpyDeviceToHost, c->stream));
    if (inter) CU(c, cudaMemcpyAsync(inter, c->d_in, P * 4, cudaMemcpyDeviceToHost, c->stream));
    if (uni) CU(c, cudaMemcpyAsync(uni, c->d_un, P * 4, cudaMemcpyDeviceToHost, c->stream));
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return flags_inspect(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
}

int pansim_pair_counts_rows_device(pansim_ctx *c, uint32_t row_begin, uint32_t row_end, void *d_cd, void *d_in, void *d_un,
                                   size_t *n_pairs_out)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    size_t P = 0;
    if (int rc = pair_counts_rows_impl(c, row_begin, row_end, (uint32_t *)d_cd, (uint32_t *)d_in, (uint32_t *)d_un, &P)) return rc;
    if (int rc = comm_allreduce_counts(c, (uint32_t *)d_cd, P)) return rc;
    if (n_pairs_out) *n_pairs_out = P;
    if (int rc = flags_enqueue_readback(c)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return flags_inspect(c, PANSIM_ERR_WEIGHTS, "WeightedIndex::new would fail: a weight is negative/NaN or the total is not positive (population.rs:440)");
}

int pansim_gene_counts(pansim_ctx *c, uint32_t *counts)
{
    if (!c || (!counts && c->G)) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (c->G == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    acc_gene_counts_kernel<<<c->acc_words, 256, 0, c->stream>>>(c->acc[c->acc_cur], c->N, c->G, c->acc_stride_words, c->d_gain_thr);
    LAUNCH_CHECK(c);
    CU(c, cudaMemcpyAsync(counts, c->d_gain_thr, (size_t)c->G * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- core-genome diversity (diversity.cuh) ----------------------------------------------------
static int ensure_div(pansim_ctx *c, size_t n, bool sfs)
{
    if (n > c->div_cap) {
        if (c->d_div) cudaFree(c->d_div);
        if (c->h_div) cudaFreeHost(c->h_div);
        c->d_div = nullptr; c->h_div = nullptr; c->div_cap = 0;
        CU(c, cudaMalloc(&c->d_div, n * 4 * sizeof(unsigned long long)));
        CU(c, cudaMallocHost(&c->h_div, n * 4 * sizeof(unsigned long long)));
        c->div_cap = n;
    }
    if (sfs && !c->d_sfs) {
        CU(c, cudaMalloc(&c->d_sfs, ((size_t)c->N + 1) * sizeof(unsigned long long)));
        CU(c, cudaMallocHost(&c->h_sfs, ((size_t)c->N + 1) * sizeof(unsigned long long)));
    }
    return 0;
}

// the column reduction of the current core buffer on `st`: adds into d_out[0..2] (and d_sfs[0..N]), which
// the caller has zeroed; the rows must be materialised
static int launch_diversity(pansim_ctx *c, cudaStream_t st, unsigned long long *d_out, uint4 *d_counts, unsigned long long *d_sfs)
{
    if (c->Ll == 0) return 0;
    DiversityArgs a;
    a.state = reinterpret_cast<const uint32_t *>(c->core[c->core_cur]);
    a.row_words = c->core_stride / 4;
    a.n_sites = c->Ll;
    a.n_rows = c->N;
    a.anc = c->d_anc;
    a.out = d_out;
    a.counts = d_counts;
    a.sfs = d_sfs;
    const uint32_t grid = div_up64(c->Ll, DV_SITES);
    if (d_counts)
        diversity_kernel<true, false><<<grid, DV_THREADS, 0, st>>>(a);
    else if (d_sfs)
        diversity_kernel<false, true><<<grid, DV_THREADS, std::min<size_t>((size_t)c->N + 1, DV_SFS_BINS) * 4, st>>>(a);
    else
        diversity_kernel<false, false><<<grid, DV_THREADS, 0, st>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

static void diversity_from_host(const pansim_ctx *c, const unsigned long long *h, pansim_diversity *out)
{
    out->sites = c->Ll;
    out->segregating = h[0];
    out->multiallelic = h[1];
    out->pair_diff_sum = h[2];
}

// one call's reduction enqueued on c->stream, results into the pinned h_div / h_sfs (the group variant
// enqueues on every shard before it synchronises)
static int core_diversity_enqueue(pansim_ctx *c, bool sfs)
{
    if (int rc = require_state(c)) return rc;
    if (sfs && !c->has_anc) FAIL(c, PANSIM_ERR_STATE, "the SFS needs the ancestral row: call pansim_set_initial first");
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_div(c, 1, sfs)) return rc;
    c->ps = c->stream;
    if (c->Ll)
        if (int rc = core_materialize(c, c->stream)) return rc;
    CU(c, cudaMemsetAsync(c->d_div, 0, 4 * sizeof(unsigned long long), c->stream));
    if (sfs) CU(c, cudaMemsetAsync(c->d_sfs, 0, ((size_t)c->N + 1) * sizeof(unsigned long long), c->stream));
    timing_begin(c);                    // pansim_get_timing: total_ms = the reduction kernel alone
    if (int rc = launch_diversity(c, c->stream, c->d_div, nullptr, sfs ? c->d_sfs : nullptr)) return rc;
    timing_end(c);
    CU(c, cudaMemcpyAsync(c->h_div, c->d_div, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    if (sfs) CU(c, cudaMemcpyAsync(c->h_sfs, c->d_sfs, ((size_t)c->N + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    return flags_enqueue_readback(c);
}

static int core_diversity_finish(pansim_ctx *c, pansim_diversity *out, uint64_t *sfs)
{
    CU(c, cudaSetDevice(c->cfg.device));
    CU(c, cudaStreamSynchronize(c->stream));
    if (int rc = flags_inspect(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG)) return rc;
    diversity_from_host(c, c->h_div, out);
    if (sfs) memcpy(sfs, c->h_sfs, ((size_t)c->N + 1) * sizeof(uint64_t));
    return 0;
}

int pansim_core_allele_counts(pansim_ctx *c, uint32_t *counts)
{
    if (!c || !counts) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (c->Ll == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_div(c, 1, false)) return rc;
    if (int rc = ensure_stage(c, (size_t)c->Ll * 16)) return rc;
    c->ps = c->stream;
    if (int rc = core_materialize(c, c->stream)) return rc;
    CU(c, cudaMemsetAsync(c->d_div, 0, 4 * sizeof(unsigned long long), c->stream));
    if (int rc = launch_diversity(c, c->stream, c->d_div, reinterpret_cast<uint4 *>(c->d_stage), nullptr)) return rc;
    CU(c, cudaMemcpyAsync(counts, c->d_stage, (size_t)c->Ll * 16, cudaMemcpyDeviceToHost, c->stream));
    return check_device_flag(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG);
}

int pansim_core_diversity(pansim_ctx *c, pansim_diversity *out, uint64_t *sfs)
{
    if (!c || !out) return PANSIM_ERR_INVALID;
    if (int rc = core_diversity_enqueue(c, sfs != nullptr)) return rc;
    return core_diversity_finish(c, out, sfs);
}

// One generation of the diversity batch: stats_generation (the step, then on stream_pairs the materialised
// rows and, with P > 0, the distance pass) followed on the same stream by the reduction into d_out. Whatever
// the caller enqueues next on c->ps (all-reduce, statistics launch or the bare ev_pairs record) comes after
// the reduction, so the back-pressure of generation g + 2 on ev_pairs[slot] also keeps core step g + 2 from
// overwriting the buffer the reduction reads.
static int diversity_generation(pansim_ctx *c, uint32_t gen, int slot, size_t P, bool want_acc, unsigned long long *d_out,
                                uint32_t **cd_out, uint32_t **in_out, uint32_t **un_out)
{
    if (int rc = stats_generation(c, gen, slot, P, want_acc, cd_out, in_out, un_out)) return rc;
    if (int rc = launch_diversity(c, c->ps, d_out, nullptr, nullptr)) { c->ps = c->stream; return rc; }
    return 0;
}

// ev_pairs[slot] behind the reduction when no statistics kernel follows (launch_pair_stats records it otherwise)
static int record_pass_done(pansim_ctx *c, int slot)
{
    CU(c, cudaEventRecord(c->ev_pairs[slot], c->ps));
    c->ev_pairs_valid[slot] = true;
    return 0;
}

int pansim_run_generations_diversity(pansim_ctx *c, uint32_t gen0, uint32_t n, const uint32_t *r1, const uint32_t *r2, size_t P,
                                     double *stats_out, pansim_diversity *div_out)
{
    if (!c || !div_out || (P && (!r1 || !r2 || !stats_out))) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (P)
        if (int rc = require_whole_alignment(c, "pansim_run_generations_diversity with pairs")) return rc;
    if (n == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    if (P)
        if (int rc = ensure_pairs(c, P)) return rc;
    if (int rc = ensure_stats(c, n, P, P > 0)) return rc;
    if (int rc = ensure_div(c, n, false)) return rc;
    if (P)
        if (int rc = pair_prepare(c, r1, r2, P)) return rc;
    if (c->dump_enabled) CU(c, cudaMemsetAsync(c->d_dump_counters, 0, 2 * sizeof(uint32_t), c->stream));
    timing_begin(c);
    CU(c, cudaMemsetAsync(c->d_div, 0, (size_t)n * 4 * sizeof(unsigned long long), c->stream));
    for (uint32_t g = 0; g < n; g++) {
        const int slot = (int)(g & 1u);
        uint32_t *cd = nullptr, *in = nullptr, *un = nullptr;
        if (int rc = diversity_generation(c, gen0 + g, slot, P, true, c->d_div + (size_t)g * 4, &cd, &in, &un)) return rc;
        if (P) {
            if (int rc = comm_allreduce_counts(c, cd, P)) return rc;
            if (int rc = launch_pair_stats(c, slot, P, cd, in, un, c->d_stats + (size_t)g * 4)) return rc;
        } else {
            if (int rc = record_pass_done(c, slot)) return rc;
        }
    }
    if (int rc = stats_batch_end(c)) return rc;
    timing_end(c);
    if (P) CU(c, cudaMemcpyAsync(c->h_stats, c->d_stats, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(c->h_div, c->d_div, (size_t)n * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    if (int rc = check_device_flag(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG)) return rc;
    if (P) memcpy(stats_out, c->h_stats, (size_t)n * 4 * sizeof(double));
    for (uint32_t g = 0; g < n; g++) diversity_from_host(c, c->h_div + (size_t)g * 4, div_out + g);
    return 0;
}

// Tajima (1989), Genetics 123:585-595, eq. 4-9 and 38, evaluated in one fixed order so every host gets the same bits
void pansim_diversity_stats(const pansim_diversity *d, uint32_t pop_size, double out[3])
{
    const double nan = std::numeric_limits<double>::quiet_NaN();
    if (!d || !out) return;
    if (pop_size < 2) { out[0] = out[1] = out[2] = nan; return; }
    const double n = (double)pop_size, S = (double)d->segregating;
    double a1 = 0.0, a2 = 0.0;
    for (uint32_t i = 1; i < pop_size; i++) {
        const double x = (double)i;
        a1 += 1.0 / x;
        a2 += 1.0 / (x * x);
    }
    const double pairs = (double)((uint64_t)pop_size * (pop_size - 1u) / 2u);
    const double pi = (double)d->pair_diff_sum / pairs;
    const double theta_w = S / a1;
    const double b1 = (n + 1.0) / (3.0 * (n - 1.0));
    const double b2 = (2.0 * (n * n + n + 3.0)) / (9.0 * n * (n - 1.0));
    const double c1 = b1 - 1.0 / a1;
    const double c2 = b2 - (n + 2.0) / (a1 * n) + a2 / (a1 * a1);
    const double e1 = c1 / a1;
    const double e2 = c2 / (a1 * a1 + a2);
    const double var = e1 * S + e2 * S * (S - 1.0);
    const double den = std::sqrt(var);
    out[0] = pi;
    out[1] = theta_w;
    out[2] = (d->segregating == 0 || !(den > 0.0)) ? nan : (pi - theta_w) / den;
}

// ---- core-genome VCF (vcf.cuh) ----------------------------------------------------------------
constexpr unsigned long long VCF_CHUNK_BYTES = 32ull << 20;     // text per chunk (one line where a line is longer)

// *slot = bytes of device memory unless already allocated; a failed allocation leaves *slot null
static int alloc_once(pansim_ctx *c, void **slot, size_t bytes)
{
    if (*slot) return 0;
    void *p = nullptr;
    CU(c, cudaMalloc(&p, bytes));
    *slot = p;
    return 0;
}

// the per-site allele counts of the VCF and FASTA site passes (one buffer: each pass fills it before it reads it)
static int ensure_site_counts(pansim_ctx *c)
{
    return alloc_once(c, reinterpret_cast<void **>(&c->d_vcf_counts), (size_t)c->Ll * sizeof(uint4));
}

static int ensure_vcf(pansim_ctx *c)
{
    if (int rc = ensure_site_counts(c)) return rc;
    if (c->d_vcf_nchunks) return 0;
    const size_t blocks = div_up64(c->Ll, VS_SITES);
    CU(c, cudaMalloc(&c->d_vcf_desc, blocks * VS_SITES));
    CU(c, cudaMalloc(&c->d_vcf_off, ((size_t)c->Ll + 1) * sizeof(unsigned long long)));
    CU(c, cudaMalloc(&c->d_vcf_block, blocks * sizeof(unsigned long long)));
    CU(c, cudaMalloc(&c->d_vcf_bounds, 2 * ((size_t)c->Ll + 1) * sizeof(unsigned long long)));
    CU(c, cudaMalloc(&c->d_vcf_nchunks, sizeof(uint32_t)));
    return 0;
}

// the site pass on c->stream over materialised rows: allele counts (the counts instance of the diversity
// reduction), descriptors, line offsets (d_vcf_off[Ll] = the whole text) and the chunk bounds
static int vcf_site_pass(pansim_ctx *c)
{
    CU(c, cudaMemsetAsync(c->d_div, 0, 4 * sizeof(unsigned long long), c->stream));
    if (int rc = launch_diversity(c, c->stream, c->d_div, c->d_vcf_counts, nullptr)) return rc;
    VcfSiteArgs a;
    a.counts = c->d_vcf_counts;
    a.anc = c->d_anc;
    a.n_sites = c->Ll;
    a.pos0 = c->site_begin + 1;
    a.n_rows = c->N;
    a.desc = c->d_vcf_desc;
    a.off = c->d_vcf_off;
    a.block = c->d_vcf_block;
    const uint32_t blocks = div_up64(c->Ll, VS_SITES);
    vcf_site_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    vcf_scan_blocks_kernel<<<1, VS_SCAN_THREADS, 0, c->stream>>>(a.block, blocks, c->d_vcf_off + c->Ll);
    LAUNCH_CHECK(c);
    vcf_offsets_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    vcf_chunk_kernel<<<1, VS_SCAN_THREADS, 0, c->stream>>>(c->d_vcf_off, c->Ll, VCF_CHUNK_BYTES, c->d_vcf_bounds, c->d_vcf_nchunks);
    LAUNCH_CHECK(c);
    return 0;
}

// materialise, run the site pass and read back the chunk bounds only: bounds[2k] = first site of chunk k,
// bounds[2k + 1] = its byte offset, the last pair = (Ll, whole text). Empty for a context without sites.
static int vcf_prepare(pansim_ctx *c, std::vector<unsigned long long> &bounds)
{
    bounds.clear();
    if (int rc = require_state(c)) return rc;
    if (!c->has_anc) FAIL(c, PANSIM_ERR_STATE, "the VCF needs the ancestral row: call pansim_set_initial first");
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->Ll == 0) return 0;
    if (int rc = ensure_div(c, 1, false)) return rc;
    if (int rc = ensure_vcf(c)) return rc;
    c->ps = c->stream;
    if (int rc = core_materialize(c, c->stream)) return rc;
    if (int rc = check_hr_flag(c)) return rc;
    if (int rc = vcf_site_pass(c)) return rc;
    uint32_t n = 0;
    CU(c, cudaMemcpyAsync(&n, c->d_vcf_nchunks, sizeof n, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    bounds.resize(2 * ((size_t)n + 1));
    CU(c, cudaMemcpyAsync(bounds.data(), c->d_vcf_bounds, bounds.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// the lines of chunk k (bounds of vcf_prepare) into dst
static int launch_vcf_expand(pansim_ctx *c, const unsigned long long *bk, char *dst)
{
    VcfExpandArgs a;
    a.state = reinterpret_cast<const uint32_t *>(c->core[c->core_cur]);
    a.row_words = c->core_stride / 4;
    a.n_rows = c->N;
    a.desc = c->d_vcf_desc;
    a.off = c->d_vcf_off;
    a.site0 = bk[0];
    a.site1 = bk[2];
    a.base = bk[1];
    a.pos0 = c->site_begin + 1;
    a.out = dst;
    if (bk[3] == bk[1]) return 0;                                   // no line in the chunk
    const dim3 grid(div_up64(a.site1, VX_SITES) - (uint32_t)(a.site0 / VX_SITES), div_up64(c->N, VX_ROWS));
    vcf_expand_kernel<<<grid, VX_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

static size_t vcf_max_chunk(const std::vector<unsigned long long> &bd)
{
    size_t cap = 0;
    for (size_t k = 0; k + 3 < bd.size(); k += 2) cap = std::max<size_t>(cap, bd[k + 3] - bd[k + 1]);
    return cap;
}

// header lines of the file: the contig is the whole alignment, sample ind_i is row i
static std::string vcf_header(uint64_t core_size, uint32_t N)
{
    std::string h = "##fileformat=VCFv4.2\n##source=pansim_b200\n##contig=<ID=core,length=" + std::to_string(core_size) +
                    ">\n##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
                    "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT";
    h.reserve(h.size() + (size_t)N * 12 + 1);
    for (uint32_t i = 0; i < N; i++) {
        h += "\tind_";
        h += std::to_string(i);
    }
    h += '\n';
    return h;
}

// the one writer behind pansim_write_core_vcf and pansim_group_write_core_vcf: optionally the header, then
// the context's lines with global POS, appended to f; *total counts the bytes handed to f
static int write_core_vcf_to(pansim_ctx *c, FILE *f, bool header, uint64_t *total)
{
    std::vector<unsigned long long> bd;
    if (int rc = vcf_prepare(c, bd)) return rc;
    auto sink = [&](const char *p, size_t n) { *total += n; return fwrite(p, 1, n, f) == n ? 0 : 1; };
    if (header) {
        const std::string h = vcf_header(c->L, c->N);
        if (sink(h.data(), h.size())) FAIL(c, PANSIM_ERR_INVALID, "VCF export: writing the header failed");
    }
    const size_t cap = vcf_max_chunk(bd);
    if (cap == 0) return 0;                                         // no site differs from the ancestral row
    const size_t n_chunks = bd.size() / 2 - 1;
    return stream_text_chunks(c, n_chunks, cap, "VCF", [&](size_t k, char *dst, size_t *bytes) -> int {
        *bytes = bd[2 * k + 3] - bd[2 * k + 1];
        return launch_vcf_expand(c, &bd[2 * k], dst);
    }, sink);
}

int pansim_write_core_vcf(pansim_ctx *c, const char *path, int with_header, uint64_t *bytes_out)
{
    if (!c || !path) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    if (!c->has_anc) FAIL(c, PANSIM_ERR_STATE, "the VCF needs the ancestral row: call pansim_set_initial first");
    FILE *f = fopen(path, "wb");
    if (!f) FAIL(c, PANSIM_ERR_INVALID, "cannot create %s", path);
    uint64_t total = 0;
    const int rc = write_core_vcf_to(c, f, with_header != 0, &total);
    const int rc2 = fclose(f);
    if (bytes_out) *bytes_out = total;
    if (rc) return rc;
    if (rc2) FAIL(c, PANSIM_ERR_INVALID, "closing %s failed", path);
    return 0;
}

int pansim_core_vcf_kernel_ms(pansim_ctx *c, uint32_t repeats, float *site_ms, float *expand_ms, uint64_t *text_bytes)
{
    if (!c || !repeats) return PANSIM_ERR_INVALID;
    std::vector<unsigned long long> bd;
    if (int rc = vcf_prepare(c, bd)) return rc;                     // also the warm-up of the site pass
    if (bd.empty()) FAIL(c, PANSIM_ERR_INVALID, "no core sites on this context");
    if (int rc = ensure_txt_staging(c, std::max<size_t>(1, vcf_max_chunk(bd)), "VCF")) return rc;
    const size_t n_chunks = bd.size() / 2 - 1;
    for (size_t k = 0; k < n_chunks; k++)                           // warm-up of the expansion
        if (int rc = launch_vcf_expand(c, &bd[2 * k], c->d_txt[k & 1])) return rc;
    cudaEvent_t ev[3];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    int rc = 0;
    cudaEventRecord(ev[0], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++) rc = vcf_site_pass(c);
    cudaEventRecord(ev[1], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++)
        for (size_t k = 0; k < n_chunks && !rc; k++) rc = launch_vcf_expand(c, &bd[2 * k], c->d_txt[k & 1]);
    cudaEventRecord(ev[2], c->stream);
    const cudaError_t e = cudaEventSynchronize(ev[2]);
    float t0 = 0.f, t1 = 0.f;
    cudaEventElapsedTime(&t0, ev[0], ev[1]);
    cudaEventElapsedTime(&t1, ev[1], ev[2]);
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (e != cudaSuccess) FAIL(c, PANSIM_ERR_CUDA, "VCF kernels failed: %s", cudaGetErrorString(e));
    if (site_ms) *site_ms = t0 / (float)repeats;
    if (expand_ms) *expand_ms = t1 / (float)repeats;
    if (text_bytes) *text_bytes = bd.back();
    return 0;
}

// ---- core-genome FASTA (fasta.cuh) ------------------------------------------------------------
constexpr uint64_t FASTA_CHUNK_BYTES = 32ull << 20;   // text per chunk: whole records (one record where a record is longer)

// every buffer is allocated on its own when missing, so a failed allocation leaves nothing to leak on the next call
static int ensure_fasta(pansim_ctx *c)
{
    if (int rc = ensure_site_counts(c)) return rc;
    const size_t blocks = div_up64(c->Ll, VS_SITES);
    if (int rc = alloc_once(c, reinterpret_cast<void **>(&c->d_fa_block), (blocks + 1) * sizeof(unsigned long long))) return rc;
    if (int rc = alloc_once(c, reinterpret_cast<void **>(&c->d_fa_const), 4 * sizeof(unsigned long long))) return rc;
    if (int rc = alloc_once(c, reinterpret_cast<void **>(&c->d_fa_cols), (size_t)c->Ll * sizeof(uint32_t))) return rc;
    if (!c->h_fa) {
        void *p = nullptr;
        CU(c, cudaMallocHost(&p, 5 * sizeof(unsigned long long)));
        c->h_fa = static_cast<unsigned long long *>(p);
    }
    return 0;
}

// the SNP-mode site pass on c->stream over materialised rows: allele counts (the counts instance of the diversity
// reduction), polymorphic sites and constant-site letters per block, the scan of the blocks and the column list
static int fasta_site_pass(pansim_ctx *c)
{
    CU(c, cudaMemsetAsync(c->d_div, 0, 4 * sizeof(unsigned long long), c->stream));
    CU(c, cudaMemsetAsync(c->d_fa_const, 0, 4 * sizeof(unsigned long long), c->stream));
    if (int rc = launch_diversity(c, c->stream, c->d_div, c->d_vcf_counts, nullptr)) return rc;
    FastaSiteArgs a;
    a.counts = c->d_vcf_counts;
    a.n_sites = c->Ll;
    a.block = c->d_fa_block;
    a.consts = c->d_fa_const;
    a.cols = c->d_fa_cols;
    const uint32_t blocks = div_up64(c->Ll, VS_SITES);
    fasta_site_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    vcf_scan_blocks_kernel<<<1, VS_SCAN_THREADS, 0, c->stream>>>(a.block, blocks, a.block + blocks);
    LAUNCH_CHECK(c);
    fasta_compact_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

// Materialise the rows and, in SNP mode, enqueue the site pass and the read-back of the column count and the
// constant-site letters into h_fa, without waiting for them (the group enqueues on every shard first). Whole mode
// needs no pass: every local site is a column.
static int fasta_enqueue(pansim_ctx *c, bool snps)
{
    if (int rc = require_state(c)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->Ll == 0) return 0;
    c->ps = c->stream;
    if (int rc = core_materialize(c, c->stream)) return rc;
    if (int rc = check_hr_flag(c)) return rc;
    if (!snps) return 0;
    if (int rc = ensure_div(c, 1, false)) return rc;
    if (int rc = ensure_fasta(c)) return rc;
    if (int rc = fasta_site_pass(c)) return rc;
    CU(c, cudaMemcpyAsync(c->h_fa, c->d_fa_block + div_up64(c->Ll, VS_SITES), sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(c->h_fa + 1, c->d_fa_const, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

// the column count and constant-site letters of fasta_enqueue, once it has finished
static int fasta_columns(pansim_ctx *c, bool snps, uint64_t *cols, uint64_t consts[4])
{
    for (int k = 0; k < 4; k++) consts[k] = 0;
    *cols = snps ? 0 : c->Ll;
    if (!snps || c->Ll == 0) return 0;
    CU(c, cudaSetDevice(c->cfg.device));
    CU(c, cudaStreamSynchronize(c->stream));
    *cols = c->h_fa[0];
    for (int k = 0; k < 4; k++) consts[k] = c->h_fa[1 + k];
    return 0;
}

// rows [r0, r1) with `cols` columns into dst on c->stream: whole records when framed, the letters only otherwise
static int launch_fasta_expand(pansim_ctx *c, bool snps, uint64_t cols, uint32_t r0, uint32_t r1, bool framed, char *dst)
{
    if (r0 == r1 || (!framed && cols == 0)) return 0;
    FastaExpandArgs a;
    a.state = reinterpret_cast<const uint32_t *>(c->core[c->core_cur]);
    a.row_words = c->core_stride / 4;
    a.cols = snps ? c->d_fa_cols : nullptr;
    a.n_cols = cols;
    a.row0 = r0;
    a.row1 = r1;
    a.framed = framed ? 1u : 0u;
    a.out = dst;
    const dim3 grid(std::max<uint32_t>(1, div_up64(cols, FX_COLS)), div_up64(r1 - r0, FX_ROWS));
    fasta_expand_kernel<<<grid, FX_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

// rows per chunk of at most FASTA_CHUNK_BYTES when a row takes at most row_bytes (at least one row)
static uint32_t fasta_rows_per_chunk(uint64_t row_bytes, uint32_t n_rows)
{
    return (uint32_t)std::min<uint64_t>(std::max<uint32_t>(1, n_rows), std::max<uint64_t>(1, FASTA_CHUNK_BYTES / std::max<uint64_t>(1, row_bytes)));
}

// the largest record of rows below n_rows
static uint64_t fasta_max_record(uint32_t n_rows, uint64_t cols) { return 7 + vcf_digits(n_rows ? n_rows - 1 : 0) + cols; }

// rows [row_begin, row_end) streamed to sink in chunks of whole records (framed) or of letter rows
extern "C++" {
template <typename Sink>
static int fasta_stream(pansim_ctx *c, bool snps, uint64_t cols, uint32_t row_begin, uint32_t row_end, bool framed, Sink &&sink)
{
    const uint64_t row_bytes = framed ? fasta_max_record(row_end, cols) : cols;
    if (row_begin == row_end || row_bytes == 0) return 0;
    const uint32_t rows_per = fasta_rows_per_chunk(row_bytes, row_end - row_begin);
    const size_t n_chunks = div_up64(row_end - row_begin, rows_per);
    return stream_text_chunks(c, n_chunks, (size_t)rows_per * row_bytes, "FASTA", [&](size_t k, char *dst, size_t *bytes) -> int {
        const uint32_t r0 = row_begin + (uint32_t)k * rows_per, r1 = std::min(row_end, r0 + rows_per);
        *bytes = framed ? fasta_record_offset(r1, cols) - fasta_record_offset(r0, cols) : (uint64_t)(r1 - r0) * cols;
        return launch_fasta_expand(c, snps, cols, r0, r1, framed, dst);
    }, sink);
}
}  // extern "C++"

int pansim_write_core_fasta(pansim_ctx *c, const char *path, int snps_only, uint64_t *columns_out, uint64_t *const_counts,
                            uint64_t *bytes_out)
{
    if (!c || !path) return PANSIM_ERR_INVALID;
    if (int rc = require_state(c)) return rc;
    const bool snps = snps_only != 0;
    FILE *f = fopen(path, "wb");
    if (!f) FAIL(c, PANSIM_ERR_INVALID, "cannot create %s", path);
    uint64_t total = 0, cols = 0, consts[4];
    int rc = fasta_enqueue(c, snps);
    if (!rc) rc = fasta_columns(c, snps, &cols, consts);
    if (!rc) rc = fasta_stream(c, snps, cols, 0, c->N, true, [&](const char *p, size_t n) { total += n; return fwrite(p, 1, n, f) == n ? 0 : 1; });
    const int rc2 = fclose(f);
    if (bytes_out) *bytes_out = total;
    if (rc) return rc;
    if (rc2) FAIL(c, PANSIM_ERR_INVALID, "closing %s failed", path);
    if (columns_out) *columns_out = cols;
    if (const_counts) memcpy(const_counts, consts, sizeof consts);
    return 0;
}

int pansim_export_core_fasta_rows(pansim_ctx *c, int snps_only, uint32_t row_begin, uint32_t row_end, char *out, uint64_t *columns_out)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (row_begin > row_end || row_end > c->N) FAIL(c, PANSIM_ERR_INVALID, "rows [%u, %u) out of range", row_begin, row_end);
    const bool snps = snps_only != 0;
    uint64_t cols = 0, consts[4];
    if (int rc = fasta_enqueue(c, snps)) return rc;
    if (int rc = fasta_columns(c, snps, &cols, consts)) return rc;
    if (columns_out) *columns_out = cols;
    if (!out) return 0;
    char *dst = out;
    return fasta_stream(c, snps, cols, row_begin, row_end, false, [&](const char *p, size_t n) { memcpy(dst, p, n); dst += n; return 0; });
}

int pansim_core_fasta_kernel_ms(pansim_ctx *c, int snps_only, uint32_t repeats, float *site_ms, float *expand_ms, uint64_t *text_bytes)
{
    if (!c || !repeats) return PANSIM_ERR_INVALID;
    const bool snps = snps_only != 0;
    uint64_t cols = 0, consts[4];
    if (int rc = fasta_enqueue(c, snps)) return rc;                 // also the warm-up of the site pass
    if (int rc = fasta_columns(c, snps, &cols, consts)) return rc;
    if (c->Ll == 0) FAIL(c, PANSIM_ERR_INVALID, "no core sites on this context");
    const uint64_t row_bytes = fasta_max_record(c->N, cols);
    const uint32_t rows_per = fasta_rows_per_chunk(row_bytes, c->N);
    const size_t n_chunks = div_up64(c->N, rows_per);
    if (int rc = ensure_txt_staging(c, (size_t)rows_per * row_bytes, "FASTA")) return rc;
    auto expand_all = [&]() -> int {
        for (size_t k = 0; k < n_chunks; k++) {
            const uint32_t r0 = (uint32_t)k * rows_per, r1 = std::min(c->N, r0 + rows_per);
            if (int rc = launch_fasta_expand(c, snps, cols, r0, r1, true, c->d_txt[k & 1])) return rc;
        }
        return 0;
    };
    if (int rc = expand_all()) return rc;                           // warm-up of the expansion
    cudaEvent_t ev[3];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    int rc = 0;
    cudaEventRecord(ev[0], c->stream);
    for (uint32_t r = 0; r < repeats && !rc && snps; r++) rc = fasta_site_pass(c);
    cudaEventRecord(ev[1], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++) rc = expand_all();
    cudaEventRecord(ev[2], c->stream);
    const cudaError_t e = cudaEventSynchronize(ev[2]);
    float t0 = 0.f, t1 = 0.f;
    cudaEventElapsedTime(&t0, ev[0], ev[1]);
    cudaEventElapsedTime(&t1, ev[1], ev[2]);
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (e != cudaSuccess) FAIL(c, PANSIM_ERR_CUDA, "FASTA kernels failed: %s", cudaGetErrorString(e));
    if (site_ms) *site_ms = t0 / (float)repeats;
    if (expand_ms) *expand_ms = t1 / (float)repeats;
    if (text_bytes) *text_bytes = fasta_record_offset(c->N, cols);
    return 0;
}

// ---- core-genome linkage disequilibrium (ld.cuh) ---------------------------------------------
using LdBuf = pansim_ctx::LdBuf;

// counts and ranks of n_sites sites, the compacted arrays of n_used used sites (grown, never shrunk)
static int ld_ensure_sites(pansim_ctx *c, LdBuf &b, size_t n_sites, size_t n_used)
{
    if (n_sites > b.site_cap) {
        for (void *p : {(void *)b.counts, (void *)b.block, (void *)b.rank})
            if (p) cudaFree(p);
        b.counts = nullptr; b.block = nullptr; b.rank = nullptr; b.site_cap = 0;
        CU(c, cudaMalloc(&b.counts, n_sites * sizeof(uint4)));
        CU(c, cudaMalloc(&b.block, ((size_t)div_up64(n_sites, VS_SITES) + 1) * sizeof(unsigned long long)));
        CU(c, cudaMalloc(&b.rank, n_sites * sizeof(uint32_t)));
        b.site_cap = n_sites;
    }
    if (n_used > b.used_cap) {
        for (void *p : {(void *)b.pos, (void *)b.a, (void *)b.inv})
            if (p) cudaFree(p);
        b.pos = nullptr; b.a = nullptr; b.inv = nullptr; b.used_cap = 0;
        CU(c, cudaMalloc(&b.pos, n_used * sizeof(uint32_t)));
        CU(c, cudaMalloc(&b.a, n_used * sizeof(uint32_t)));
        CU(c, cudaMalloc(&b.inv, n_used * sizeof(double)));
        b.used_cap = n_used;
    }
    return 0;
}

// the site-major bit rows of n_used used sites (kept with the context, like the intersection matrix)
static int ld_ensure_x(pansim_ctx *c, LdBuf &b, size_t n_used)
{
    const size_t bytes = std::max<size_t>(1, n_used) * ld_row_words(c->N) * sizeof(uint32_t);
    if (bytes <= b.x_cap) return 0;
    if (b.x) cudaFree(b.x);
    b.x = nullptr; b.x_cap = 0;
    if (cudaMalloc(&b.x, bytes) != cudaSuccess) {
        cudaGetLastError();
        FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (LD bit rows) failed", bytes);
    }
    b.x_cap = bytes;
    return 0;
}

static int ld_ensure_host(pansim_ctx *c, size_t n_bins)
{
    if (!c->h_ld) CU(c, cudaMallocHost(&c->h_ld, 4 * sizeof(unsigned long long)));
    if (!c->ev_ld) CU(c, cudaEventCreateWithFlags(&c->ev_ld, cudaEventDisableTiming));
    if (n_bins > c->h_ld_bins_cap) {
        if (c->h_ld_bins) cudaFreeHost(c->h_ld_bins);
        c->h_ld_bins = nullptr; c->h_ld_bins_cap = 0;
        CU(c, cudaMallocHost(&c->h_ld_bins, n_bins * 4 * sizeof(unsigned long long)));
        c->h_ld_bins_cap = n_bins;
    }
    return 0;
}

// site pass over the first n local sites of c (materialised rows) into b on c->stream: allele counts, used sites,
// their ranks and compacted arrays; the number of used sites is b.block[n_blocks], copied to *h_used if given
static int ld_site_pass(pansim_ctx *c, LdBuf &b, uint64_t n, uint32_t min_minor, unsigned long long *h_used)
{
    DiversityArgs d;
    d.state = reinterpret_cast<const uint32_t *>(c->core[c->core_cur]);
    d.row_words = c->core_stride / 4;
    d.n_sites = n;
    d.n_rows = c->N;
    d.anc = c->d_anc;
    d.out = c->d_div;
    d.counts = b.counts;
    d.sfs = nullptr;
    CU(c, cudaMemsetAsync(c->d_div, 0, 4 * sizeof(unsigned long long), c->stream));
    diversity_kernel<true, false><<<div_up64(n, DV_SITES), DV_THREADS, 0, c->stream>>>(d);
    LAUNCH_CHECK(c);
    LdSiteArgs a;
    a.counts = b.counts;
    a.anc = c->d_anc;
    a.n_sites = n;
    a.n_rows = c->N;
    a.min_minor = min_minor;
    a.pos0 = (uint32_t)c->site_begin;
    a.block = b.block;
    a.rank = b.rank;
    a.pos = b.pos;
    a.a = b.a;
    a.inv = b.inv;
    const uint32_t blocks = div_up64(n, VS_SITES);
    ld_site_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    vcf_scan_blocks_kernel<<<1, VS_SCAN_THREADS, 0, c->stream>>>(b.block, blocks, b.block + blocks);
    LAUNCH_CHECK(c);
    ld_compact_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    if (h_used) CU(c, cudaMemcpyAsync(h_used, b.block + blocks, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

// derived bit rows of the used sites among the first n local sites of c into x (row k = rank k)
static int ld_transpose(pansim_ctx *c, const LdBuf &b, uint64_t n, uint32_t *x)
{
    LdTransposeArgs a;
    a.state = reinterpret_cast<const uint32_t *>(c->core[c->core_cur]);
    a.row_words = c->core_stride / 4;
    a.n_rows = c->N;
    a.n_sites = n;
    a.anc = c->d_anc;
    a.rank = b.rank;
    a.kw = ld_row_words(c->N);
    a.x = x;
    const dim3 grid(div_up64(n, LT_SITES), div_up64((uint64_t)a.kw * 32, LT_ROWS));
    ld_transpose_kernel<<<grid, LT_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

// tile-pair offsets of the `own` used sites against all `own + halo` of them; the total goes to *h_tiles if given
static int ld_tile_list(pansim_ctx *c, uint64_t own, uint64_t all, uint32_t max_dist, unsigned long long *h_tiles)
{
    const uint32_t n_i = div_up64(own, LD_TILE);
    if ((size_t)n_i + 1 > c->ld_tiles_cap) {
        if (c->d_ld_tiles) cudaFree(c->d_ld_tiles);
        c->d_ld_tiles = nullptr; c->ld_tiles_cap = 0;
        CU(c, cudaMalloc(&c->d_ld_tiles, ((size_t)n_i + 1) * sizeof(unsigned long long)));
        c->ld_tiles_cap = (size_t)n_i + 1;
    }
    ld_tiles_kernel<<<div_up64(n_i, 256), 256, 0, c->stream>>>(c->ld.pos, (uint32_t)own, (uint32_t)all, max_dist, c->d_ld_tiles);
    LAUNCH_CHECK(c);
    vcf_scan_blocks_kernel<<<1, VS_SCAN_THREADS, 0, c->stream>>>(c->d_ld_tiles, n_i, c->d_ld_tiles + n_i);
    LAUNCH_CHECK(c);
    if (h_tiles) CU(c, cudaMemcpyAsync(h_tiles, c->d_ld_tiles + n_i, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

static uint32_t ld_n_bins(const pansim_ld_params *p) { return (uint32_t)(((uint64_t)p->max_dist + p->bin_width - 1) / p->bin_width); }

// zeroed bins, then the pair kernel over `tiles` tile pairs
static int ld_pairs(pansim_ctx *c, const pansim_ld_params *p, uint64_t own, uint64_t all, uint64_t tiles)
{
    const uint32_t n_bins = ld_n_bins(p);
    if (n_bins > c->ld_bins_cap) {
        if (c->d_ld_bins) cudaFree(c->d_ld_bins);
        c->d_ld_bins = nullptr; c->ld_bins_cap = 0;
        CU(c, cudaMalloc(&c->d_ld_bins, (size_t)n_bins * 4 * sizeof(unsigned long long)));
        c->ld_bins_cap = n_bins;
    }
    CU(c, cudaMemsetAsync(c->d_ld_bins, 0, (size_t)n_bins * 4 * sizeof(unsigned long long), c->stream));
    if (!tiles) return 0;
    if (tiles > 0x7FFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "%llu LD tile pairs: more than one launch holds", (unsigned long long)tiles);
    LdPairArgs a;
    a.x = c->ld.x;
    a.kw = ld_row_words(c->N);
    a.k_iters = a.kw * 32 / LD_KB;
    a.pos = c->ld.pos;
    a.a = c->ld.a;
    a.inv = c->ld.inv;
    a.n_own = (uint32_t)own;
    a.n_all = (uint32_t)all;
    a.n_rows = c->N;
    a.max_dist = p->max_dist;
    a.bin_width = p->bin_width;
    a.n_bins = n_bins;
    a.tile_off = c->d_ld_tiles;
    a.n_i = div_up64(own, LD_TILE);
    a.bins = c->d_ld_bins;
    const size_t smem = ld_pair_smem_bytes(n_bins);
    CU(c, cudaFuncSetAttribute(ld_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ld_pair_kernel<<<(uint32_t)tiles, LD_THREADS, smem, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

// Refusals leave the context as it was. Errors of `next` are reported on c.
static int ld_validate(pansim_ctx *c, pansim_ctx *next, const pansim_ld_params *p)
{
    if (!p->max_dist || !p->bin_width || !p->min_minor) FAIL(c, PANSIM_ERR_INVALID, "LD: max_dist, bin_width and min_minor must be >= 1");
    if (int rc = require_state(c)) return rc;
    if (!c->has_anc) FAIL(c, PANSIM_ERR_STATE, "LD needs the ancestral row: call pansim_set_initial first");
    if (c->site_end > 0xFFFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "LD: site positions above 2^32-1");
    if (next) {
        if (next == c || next->N != c->N || next->site_begin != c->site_end)
            FAIL(c, PANSIM_ERR_INVALID, "LD: next must hold the sites right after this context's, with the same pop_size");
        if (!next->has_core || !next->has_anc) FAIL(c, PANSIM_ERR_STATE, "LD: the next context has no state or no ancestral row");
        if (p->max_dist > next->Ll) FAIL(c, PANSIM_ERR_INVALID, "LD: max_dist %u exceeds the %llu sites of the next context", p->max_dist, (unsigned long long)next->Ll);
    }
    return 0;
}

// One context's share of the LD pass in three enqueued phases; between them the host reads the used-site and
// tile-pair counts. A list of jobs runs every phase on all of them before it waits, so the devices overlap.
struct LdJob {
    pansim_ctx *c, *next;
    uint64_t own = 0, halo = 0, tiles = 0;
};

static int ld_sync(pansim_ctx *c)
{
    CU(c, cudaSetDevice(c->cfg.device));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// a failure on `next` reported on c
static int ld_on_next(pansim_ctx *c, pansim_ctx *next, int rc)
{
    if (rc) c->err = "next context: " + next->err;
    return rc;
}

static int ld_phase_sites(LdJob &j, const pansim_ld_params *p)
{
    pansim_ctx *c = j.c, *nx = j.next;
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = ensure_div(c, 1, false)) return rc;
    if (int rc = ld_ensure_host(c, ld_n_bins(p))) return rc;
    if (int rc = ld_ensure_sites(c, c->ld, c->Ll, c->Ll + (nx ? p->max_dist : 0))) return rc;
    c->ps = c->stream;
    if (int rc = core_materialize(c, c->stream)) return rc;
    if (int rc = check_hr_flag(c)) return rc;
    c->h_ld[1] = 0;
    if (int rc = ld_site_pass(c, c->ld, c->Ll, p->min_minor, c->h_ld)) return rc;
    if (nx) {
        CU(c, cudaSetDevice(nx->cfg.device));
        int rc = ensure_div(nx, 1, false);
        if (!rc) rc = ld_ensure_sites(nx, nx->ld_halo, p->max_dist, p->max_dist);
        if (!rc) rc = ld_ensure_host(nx, 1);
        if (!rc) { nx->ps = nx->stream; rc = core_materialize(nx, nx->stream); }
        if (!rc) rc = check_hr_flag(nx);
        if (!rc) rc = ld_site_pass(nx, nx->ld_halo, p->max_dist, p->min_minor, c->h_ld + 1);
        if (rc) return ld_on_next(c, nx, rc);
    }
    return 0;
}

static int ld_phase_rows(LdJob &j, const pansim_ld_params *p)
{
    pansim_ctx *c = j.c, *nx = j.next;
    if (int rc = ld_sync(c)) return rc;
    if (nx)
        if (int rc = ld_sync(nx)) return ld_on_next(c, nx, rc);
    j.own = c->h_ld[0];
    j.halo = nx ? c->h_ld[1] : 0;
    CU(c, cudaSetDevice(c->cfg.device));
    if (!j.own) return 0;
    const uint64_t kw = ld_row_words(c->N);
    if (int rc = ld_ensure_x(c, c->ld, j.own + j.halo)) return rc;
    if (int rc = ld_transpose(c, c->ld, c->Ll, c->ld.x)) return rc;
    if (j.halo) {
        // the halo: the used sites among the next context's first max_dist sites, made on its device and stream,
        // then copied behind ctx's own used sites
        CU(c, cudaSetDevice(nx->cfg.device));
        int rc = ld_ensure_x(nx, nx->ld_halo, j.halo);
        if (!rc) rc = ld_transpose(nx, nx->ld_halo, p->max_dist, nx->ld_halo.x);
        if (!rc && cudaEventRecord(nx->ev_ld, nx->stream) != cudaSuccess) { nx->err = "cudaEventRecord failed"; rc = PANSIM_ERR_CUDA; }
        if (rc) return ld_on_next(c, nx, rc);
        CU(c, cudaSetDevice(c->cfg.device));
        CU(c, cudaStreamWaitEvent(c->stream, nx->ev_ld, 0));
        const LdBuf &h = nx->ld_halo;
        struct Part { void *dst; const void *src; size_t bytes; } parts[] = {
            {c->ld.x + j.own * kw, h.x, j.halo * kw * sizeof(uint32_t)}, {c->ld.pos + j.own, h.pos, j.halo * sizeof(uint32_t)},
            {c->ld.a + j.own, h.a, j.halo * sizeof(uint32_t)}, {c->ld.inv + j.own, h.inv, j.halo * sizeof(double)}};
        for (const Part &q : parts) {
            if (c->cfg.device == nx->cfg.device) CU(c, cudaMemcpyAsync(q.dst, q.src, q.bytes, cudaMemcpyDeviceToDevice, c->stream));
            else CU(c, cudaMemcpyPeerAsync(q.dst, c->cfg.device, q.src, nx->cfg.device, q.bytes, c->stream));
        }
    }
    return ld_tile_list(c, j.own, j.own + j.halo, p->max_dist, c->h_ld + 2);
}

static int ld_phase_pairs(LdJob &j, const pansim_ld_params *p)
{
    pansim_ctx *c = j.c;
    if (int rc = ld_sync(c)) return rc;
    j.tiles = j.own ? c->h_ld[2] : 0;
    if (int rc = ld_pairs(c, p, j.own, j.own + j.halo, j.tiles)) return rc;
    CU(c, cudaMemcpyAsync(c->h_ld_bins, c->d_ld_bins, (size_t)ld_n_bins(p) * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    return flags_enqueue_readback(c);
}

// adds job j's bins into out (the 128-bit sums with carry)
static int ld_finish(LdJob &j, const pansim_ld_params *p, pansim_ld_bin *out, uint64_t *used)
{
    pansim_ctx *c = j.c;
    if (int rc = ld_sync(c)) return rc;
    if (int rc = flags_inspect(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG)) return rc;
    for (uint32_t b = 0; b < ld_n_bins(p); b++) {
        const unsigned long long *h = c->h_ld_bins + 4 * (size_t)b;
        out[b].pairs += h[0];
        out[b].four_gamete += h[1];
        const uint64_t lo = out[b].r2_lo + h[3];
        out[b].r2_hi += h[2] + (lo < h[3] ? 1u : 0u);
        out[b].r2_lo = lo;
    }
    *used += j.own;
    return 0;
}

// the phases over all jobs; on failure *failed = the job's index
static int ld_run(std::vector<LdJob> &jobs, const pansim_ld_params *p, pansim_ld_bin *bins, uint64_t *used, size_t *failed)
{
    memset(bins, 0, (size_t)ld_n_bins(p) * sizeof(pansim_ld_bin));
    *used = 0;
    for (auto phase : {ld_phase_sites, ld_phase_rows, ld_phase_pairs})
        for (size_t i = 0; i < jobs.size(); i++)
            if (int rc = phase(jobs[i], p)) { *failed = i; return rc; }
    for (size_t i = 0; i < jobs.size(); i++)
        if (int rc = ld_finish(jobs[i], p, bins, used)) { *failed = i; return rc; }
    return 0;
}

int pansim_core_ld(pansim_ctx *c, pansim_ctx *next, const pansim_ld_params *p, pansim_ld_bin *bins, uint64_t *sites_used)
{
    if (!c || !p || !bins) return PANSIM_ERR_INVALID;
    if (int rc = ld_validate(c, next, p)) return rc;
    std::vector<LdJob> jobs{{c, next}};
    uint64_t used = 0;
    size_t failed = 0;
    if (int rc = ld_run(jobs, p, bins, &used, &failed)) return rc;
    if (sites_used) *sites_used = used;
    return 0;
}

int pansim_core_ld_kernel_ms(pansim_ctx *c, const pansim_ld_params *p, uint32_t repeats, float *site_ms, float *transpose_ms,
                             float *pair_ms, uint64_t *pairs)
{
    if (!c || !p || !repeats) return PANSIM_ERR_INVALID;
    if (int rc = ld_validate(c, nullptr, p)) return rc;
    std::vector<LdJob> jobs{{c, nullptr}};
    std::vector<pansim_ld_bin> bins(ld_n_bins(p));
    uint64_t used = 0;
    size_t failed = 0;
    if (int rc = ld_run(jobs, p, bins.data(), &used, &failed)) return rc;       // also the warm-up
    const LdJob &j = jobs[0];
    cudaEvent_t ev[4];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    int rc = 0;
    cudaEventRecord(ev[0], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++) rc = ld_site_pass(c, c->ld, c->Ll, p->min_minor, nullptr);
    cudaEventRecord(ev[1], c->stream);
    for (uint32_t r = 0; r < repeats && !rc && j.own; r++) rc = ld_transpose(c, c->ld, c->Ll, c->ld.x);
    cudaEventRecord(ev[2], c->stream);
    for (uint32_t r = 0; r < repeats && !rc && j.own; r++) {
        rc = ld_tile_list(c, j.own, j.own, p->max_dist, nullptr);
        if (!rc) rc = ld_pairs(c, p, j.own, j.own, j.tiles);
    }
    cudaEventRecord(ev[3], c->stream);
    const cudaError_t e = cudaEventSynchronize(ev[3]);
    float t[3] = {0.f, 0.f, 0.f};
    for (int k = 0; k < 3; k++) cudaEventElapsedTime(&t[k], ev[k], ev[k + 1]);
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (e != cudaSuccess) FAIL(c, PANSIM_ERR_CUDA, "LD kernels failed: %s", cudaGetErrorString(e));
    if (site_ms) *site_ms = t[0] / (float)repeats;
    if (transpose_ms) *transpose_ms = t[1] / (float)repeats;
    if (pair_ms) *pair_ms = t[2] / (float)repeats;
    if (pairs) {
        *pairs = 0;
        for (const pansim_ld_bin &b : bins) *pairs += b.pairs;
    }
    return 0;
}

// mean r^2 of a bin from its exact integer sum; the same bits on every host
double pansim_ld_mean_r2(const pansim_ld_bin *b)
{
    if (!b || !b->pairs) return std::numeric_limits<double>::quiet_NaN();
    return (std::ldexp((double)b->r2_hi, 32) + std::ldexp((double)b->r2_lo, -32)) / (double)b->pairs;
}

// ---- accessory-gene LD (gene_ld.cuh, DESIGN.md section 15) ---------------------------------------
// output words: the class totals, the histogram [3][r2_bins], then the used genes of group 1
static size_t gene_ld_out_words(uint32_t r2_bins) { return GL_OUT_CLASSES + 3 * (size_t)r2_bins + 1; }

// the per-gene arrays (G is fixed per context, so they are allocated once) and the outputs for r2_bins
static int gene_ld_ensure(pansim_ctx *c, uint32_t r2_bins)
{
    auto &b = c->gl;
    if (!b.counts) {
        const size_t G = c->G;
        CU(c, cudaMalloc(&b.counts, G * sizeof(uint32_t)));
        CU(c, cudaMalloc(&b.rank, G * sizeof(uint32_t)));
        CU(c, cudaMalloc(&b.a, G * sizeof(uint32_t)));
        CU(c, cudaMalloc(&b.grp, G * sizeof(uint32_t)));
        CU(c, cudaMalloc(&b.inv, G * sizeof(double)));
        CU(c, cudaMalloc(&b.block, ((size_t)div_up64(G, VS_SITES) + 1) * sizeof(unsigned long long)));
    }
    const size_t words = gene_ld_out_words(r2_bins);
    if (words > b.out_cap) {
        if (b.out) cudaFree(b.out);
        if (b.h_out) cudaFreeHost(b.h_out);
        b.out = nullptr; b.h_out = nullptr; b.out_cap = 0;
        CU(c, cudaMalloc(&b.out, words * sizeof(unsigned long long)));
        CU(c, cudaMallocHost(&b.h_out, words * sizeof(unsigned long long)));
        b.out_cap = words;
    }
    return 0;
}

// the gene-major bit rows of n_used used genes (kept with the context, like the core LD rows)
static int gene_ld_ensure_x(pansim_ctx *c, size_t n_used)
{
    const size_t bytes = std::max<size_t>(1, n_used) * ld_row_words(c->N) * sizeof(uint32_t);
    if (bytes <= c->gl.x_cap) return 0;
    if (c->gl.x) cudaFree(c->gl.x);
    c->gl.x = nullptr; c->gl.x_cap = 0;
    if (cudaMalloc(&c->gl.x, bytes) != cudaSuccess) {
        cudaGetLastError();
        FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (gene LD bit rows) failed", bytes);
    }
    c->gl.x_cap = bytes;
    return 0;
}

// gene pass on c->stream: presence counts (K8), used genes, their ranks and compacted arrays, the used genes of
// group 1 (zeroed here); the number of used genes is block[n_blocks], copied to *h_used if given
static int gene_ld_gene_pass(pansim_ctx *c, const pansim_gene_ld_params *p, uint32_t r2_bins, unsigned long long *h_used)
{
    auto &b = c->gl;
    acc_gene_counts_kernel<<<c->acc_words, 256, 0, c->stream>>>(c->acc[c->acc_cur], c->N, c->G, c->acc_stride_words, b.counts);
    LAUNCH_CHECK(c);
    unsigned long long *used1 = b.out + gene_ld_out_words(r2_bins) - 1;
    CU(c, cudaMemsetAsync(used1, 0, sizeof(unsigned long long), c->stream));
    GeneLdArgs a;
    a.counts = b.counts;
    a.n_genes = c->G;
    a.n_rows = c->N;
    a.min_minor = p->min_minor;
    const bool two = c->cfg.n_compartments == 2;
    a.lo1 = two ? c->cfg.comp_lo[1] : 0u;
    a.hi1 = two ? c->cfg.comp_hi[1] : 0u;
    a.block = b.block;
    a.rank = b.rank;
    a.a = b.a;
    a.grp = b.grp;
    a.inv = b.inv;
    a.used1 = used1;
    const uint32_t blocks = div_up64(c->G, VS_SITES);
    gene_ld_mark_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    vcf_scan_blocks_kernel<<<1, VS_SCAN_THREADS, 0, c->stream>>>(b.block, blocks, b.block + blocks);
    LAUNCH_CHECK(c);
    gene_ld_compact_kernel<<<blocks, VS_THREADS, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    if (h_used) CU(c, cudaMemcpyAsync(h_used, b.block + blocks, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

// presence bit rows of the used genes into gl.x (row k = rank k)
static int gene_ld_transpose(pansim_ctx *c)
{
    GeneLdTransposeArgs a;
    a.state = c->acc[c->acc_cur];
    a.stride_words = c->acc_stride_words;
    a.n_rows = c->N;
    a.n_genes = c->G;
    a.rank = c->gl.rank;
    a.kw = ld_row_words(c->N);
    a.x = c->gl.x;
    const dim3 grid(c->acc_words, div_up64(a.kw / 2, GT_WARPS));
    gene_ld_transpose_kernel<<<grid, GT_WARPS * 32, 0, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

static uint64_t gene_ld_tile_pairs(uint64_t used)
{
    const uint64_t t = (used + LD_TILE - 1) / LD_TILE;
    return t * (t + 1) / 2;
}

// zeroed class totals and histogram, then the pair kernel over every tile pair of the `used` genes
static int gene_ld_pairs(pansim_ctx *c, uint32_t r2_bins, uint64_t used)
{
    CU(c, cudaMemsetAsync(c->gl.out, 0, (GL_OUT_CLASSES + 3 * (size_t)r2_bins) * sizeof(unsigned long long), c->stream));
    if (used < 2) return 0;
    const uint64_t tiles = gene_ld_tile_pairs(used);
    if (tiles > 0x7FFFFFFFull) FAIL(c, PANSIM_ERR_INVALID, "%llu gene LD tile pairs: more than one launch holds", (unsigned long long)tiles);
    GeneLdPairArgs a;
    a.x = c->gl.x;
    a.kw = ld_row_words(c->N);
    a.k_iters = a.kw * 32 / LD_KB;
    a.a = c->gl.a;
    a.grp = c->gl.grp;
    a.inv = c->gl.inv;
    a.n_used = (uint32_t)used;
    a.n_rows = c->N;
    a.n_tiles = div_up64(used, LD_TILE);
    a.r2_bins = r2_bins;
    a.out = c->gl.out;
    const size_t smem = gene_ld_pair_smem_bytes(r2_bins);
    CU(c, cudaFuncSetAttribute(gene_ld_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gene_ld_pair_kernel<<<(uint32_t)tiles, LD_THREADS, smem, c->stream>>>(a);
    LAUNCH_CHECK(c);
    return 0;
}

// Refusals leave the context as it was.
static int gene_ld_validate(pansim_ctx *c, const pansim_gene_ld_params *p)
{
    if (!p->r2_bins || p->r2_bins > GL_MAX_BINS || !p->min_minor)
        FAIL(c, PANSIM_ERR_INVALID, "gene LD: r2_bins must be 1..%u and min_minor >= 1", GL_MAX_BINS);
    if (!c->has_acc) FAIL(c, PANSIM_ERR_STATE, "gene LD: no accessory state: call pansim_set_initial or pansim_upload_acc first");
    return 0;
}

// the gene pass, the transpose and the pair pass into the pinned outputs (G >= 1, N >= 2); *used = the used genes
static int gene_ld_run(pansim_ctx *c, const pansim_gene_ld_params *p, uint64_t *used)
{
    CU(c, cudaSetDevice(c->cfg.device));
    if (int rc = gene_ld_ensure(c, p->r2_bins)) return rc;
    const size_t words = gene_ld_out_words(p->r2_bins);
    unsigned long long *h_used = c->gl.h_out + words - 1;                      // overwritten by the readback below
    if (int rc = gene_ld_gene_pass(c, p, p->r2_bins, h_used)) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    *used = *h_used;
    if (*used >= 2) {
        if (int rc = gene_ld_ensure_x(c, *used)) return rc;
        if (int rc = gene_ld_transpose(c)) return rc;
    }
    if (int rc = gene_ld_pairs(c, p->r2_bins, *used)) return rc;
    CU(c, cudaMemcpyAsync(c->gl.h_out, c->gl.out, words * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int pansim_gene_ld(pansim_ctx *c, const pansim_gene_ld_params *p, pansim_gene_ld_class classes[3], uint64_t *hist, uint64_t genes_used[2])
{
    if (!c || !p || !classes) return PANSIM_ERR_INVALID;
    if (int rc = gene_ld_validate(c, p)) return rc;
    memset(classes, 0, 3 * sizeof(pansim_gene_ld_class));
    if (hist) memset(hist, 0, 3 * (size_t)p->r2_bins * sizeof(uint64_t));
    uint64_t used = 0, used1 = 0;
    if (c->G && c->N >= 2) {                                                     // otherwise no gene is used
        if (int rc = gene_ld_run(c, p, &used)) return rc;
        const unsigned long long *h = c->gl.h_out;
        for (int k = 0; k < 3; k++) {
            const unsigned long long *w = h + GL_CLASS_WORDS * k;
            classes[k].ld = {w[0], w[1], w[2], w[3]};
            classes[k].associated = w[4];
            classes[k].dissociated = w[5];
        }
        if (hist)
            for (size_t b = 0; b < 3 * (size_t)p->r2_bins; b++) hist[b] = h[GL_OUT_CLASSES + b];
        used1 = h[gene_ld_out_words(p->r2_bins) - 1];
    }
    if (genes_used) {
        genes_used[0] = used - used1;
        genes_used[1] = used1;
    }
    return 0;
}

int pansim_gene_ld_kernel_ms(pansim_ctx *c, const pansim_gene_ld_params *p, uint32_t repeats, float *gene_ms, float *transpose_ms,
                             float *pair_ms, uint64_t *pairs)
{
    if (!c || !p || !repeats) return PANSIM_ERR_INVALID;
    pansim_gene_ld_class cls[3];
    uint64_t gu[2];
    if (int rc = pansim_gene_ld(c, p, cls, nullptr, gu)) return rc;           // also the warm-up
    const uint64_t used = gu[0] + gu[1];
    float t[3] = {0.f, 0.f, 0.f};
    if (c->G && c->N >= 2) {
        cudaEvent_t ev[4];
        for (auto &e : ev) CU(c, cudaEventCreate(&e));
        int rc = 0;
        cudaEventRecord(ev[0], c->stream);
        for (uint32_t r = 0; r < repeats && !rc; r++) rc = gene_ld_gene_pass(c, p, p->r2_bins, nullptr);
        cudaEventRecord(ev[1], c->stream);
        for (uint32_t r = 0; r < repeats && !rc && used >= 2; r++) rc = gene_ld_transpose(c);
        cudaEventRecord(ev[2], c->stream);
        for (uint32_t r = 0; r < repeats && !rc; r++) rc = gene_ld_pairs(c, p->r2_bins, used);
        cudaEventRecord(ev[3], c->stream);
        const cudaError_t e = cudaEventSynchronize(ev[3]);
        for (int k = 0; k < 3; k++) cudaEventElapsedTime(&t[k], ev[k], ev[k + 1]);
        for (auto &x : ev) cudaEventDestroy(x);
        if (rc) return rc;
        if (e != cudaSuccess) FAIL(c, PANSIM_ERR_CUDA, "gene LD kernels failed: %s", cudaGetErrorString(e));
    }
    if (gene_ms) *gene_ms = t[0] / (float)repeats;
    if (transpose_ms) *transpose_ms = t[1] / (float)repeats;
    if (pair_ms) *pair_ms = t[2] / (float)repeats;
    if (pairs) *pairs = cls[0].ld.pairs + cls[1].ld.pairs + cls[2].ld.pairs;
    return 0;
}

// ---- pangenome accumulation and gene frequency spectrum (pangenome.cuh, DESIGN.md section 16) ------------------
static_assert(PG_ORDER_TAG == PANSIM_GENE_ACC_ORDER_TAG, "the order draw's counter word is documented in the header");
static_assert(PANSIM_GENE_ACC_MAX_PERMS <= 65535u, "orders are grid.z of the walk");
// Chunks of the N steps of an order: one, unless the word slices x orders leave resident walk CTAs unused; then as
// many as fill at most one wave of them (a partial second wave would run at a fraction of the SMs), each chunk at
// least 256 steps and a whole number of batches.
static void gene_acc_plan(const pansim_ctx *c, uint32_t P, uint32_t *chunk_rows, uint32_t *n_chunks)
{
    const uint64_t base = (uint64_t)div_up64(c->acc_words, PG_SLICE_WORDS) * P, slots = (uint64_t)std::max(1, c->ga.walk_slots);
    uint64_t chunks = 1;
    if (base && base < slots) chunks = std::max<uint64_t>(1, std::min<uint64_t>(slots / base, c->N / 256));
    *chunk_rows = div_up64(div_up64(c->N, chunks), PG_BATCH) * PG_BATCH;
    *n_chunks = div_up64(c->N, *chunk_rows);
}

// orders, deltas and curves for P orders (kept with the context, grown when P grows) and the chunk summaries
static int gene_acc_ensure(pansim_ctx *c, uint32_t P, uint32_t n_chunks)
{
    auto &b = c->ga;
    if (P > b.perm_cap) {
        for (uint32_t **q : {&b.orders, &b.delta, &b.curves})
            if (*q) { cudaFree(*q); *q = nullptr; }
        b.perm_cap = 0;
        const size_t pn = (size_t)P * c->N * sizeof(uint32_t);
        if (cudaMalloc(&b.orders, pn) != cudaSuccess || cudaMalloc(&b.delta, pn * PG_STATS) != cudaSuccess ||
            cudaMalloc(&b.curves, pn * 4) != cudaSuccess) {
            cudaGetLastError();
            FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (gene accumulation, %u orders) failed", pn * 8, P);
        }
        b.perm_cap = P;
    }
    const size_t words = n_chunks > 1 ? (size_t)P * n_chunks * 3 * c->acc_words : 0;
    if (words > b.summary_cap) {
        if (b.summary) cudaFree(b.summary);
        b.summary = nullptr; b.summary_cap = 0;
        if (cudaMalloc(&b.summary, words * sizeof(uint32_t)) != cudaSuccess) {
            cudaGetLastError();
            FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc of %zu bytes (gene accumulation chunk summaries) failed", words * 4);
        }
        b.summary_cap = words;
    }
    return 0;
}

// P orders into ga.orders; the swap indices go to shared memory when 8 N bytes fit, else to ga.delta
static int gene_acc_orders(pansim_ctx *c, uint64_t seed, uint32_t P)
{
    PgOrderArgs a;
    a.rk = philox_key_schedule(make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    a.n_rows = c->N;
    a.orders = c->ga.orders;
    a.scratch = c->ga.delta;
    const size_t smem = 2 * (size_t)c->N * sizeof(uint32_t);
    if (smem <= (size_t)c->ga.order_smem_max) {
        pg_order_kernel<true><<<P, PG_ORDER_THREADS, smem, c->stream>>>(a);
    } else {
        pg_order_kernel<false><<<P, PG_ORDER_THREADS, 0, c->stream>>>(a);
    }
    LAUNCH_CHECK(c);
    return 0;
}

// the walk over the orders in ga.orders (zeroed deltas, chunk summaries, walk) and the curves
static int gene_acc_accumulate(pansim_ctx *c, uint32_t P, uint32_t chunk_rows, uint32_t n_chunks)
{
    auto &b = c->ga;
    const size_t pn = (size_t)P * c->N;
    CU(c, cudaMemsetAsync(b.delta, 0, pn * PG_STATS * sizeof(uint32_t), c->stream));
    if (c->G) {
        PgWalkArgs a;
        a.state = c->acc[c->acc_cur];
        a.stride_words = c->acc_stride_words;
        a.n_words = c->acc_words;
        a.n_genes = c->G;
        a.n_rows = c->N;
        a.orders = b.orders;
        a.chunk_rows = chunk_rows;
        a.n_chunks = n_chunks;
        a.summary = b.summary;
        a.delta = b.delta;
        const uint32_t slices = div_up64(c->acc_words, PG_SLICE_WORDS);
        if (n_chunks > 1) {
            pg_summary_kernel<<<dim3(slices, n_chunks - 1, P), PG_SLICE_WORDS, 0, c->stream>>>(a);
            LAUNCH_CHECK(c);
        }
        pg_walk_kernel<<<dim3(slices, n_chunks, P), PG_SLICE_WORDS, 0, c->stream>>>(a);
        LAUNCH_CHECK(c);
    }
    PgCurveArgs q;
    q.delta = b.delta;
    q.n_rows = c->N;
    q.c0 = c->cfg.core_genes;
    q.pan = b.curves;
    q.core = b.curves + pn;
    q.new_genes = b.curves + 2 * pn;
    q.unique = b.curves + 3 * pn;
    pg_curves_kernel<<<P, PG_SCAN_THREADS, 0, c->stream>>>(q);
    LAUNCH_CHECK(c);
    return 0;
}

// Refusals leave the context as it was.
static int gene_acc_prepare(pansim_ctx *c, uint32_t n_perms, uint32_t *chunk_rows, uint32_t *n_chunks)
{
    if (!n_perms || n_perms > PANSIM_GENE_ACC_MAX_PERMS)
        FAIL(c, PANSIM_ERR_INVALID, "gene accumulation: n_perms must be 1..%u", PANSIM_GENE_ACC_MAX_PERMS);
    if (!c->has_acc) FAIL(c, PANSIM_ERR_STATE, "gene accumulation: no accessory state: call pansim_set_initial or pansim_upload_acc first");
    CU(c, cudaSetDevice(c->cfg.device));
    if (!c->ga.walk_slots) {       // device limits of the launches, once per context
        int per_sm = 0;
        CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pg_walk_kernel, PG_SLICE_WORDS, 0));
        CU(c, cudaDeviceGetAttribute(&c->ga.order_smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->cfg.device));
        CU(c, cudaFuncSetAttribute(pg_order_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, c->ga.order_smem_max));
        c->ga.walk_slots = std::max(1, per_sm) * std::max(1, c->sm_count);
    }
    gene_acc_plan(c, n_perms, chunk_rows, n_chunks);
    return gene_acc_ensure(c, n_perms, *n_chunks);
}

int pansim_gene_accumulation(pansim_ctx *c, uint64_t seed, uint32_t n_perms, uint32_t *orders, uint32_t *pan, uint32_t *core,
                             uint32_t *new_genes, uint32_t *unique)
{
    if (!c) return PANSIM_ERR_INVALID;
    uint32_t chunk_rows = 0, n_chunks = 0;
    if (int rc = gene_acc_prepare(c, n_perms, &chunk_rows, &n_chunks)) return rc;
    if (int rc = gene_acc_orders(c, seed, n_perms)) return rc;
    if (int rc = gene_acc_accumulate(c, n_perms, chunk_rows, n_chunks)) return rc;
    const size_t pn = (size_t)n_perms * c->N;
    if (orders) CU(c, cudaMemcpyAsync(orders, c->ga.orders, pn * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    uint32_t *out[4] = {pan, core, new_genes, unique};
    for (int k = 0; k < 4; k++)
        if (out[k]) CU(c, cudaMemcpyAsync(out[k], c->ga.curves + k * pn, pn * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int pansim_gene_accumulation_kernel_ms(pansim_ctx *c, uint64_t seed, uint32_t n_perms, uint32_t repeats, float *order_ms,
                                       float *accum_ms, uint64_t *bytes_read)
{
    if (!c || !repeats) return PANSIM_ERR_INVALID;
    if (int rc = pansim_gene_accumulation(c, seed, n_perms, nullptr, nullptr, nullptr, nullptr, nullptr)) return rc;   // also the warm-up
    uint32_t chunk_rows = 0, n_chunks = 0;
    gene_acc_plan(c, n_perms, &chunk_rows, &n_chunks);
    cudaEvent_t ev[3];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    int rc = 0;
    cudaEventRecord(ev[0], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++) rc = gene_acc_orders(c, seed, n_perms);
    cudaEventRecord(ev[1], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++) rc = gene_acc_accumulate(c, n_perms, chunk_rows, n_chunks);
    cudaEventRecord(ev[2], c->stream);
    const cudaError_t e = cudaEventSynchronize(ev[2]);
    float t[2] = {0.f, 0.f};
    for (int k = 0; k < 2; k++) cudaEventElapsedTime(&t[k], ev[k], ev[k + 1]);
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (e != cudaSuccess) FAIL(c, PANSIM_ERR_CUDA, "gene accumulation kernels failed: %s", cudaGetErrorString(e));
    if (order_ms) *order_ms = t[0] / (float)repeats;
    if (accum_ms) *accum_ms = t[1] / (float)repeats;
    if (bytes_read) *bytes_read = (uint64_t)n_perms * c->N * c->acc_words * sizeof(uint32_t);
    return 0;
}

int pansim_gene_spectrum(pansim_ctx *c, uint64_t *spectrum)
{
    if (!c || !spectrum) return PANSIM_ERR_INVALID;
    if (!c->has_acc) FAIL(c, PANSIM_ERR_STATE, "gene spectrum: no accessory state: call pansim_set_initial or pansim_upload_acc first");
    CU(c, cudaSetDevice(c->cfg.device));
    const size_t bytes = ((size_t)c->N + 1) * sizeof(unsigned long long);
    if (!c->ga.spectrum) CU(c, cudaMalloc(&c->ga.spectrum, bytes));
    CU(c, cudaMemsetAsync(c->ga.spectrum, 0, bytes, c->stream));
    if (c->G) {
        acc_gene_counts_kernel<<<c->acc_words, 256, 0, c->stream>>>(c->acc[c->acc_cur], c->N, c->G, c->acc_stride_words, c->d_gain_thr);
        LAUNCH_CHECK(c);
        pg_spectrum_kernel<<<div_up64(c->G, 256), 256, 0, c->stream>>>(c->d_gain_thr, c->G, c->ga.spectrum);
        LAUNCH_CHECK(c);
    }
    CU(c, cudaMemcpyAsync(spectrum, c->ga.spectrum, bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    spectrum[c->N] += c->cfg.core_genes;
    return 0;
}

void pansim_pangenome_classes(const uint64_t *spectrum, uint32_t pop_size, uint64_t out[5])
{
    if (!out) return;
    for (int k = 0; k < 5; k++) out[k] = 0;
    if (!spectrum) return;
    const uint64_t n = pop_size;
    for (uint64_t a = 1; a <= n; a++) {
        const uint64_t h = 100 * a;
        out[h >= 99 * n ? 0 : h >= 95 * n ? 1 : h >= 15 * n ? 2 : 3] += spectrum[a];
    }
    out[4] = out[0] + out[1] + out[2] + out[3];
}

// ---- parsimony on a node table (parsimony.cuh, DESIGN.md section 17) ---------
// Default scratch budget of one call: the smaller of 16 GiB and half the free device memory.
// PANSIM_PARSIMONY_SCRATCH_MB=<n> replaces it (a small value forces many slabs; the results are the same).
constexpr uint64_t PS_BUDGET_CAP_MB = 16384;

// The rules of the node table (include/pansim_b200.h), checked on the host: an empty string, or what is wrong. With
// csr, on success csr = child_off[n_internal + 1] followed by child[n_nodes - 1]: the children of each internal node
// in ascending id.
static std::string node_table_error(const uint32_t *parent, uint32_t n_nodes, uint32_t N, std::vector<uint32_t> *csr)
{
    char b[160];
    if (!parent) return "null node table";
    if (n_nodes < N || (uint64_t)n_nodes > 2ull * N - 1) {
        snprintf(b, sizeof b, "%u nodes for %u leaves (a tree has N .. 2N - 1)", n_nodes, N);
        return b;
    }
    const uint32_t root = n_nodes - 1, n_int = n_nodes - N;
    if (parent[root] != GEN_NONE) {
        snprintf(b, sizeof b, "the last node (%u) must be the root, parent 0xFFFFFFFF", root);
        return b;
    }
    std::vector<uint32_t> local;
    std::vector<uint32_t> &off = csr ? *csr : local;
    off.assign((size_t)n_int + 1 + (csr ? root : 0), 0);
    for (uint32_t k = 0; k < root; k++) {
        const uint32_t p = parent[k];
        if (p <= k || p < N || p >= n_nodes) {
            snprintf(b, sizeof b, "node %u has parent %u (an internal node with a larger id)", k, p);
            return b;
        }
        off[p - N + 1]++;
    }
    for (uint32_t v = 0; v < n_int; v++)
        if (off[v + 1] < 2) {
            snprintf(b, sizeof b, "internal node %u has %u children (at least 2)", N + v, off[v + 1]);
            return b;
        }
    if (!csr) return "";
    for (uint32_t v = 0; v < n_int; v++) off[v + 1] += off[v];
    std::vector<uint32_t> fill(off.begin(), off.begin() + n_int);
    uint32_t *child = off.data() + n_int + 1;
    for (uint32_t k = 0; k < root; k++) child[fill[parent[k] - N]++] = k;
    return "";
}

static int parsimony_tree(pansim_ctx *c, const uint32_t *parent, uint32_t n_nodes, std::vector<uint32_t> &csr)
{
    const std::string e = node_table_error(parent, n_nodes, c->N, &csr);
    if (!e.empty()) FAIL(c, PANSIM_ERR_INVALID, "parsimony: %s", e.c_str());
    return 0;
}

// the device buffers of one call, freed when it returns
struct ParsimonyCall {
    uint32_t *tree = nullptr, *scores = nullptr;
    unsigned long long *out = nullptr;       // summary [5], then the branch arrays [NB][n_nodes]
    void *scratch = nullptr;
    uint32_t cols_slab = 0, n_nodes = 0, nb = 1;
    uint64_t n_chars = 0, n_cols = 0;
    size_t smem = 0;
    bool genes = false;
    ParsimonyArgs a{};
    ~ParsimonyCall()
    {
        for (void *p : {(void *)tree, (void *)scores, (void *)out, scratch})
            if (p) cudaFree(p);
    }
};

static uint64_t parsimony_budget()
{
    if (const char *e = std::getenv("PANSIM_PARSIMONY_SCRATCH_MB"))
        if (const uint64_t mb = std::strtoull(e, nullptr, 10)) return mb << 20;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = 0; }
    return std::min<uint64_t>(PS_BUDGET_CAP_MB << 20, free_b / 2);
}

// Checks, the per-character counts, the buffers and the uploaded table; refusals leave the context as it was.
static int parsimony_prepare(pansim_ctx *c, bool genes, const uint32_t *parent, uint32_t n_nodes, ParsimonyCall &w)
{
    if (int rc = require_state(c)) return rc;
    std::vector<uint32_t> csr;
    if (int rc = parsimony_tree(c, parent, n_nodes, csr)) return rc;
    CU(c, cudaSetDevice(c->cfg.device));
    const uint32_t N = c->N, n_int = n_nodes - N, ns = genes ? 2 : 4;
    w.genes = genes;
    w.n_nodes = n_nodes;
    w.nb = genes ? 2 : 1;
    w.n_chars = genes ? c->G : c->Ll;
    w.n_cols = (w.n_chars + 31) / 32;
    const uint64_t pad_cols = (w.n_cols + PS_THREADS - 1) / PS_THREADS * PS_THREADS;
    uint64_t cols = n_int ? parsimony_budget() / ((uint64_t)n_int * ns * 4) : pad_cols;
    cols = std::min(pad_cols, std::max<uint64_t>(PS_THREADS, cols / PS_THREADS * PS_THREADS));
    w.cols_slab = (uint32_t)std::min<uint64_t>(cols, 0x7FFFFF80ull);
    const size_t out_words = 5 + (size_t)w.nb * n_nodes;
    auto alloc = [&](void **p, size_t bytes, const char *what) -> int {
        if (cudaMalloc(p, bytes) != cudaSuccess) {
            cudaGetLastError();
            *p = nullptr;
            FAIL(c, PANSIM_ERR_NOMEM, "parsimony: cudaMalloc of %zu bytes (%s) failed", bytes, what);
        }
        return 0;
    };
    if (int rc = alloc((void **)&w.tree, csr.size() * 4, "node table")) return rc;
    if (int rc = alloc((void **)&w.out, out_words * 8, "results")) return rc;
    if (int rc = alloc((void **)&w.scores, std::max<uint64_t>(w.n_chars, 1) * 4, "character scores")) return rc;
    if (n_int && w.n_cols)
        if (int rc = alloc(&w.scratch, (size_t)n_int * w.cols_slab * ns * 4, "scratch")) return rc;
    CU(c, cudaMemcpyAsync(w.tree, csr.data(), csr.size() * 4, cudaMemcpyHostToDevice, c->stream));
    const uint32_t *rows = nullptr;
    uint64_t row_words = 0;
    if (!genes) {
        if (c->Ll) {
            if (int rc = ensure_div(c, 1, false)) return rc;
            if (int rc = ensure_site_counts(c)) return rc;
            c->ps = c->stream;
            if (int rc = core_materialize(c, c->stream)) return rc;
            CU(c, cudaMemsetAsync(c->d_div, 0, 4 * sizeof(unsigned long long), c->stream));
            if (int rc = launch_diversity(c, c->stream, c->d_div, c->d_vcf_counts, nullptr)) return rc;
        }
        rows = reinterpret_cast<const uint32_t *>(c->core[c->core_cur]);
        row_words = c->core_stride / 4;
    } else {
        if (c->G) {
            acc_gene_counts_kernel<<<c->acc_words, 256, 0, c->stream>>>(c->acc[c->acc_cur], c->N, c->G, c->acc_stride_words, c->d_gain_thr);
            LAUNCH_CHECK(c);
        }
        rows = c->acc[c->acc_cur];
        row_words = c->acc_stride_words;
    }
    ParsimonyArgs &a = w.a;
    a.rows = rows;
    a.row_words = row_words;
    a.n_leaves = N;
    a.n_internal = n_int;
    a.child_off = w.tree;
    a.child = w.tree + n_int + 1;
    a.col0 = 0;
    a.cols_pad = w.cols_slab;
    a.n_cols = w.n_cols;
    a.n_chars = w.n_chars;
    a.dmax = 32u - (uint32_t)__builtin_clz(N);
    a.scratch = w.scratch;
    a.site_counts = c->d_vcf_counts;
    a.gene_counts = c->d_gain_thr;
    a.scores = w.scores;
    a.summary = w.out;
    a.branch0 = w.out + 5;
    a.branch1 = w.out + 5 + (genes ? n_nodes : 0);
    w.smem = (size_t)ns * a.dmax * PS_THREADS * 4;
    if (w.smem > 48 * 1024) {
        const cudaError_t e = genes ? cudaFuncSetAttribute(parsimony_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w.smem)
                                    : cudaFuncSetAttribute(parsimony_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w.smem);
        CU(c, e);
    }
    return 0;
}

// zeroed results, then the slabs of columns one after the other on c->stream
static int parsimony_launch(pansim_ctx *c, ParsimonyCall &w)
{
    CU(c, cudaMemsetAsync(w.out, 0, (5 + (size_t)w.nb * w.n_nodes) * 8, c->stream));
    for (uint64_t col0 = 0; col0 < w.n_cols; col0 += w.cols_slab) {
        ParsimonyArgs a = w.a;
        a.col0 = col0;
        const uint64_t cols = std::min<uint64_t>(w.cols_slab, w.n_cols - col0);
        const uint32_t grid = div_up64(cols, PS_THREADS);
        if (w.genes)
            parsimony_kernel<2><<<grid, PS_THREADS, w.smem, c->stream>>>(a);
        else
            parsimony_kernel<4><<<grid, PS_THREADS, w.smem, c->stream>>>(a);
        LAUNCH_CHECK(c);
    }
    return 0;
}

static int parsimony_call(pansim_ctx *c, bool genes, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out,
                          uint32_t *chars, uint64_t *branch0, uint64_t *branch1)
{
    if (!c) return PANSIM_ERR_INVALID;
    ParsimonyCall w;
    if (int rc = parsimony_prepare(c, genes, parent, n_nodes, w)) return rc;
    if (int rc = parsimony_launch(c, w)) return rc;
    unsigned long long sum[5];
    CU(c, cudaMemcpyAsync(sum, w.out, sizeof sum, cudaMemcpyDeviceToHost, c->stream));
    if (chars && w.n_chars) CU(c, cudaMemcpyAsync(chars, w.scores, w.n_chars * 4, cudaMemcpyDeviceToHost, c->stream));
    if (branch0) CU(c, cudaMemcpyAsync(branch0, w.a.branch0, (size_t)n_nodes * 8, cudaMemcpyDeviceToHost, c->stream));
    if (branch1) CU(c, cudaMemcpyAsync(branch1, w.a.branch1, (size_t)n_nodes * 8, cudaMemcpyDeviceToHost, c->stream));
    if (int rc = check_device_flag(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG)) return rc;
    if (out) *out = {w.n_chars, sum[0], sum[1], sum[2], sum[3], sum[4]};
    return 0;
}

int pansim_core_parsimony(pansim_ctx *c, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out, uint32_t *site_changes,
                          uint64_t *branch_changes)
{
    return parsimony_call(c, false, parent, n_nodes, out, site_changes, branch_changes, nullptr);
}

int pansim_gene_parsimony(pansim_ctx *c, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out, uint32_t *gene_changes,
                          uint64_t *gains, uint64_t *losses)
{
    return parsimony_call(c, true, parent, n_nodes, out, gene_changes, gains, losses);
}

int pansim_parsimony_kernel_ms(pansim_ctx *c, const uint32_t *parent, uint32_t n_nodes, int genes, uint32_t repeats, float *ms,
                               uint64_t *bytes_read, uint32_t *slabs)
{
    if (!c || !repeats) return PANSIM_ERR_INVALID;
    ParsimonyCall w;
    if (int rc = parsimony_prepare(c, genes != 0, parent, n_nodes, w)) return rc;
    if (int rc = parsimony_launch(c, w)) return rc;      // warm-up
    cudaEvent_t ev[2];
    for (auto &e : ev) CU(c, cudaEventCreate(&e));
    int rc = 0;
    cudaEventRecord(ev[0], c->stream);
    for (uint32_t r = 0; r < repeats && !rc; r++) rc = parsimony_launch(c, w);
    cudaEventRecord(ev[1], c->stream);
    const cudaError_t e = cudaEventSynchronize(ev[1]);
    float t = 0.f;
    cudaEventElapsedTime(&t, ev[0], ev[1]);
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (e != cudaSuccess) FAIL(c, PANSIM_ERR_CUDA, "parsimony kernel failed: %s", cudaGetErrorString(e));
    if (ms) *ms = t / (float)repeats;
    // per column: every leaf read twice (8 / 4 bytes), every non-root internal set read twice (as a child going up,
    // then as a child going down), the root's set and every internal node's assigned state read once (16 / 8 bytes)
    const uint64_t leaf_b = genes ? 4 : 8, set_b = genes ? 8 : 16, n_int = n_nodes - c->N;
    if (bytes_read) *bytes_read = w.n_cols * (2 * (uint64_t)c->N * leaf_b + (n_int ? 3 * n_int - 1 : 0) * set_b);
    if (slabs) *slabs = (uint32_t)((w.n_cols + w.cols_slab - 1) / w.cols_slab);
    return 0;
}

void pansim_parsimony_indices(const pansim_parsimony *p, double *ci, double *ri)
{
    const double nan = std::numeric_limits<double>::quiet_NaN();
    if (!p) return;
    const double S = (double)p->tree_length, M = (double)p->min_changes, G = (double)p->max_changes;
    if (ci) *ci = p->tree_length ? M / S : nan;
    if (ri) *ri = p->max_changes != p->min_changes ? (G - S) / (G - M) : nan;
}

// ---- neighbour-joining (nj.cuh, DESIGN.md section 18) ------------------------------------------
// Pairs per row block of the matrix build (the context's pair buffers hold one block).
constexpr uint64_t NJ_BLOCK_PAIRS = 1ull << 26;
// A compaction repacks the active rows when k <= NJ_COMPACT_FRACTION x the stored dimension, and only while that
// dimension is above NJ_COMPACT_MIN (below it the scan is bound by latency, not bytes). PANSIM_NJ_COMPACT=<f> (0 < f
// < 1) replaces the fraction for measurements; the tree is the same for every schedule.
constexpr double NJ_COMPACT_FRACTION = 0.9;
constexpr uint32_t NJ_COMPACT_MIN = 512;

static uint32_t nj_nodes(uint32_t n) { return n >= 3 ? 2 * n - 2 : n == 2 ? 3 : 1; }
static uint64_t nj_pitch(uint64_t m) { return (m + 31) / 32 * 32; }

// the k at which the loop compacts, largest first
static std::vector<uint32_t> nj_schedule(uint32_t n)
{
    double f = NJ_COMPACT_FRACTION;
    if (const char *e = std::getenv("PANSIM_NJ_COMPACT")) {
        const double v = std::strtod(e, nullptr);
        if (v > 0.0 && v < 1.0) f = v;
    }
    std::vector<uint32_t> ks;
    uint32_t M = n;
    for (uint32_t k = n; k > 3; k--)
        if (M > NJ_COMPACT_MIN && (double)k <= f * (double)M) { ks.push_back(k); M = k; }
    return ks;
}

// the device buffers of one call, freed when it returns
struct NjCall {
    uint32_t n = 0;
    double *D[2] = {nullptr, nullptr};
    void *scratch = nullptr;
    double *R[2] = {nullptr, nullptr}, *length = nullptr;
    uint32_t *node[2] = {nullptr, nullptr}, *old_of = nullptr, *parent = nullptr, *done = nullptr;
    NjBest *part = nullptr, *best = nullptr;
    uint32_t max_grid = 0;
    std::vector<uint32_t> compact_at;
    ~NjCall()
    {
        for (void *p : {(void *)D[0], (void *)D[1], scratch})
            if (p) cudaFree(p);
    }
};

static int nj_alloc(pansim_ctx *c, uint32_t n, NjCall &w)
{
    CU(c, cudaSetDevice(c->cfg.device));
    w.n = n;
    w.compact_at = nj_schedule(n);
    w.max_grid = (uint32_t)c->sm_count * 8;
    const uint64_t k1 = w.compact_at.empty() ? 0 : w.compact_at[0];
    const size_t bytes[2] = {(size_t)n * nj_pitch(n) * 8, (size_t)k1 * nj_pitch(k1) * 8};
    const size_t scratch = (size_t)n * (2 * 8 + 2 * 4 + 4) + (size_t)nj_nodes(n) * 12 + ((size_t)w.max_grid + 1) * sizeof(NjBest) + 10 * 16;   // + the rounding of ten pieces
    for (int i = 0; i < 2; i++)
        if (bytes[i] && cudaMalloc(&w.D[i], bytes[i]) != cudaSuccess) {
            cudaGetLastError();
            w.D[i] = nullptr;
            FAIL(c, PANSIM_ERR_NOMEM, "neighbour-joining: cudaMalloc of the %u x %u distance matrix (%zu bytes) failed", n, n, bytes[i]);
        }
    if (cudaMalloc(&w.scratch, scratch) != cudaSuccess) {
        cudaGetLastError();
        w.scratch = nullptr;
        FAIL(c, PANSIM_ERR_NOMEM, "neighbour-joining: cudaMalloc of %zu bytes of scratch failed", scratch);
    }
    char *p = (char *)w.scratch;
    auto take = [&](size_t b) { char *q = p; p += (b + 15) / 16 * 16; return q; };
    w.best = (NjBest *)take(sizeof(NjBest));
    w.part = (NjBest *)take((size_t)w.max_grid * sizeof(NjBest));
    w.R[0] = (double *)take((size_t)n * 8);
    w.R[1] = (double *)take((size_t)n * 8);
    w.length = (double *)take((size_t)nj_nodes(n) * 8);
    w.node[0] = (uint32_t *)take((size_t)n * 4);
    w.node[1] = (uint32_t *)take((size_t)n * 4);
    w.old_of = (uint32_t *)take((size_t)n * 4);
    w.parent = (uint32_t *)take((size_t)nj_nodes(n) * 4);
    w.done = (uint32_t *)take(4);
    CU(c, cudaMemsetAsync(w.done, 0, 4, c->stream));
    CU(c, cudaMemsetAsync(w.D[0], 0, bytes[0], c->stream));
    return 0;
}

// D[0] is filled: R, the joins, the last two or three, and the table back to the host. Times the join loop between
// ev[0] and ev[1] when ev is given; *scanned / *compactions as pansim_nj_kernel_ms reports them.
static int nj_join_loop(pansim_ctx *c, NjCall &w, uint32_t *parent, double *length, cudaEvent_t *ev, uint64_t *scanned,
                        uint32_t *compactions)
{
    const uint32_t n = w.n;
    int cur = 0;
    uint32_t M = n;
    uint64_t pitch = nj_pitch(n);
    nj_rowsum_kernel<<<div_up64(n, 256), 256, 0, c->stream>>>(w.D[0], pitch, n, w.R[0], w.node[0]);
    LAUNCH_CHECK(c);
    if (ev) CU(c, cudaEventRecord(ev[0], c->stream));
    uint64_t bytes = 0;
    size_t next = 0;
    for (uint32_t k = n; k > 3; k--) {
        if (next < w.compact_at.size() && w.compact_at[next] == k) {
            const uint64_t np = nj_pitch(k);
            nj_compact_index_kernel<<<1, 1024, 0, c->stream>>>(w.R[cur], w.node[cur], M, w.old_of, w.R[cur ^ 1], w.node[cur ^ 1]);
            LAUNCH_CHECK(c);
            nj_compact_copy_kernel<<<std::min<uint32_t>(k, w.max_grid), 256, 0, c->stream>>>(w.D[cur], pitch, w.D[cur ^ 1], np, w.old_of, k);
            LAUNCH_CHECK(c);
            cur ^= 1;
            M = k;
            pitch = np;
            next++;
        }
        const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up64(M - 1, NJ_THREADS / 32), w.max_grid));
        nj_scan_kernel<<<grid, NJ_THREADS, 0, c->stream>>>(w.D[cur], pitch, M, (double)(k - 2), w.R[cur], w.part, w.done, w.best);
        LAUNCH_CHECK(c);
        nj_join_kernel<<<div_up64(M, NJ_THREADS), NJ_THREADS, 0, c->stream>>>(w.D[cur], pitch, M, w.R[cur], w.node[cur], w.best, k, n,
                                                                              w.parent, w.length);
        LAUNCH_CHECK(c);
        bytes += (uint64_t)M * (M - 1) / 2 * 8;
    }
    if (n >= 2) {
        nj_finish_kernel<<<1, 1, 0, c->stream>>>(w.D[cur], pitch, M, w.R[cur], w.node[cur], n, w.parent, w.length);
        LAUNCH_CHECK(c);
    }
    if (ev) CU(c, cudaEventRecord(ev[1], c->stream));
    const size_t nn = nj_nodes(n);
    CU(c, cudaMemcpyAsync(parent, w.parent, nn * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(length, w.length, nn * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (scanned) *scanned = bytes;
    if (compactions) *compactions = (uint32_t)w.compact_at.size();
    return 0;
}

// the distances of the pairs of the current block (c->d_r1 / d_r2 and the counts) into D[0]
static int nj_scatter(pansim_ctx *c, NjCall &w, int metric, size_t P)
{
    if (!P) return 0;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(div_up64(P, 256), (uint64_t)c->sm_count * 16);
    nj_scatter_pairs_kernel<<<grid, 256, 0, c->stream>>>(c->d_r1, c->d_r2, c->d_cd, c->d_in, c->d_un, (uint32_t)P, metric,
                                                        (double)c->L, (double)c->cfg.core_genes, w.D[0], nj_pitch(w.n));
    LAUNCH_CHECK(c);
    return 0;
}

// row blocks [i0, i1) of at most NJ_BLOCK_PAIRS pairs over rows 0 .. n-2
static std::vector<std::pair<uint32_t, uint32_t>> nj_blocks(uint32_t n, uint64_t *max_pairs)
{
    std::vector<std::pair<uint32_t, uint32_t>> out;
    *max_pairs = 0;
    uint32_t i0 = 0;
    while (i0 + 1 < n) {
        uint64_t P = 0;
        uint32_t i1 = i0;
        while (i1 + 1 < n && (i1 == i0 || P + (n - 1 - i1) <= NJ_BLOCK_PAIRS)) P += n - 1 - i1++;
        out.push_back({i0, i1});
        *max_pairs = std::max(*max_pairs, P);
        i0 = i1;
    }
    return out;
}

// The refusals of pansim_nj_tree; shard = false skips the column-shard check (a group sums its shards itself).
static int nj_check(pansim_ctx *c, int metric, bool shard)
{
    if (metric != 0 && metric != 1) FAIL(c, PANSIM_ERR_INVALID, "neighbour-joining: metric %d (0 core, 1 acc)", metric);
    if (int rc = require_state(c)) return rc;
    if (metric == 0 && c->L == 0) FAIL(c, PANSIM_ERR_INVALID, "neighbour-joining: core distances need core_size > 0");
    if (metric == 0 && shard)
        if (int rc = require_whole_alignment(c, "neighbour-joining on core distances")) return rc;
    return 0;
}

// One context's matrix: per row block, the pair counts (summed over the communicator for core) and the scatter.
static int nj_build_ctx(pansim_ctx *c, int metric, NjCall &w)
{
    uint64_t maxP = 0;
    const auto blocks = nj_blocks(w.n, &maxP);
    if (maxP)
        if (int rc = ensure_pairs(c, (size_t)maxP)) return rc;
    for (const auto &b : blocks) {
        size_t P = 0;
        if (int rc = pair_counts_rows_impl(c, b.first, b.second, metric == 0 ? c->d_cd : nullptr, metric ? c->d_in : nullptr,
                                           metric ? c->d_un : nullptr, &P)) return rc;
        if (metric == 0)
            if (int rc = comm_allreduce_counts(c, c->d_cd, P)) return rc;
        if (int rc = nj_scatter(c, w, metric, P)) return rc;
    }
    return 0;
}

static void nj_single_leaf(uint32_t *parent, double *length)
{
    parent[0] = NJ_NONE;
    length[0] = 0.0;
}

int pansim_nj_tree(pansim_ctx *c, int metric, uint32_t *parent, double *length)
{
    if (!c || !parent || !length) return PANSIM_ERR_INVALID;
    if (int rc = nj_check(c, metric, true)) return rc;
    if (c->N == 1) { nj_single_leaf(parent, length); return 0; }
    NjCall w;
    if (int rc = nj_alloc(c, c->N, w)) return rc;
    if (int rc = nj_build_ctx(c, metric, w)) return rc;
    if (int rc = nj_join_loop(c, w, parent, length, nullptr, nullptr, nullptr)) return rc;
    return check_device_flag(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG);
}

int pansim_nj_tree_matrix(pansim_ctx *c, const double *upper, uint32_t n, uint32_t *parent, double *length)
{
    if (!c || !parent || !length || n == 0 || (n > 1 && !upper)) return PANSIM_ERR_INVALID;
    const uint64_t m = (uint64_t)n * (n - 1) / 2;
    for (uint64_t e = 0; e < m; e++)
        if (!std::isfinite(upper[e]) || upper[e] < 0.0)
            FAIL(c, PANSIM_ERR_INVALID, "neighbour-joining: matrix entry %llu is %g (finite and >= 0 required)", (unsigned long long)e, upper[e]);
    if (n == 1) { nj_single_leaf(parent, length); return 0; }
    NjCall w;
    if (int rc = nj_alloc(c, n, w)) return rc;
    double *d_upper = nullptr;
    if (cudaMalloc(&d_upper, m * 8) != cudaSuccess) {
        cudaGetLastError();
        FAIL(c, PANSIM_ERR_NOMEM, "neighbour-joining: cudaMalloc of the %llu matrix entries failed", (unsigned long long)m);
    }
    cudaError_t e = cudaMemcpyAsync(d_upper, upper, m * 8, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        nj_scatter_upper_kernel<<<std::min<uint32_t>(n, w.max_grid), 256, 0, c->stream>>>(d_upper, n, w.D[0], nj_pitch(n));
        e = cudaGetLastError();
    }
    cudaStreamSynchronize(c->stream);
    cudaFree(d_upper);
    CU(c, e);
    return nj_join_loop(c, w, parent, length, nullptr, nullptr, nullptr);
}

int pansim_nj_kernel_ms(pansim_ctx *c, int metric, uint32_t repeats, float *build_ms, float *join_ms, uint64_t *bytes_scanned,
                        uint32_t *compactions)
{
    if (!c || !repeats) return PANSIM_ERR_INVALID;
    if (int rc = nj_check(c, metric, true)) return rc;
    if (c->N < 2) FAIL(c, PANSIM_ERR_INVALID, "neighbour-joining measurement needs pop_size >= 2");
    std::vector<uint32_t> parent(nj_nodes(c->N));
    std::vector<double> length(parent.size());
    cudaEvent_t ev[3];
    for (auto &x : ev) CU(c, cudaEventCreate(&x));
    double tb = 0.0, tj = 0.0;
    int rc = 0;
    for (uint32_t r = 0; r <= repeats && !rc; r++) {             // r = 0 warms up
        NjCall w;
        if ((rc = nj_alloc(c, c->N, w))) break;
        cudaEventRecord(ev[0], c->stream);
        if ((rc = nj_build_ctx(c, metric, w))) break;
        if ((rc = nj_join_loop(c, w, parent.data(), length.data(), ev + 1, bytes_scanned, compactions))) break;
        float b = 0.f, j = 0.f;
        cudaEventElapsedTime(&b, ev[0], ev[1]);
        cudaEventElapsedTime(&j, ev[1], ev[2]);
        if (r) { tb += b; tj += j; }
    }
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (build_ms) *build_ms = (float)(tb / repeats);
    if (join_ms) *join_ms = (float)(tj / repeats);
    return check_device_flag(c, PANSIM_ERR_WEIGHTS, PANSIM_WEIGHTS_MSG);
}

// ---- clonal genealogy (genealogy.cuh, DESIGN.md section 13) ------------------
// trace scratch and node table: owner, cnt, newid [N]; lineage nodes and ancestors [2][N] each; parent, individual,
// time [2N] each; n_nodes and lineages_at_start
static size_t gen_scratch_words(uint32_t N) { return (size_t)13 * N + 2; }

int pansim_enable_genealogy(pansim_ctx *c, uint32_t capacity)
{
    if (!c) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->stream_gen) CU(c, cudaStreamSynchronize(c->stream_gen));
    for (uint32_t **p : {&c->d_gen_ring, &c->d_gen_scratch, &c->d_gen_pairs}) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    c->gen_pair_cap = 0;
    c->gen_cap = 0;
    for (bool &v : c->gen_done_valid) v = false;
    genealogy_reset(c);
    if (capacity == 0) return 0;
    if (!c->stream_gen) {
        CU(c, cudaStreamCreateWithFlags(&c->stream_gen, cudaStreamNonBlocking));
        for (auto &e : c->ev_gen_done) CU(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const bool fits = (uint64_t)capacity <= (uint64_t)SIZE_MAX / 4 / c->N;
    if (!fits || cudaMalloc(&c->d_gen_ring, (size_t)capacity * c->N * 4) != cudaSuccess ||
        cudaMalloc(&c->d_gen_scratch, gen_scratch_words(c->N) * 4) != cudaSuccess) {
        cudaGetLastError();
        for (uint32_t **p : {&c->d_gen_ring, &c->d_gen_scratch}) {
            if (*p) cudaFree(*p);
            *p = nullptr;
        }
        FAIL(c, PANSIM_ERR_NOMEM, "genealogy ring of %u x %u parent vectors: cudaMalloc failed; recording stays off", capacity, c->N);
    }
    c->gen_cap = capacity;
    return 0;
}

// the node table of the current record on the device (traced again only when the record changed)
static int genealogy_trace(pansim_ctx *c, GenealogyTrace &a)
{
    const uint32_t N = c->N;
    uint32_t *w = c->d_gen_scratch;
    a.ring = c->d_gen_ring;
    a.cap = c->gen_cap;
    a.N = N;
    a.T = (uint32_t)std::min<uint64_t>(c->gen_total, c->gen_cap);
    a.base = (uint32_t)((c->gen_total - a.T) % c->gen_cap);
    a.owner = w; a.cnt = w + N; a.newid = w + 2 * (size_t)N;
    a.lin_node[0] = w + 3 * (size_t)N; a.lin_node[1] = w + 4 * (size_t)N;
    a.lin_anc[0] = w + 5 * (size_t)N; a.lin_anc[1] = w + 6 * (size_t)N;
    a.parent = w + 7 * (size_t)N; a.individual = w + 9 * (size_t)N; a.time = w + 11 * (size_t)N;
    a.out = w + 13 * (size_t)N;
    if (c->gen_traced == c->gen_epoch) return 0;
    genealogy_trace_kernel<<<1, GT_THREADS, 0, c->stream_gen>>>(a);
    LAUNCH_CHECK(c);
    uint32_t out[2];
    CU(c, cudaMemcpyAsync(out, a.out, sizeof out, cudaMemcpyDeviceToHost, c->stream_gen));
    CU(c, cudaStreamSynchronize(c->stream_gen));
    c->gen_nodes = out[0];
    c->gen_lineages = out[1];
    c->gen_traced = c->gen_epoch;
    return 0;
}

static int genealogy_require(pansim_ctx *c)
{
    if (!c->gen_cap) FAIL(c, PANSIM_ERR_STATE, "genealogy recording is off: call pansim_enable_genealogy first");
    CU(c, cudaSetDevice(c->cfg.device));
    return 0;
}

int pansim_genealogy(pansim_ctx *c, pansim_genealogy_node *nodes, pansim_genealogy_info *info)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (int rc = genealogy_require(c)) return rc;
    GenealogyTrace a;
    if (int rc = genealogy_trace(c, a)) return rc;
    if (nodes) {
        const size_t n = c->gen_nodes;
        std::vector<uint32_t> h(3 * n);
        CU(c, cudaMemcpyAsync(h.data(), a.parent, n * 4, cudaMemcpyDeviceToHost, c->stream_gen));
        CU(c, cudaMemcpyAsync(h.data() + n, a.individual, n * 4, cudaMemcpyDeviceToHost, c->stream_gen));
        CU(c, cudaMemcpyAsync(h.data() + 2 * n, a.time, n * 4, cudaMemcpyDeviceToHost, c->stream_gen));
        CU(c, cudaStreamSynchronize(c->stream_gen));
        for (size_t k = 0; k < n; k++) nodes[k] = {h[k], h[n + k], h[2 * n + k]};
    }
    if (info) {
        info->generations_total = c->gen_total;
        info->generations_kept = a.T;
        info->n_nodes = c->gen_nodes;
        info->lineages_at_start = c->gen_lineages;
    }
    return 0;
}

int pansim_genealogy_history(pansim_ctx *c, uint32_t *out)
{
    if (!c || !out) return PANSIM_ERR_INVALID;
    if (int rc = genealogy_require(c)) return rc;
    const uint64_t T = std::min<uint64_t>(c->gen_total, c->gen_cap);
    const uint64_t base = (c->gen_total - T) % c->gen_cap;
    const uint64_t first = std::min<uint64_t>(T, c->gen_cap - base);        // oldest vectors up to the end of the ring
    const size_t row = (size_t)c->N * 4;
    if (first) CU(c, cudaMemcpyAsync(out, c->d_gen_ring + base * c->N, first * row, cudaMemcpyDeviceToHost, c->stream_gen));
    if (T > first) CU(c, cudaMemcpyAsync(out + first * c->N, c->d_gen_ring, (T - first) * row, cudaMemcpyDeviceToHost, c->stream_gen));
    CU(c, cudaStreamSynchronize(c->stream_gen));
    return 0;
}

int pansim_genealogy_tmrca(pansim_ctx *c, const uint32_t *r1, const uint32_t *r2, size_t P, uint32_t *tmrca)
{
    if (!c || (P && (!r1 || !r2 || !tmrca))) return PANSIM_ERR_INVALID;
    if (int rc = genealogy_require(c)) return rc;
    for (size_t k = 0; k < P; k++)
        if (r1[k] >= c->N || r2[k] >= c->N) FAIL(c, PANSIM_ERR_INVALID, "TMRCA pair %zu = (%u, %u): index >= pop_size %u", k, r1[k], r2[k], c->N);
    GenealogyTrace a;
    if (int rc = genealogy_trace(c, a)) return rc;
    if (P == 0) return 0;
    if (P > c->gen_pair_cap) {
        if (c->d_gen_pairs) cudaFree(c->d_gen_pairs);
        c->d_gen_pairs = nullptr;
        c->gen_pair_cap = 0;
        if (cudaMalloc(&c->d_gen_pairs, 3 * P * 4) != cudaSuccess) { cudaGetLastError(); FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for %zu TMRCA pairs failed", P); }
        c->gen_pair_cap = P;
    }
    uint32_t *d1 = c->d_gen_pairs, *d2 = d1 + P, *dt = d2 + P;
    CU(c, cudaMemcpyAsync(d1, r1, P * 4, cudaMemcpyHostToDevice, c->stream_gen));
    CU(c, cudaMemcpyAsync(d2, r2, P * 4, cudaMemcpyHostToDevice, c->stream_gen));
    const unsigned grid = (unsigned)std::min<uint64_t>(div_up64(P, 256), (uint64_t)c->sm_count * 16);
    genealogy_tmrca_kernel<<<grid, 256, 0, c->stream_gen>>>(a.parent, a.time, d1, d2, P, dt);
    LAUNCH_CHECK(c);
    CU(c, cudaMemcpyAsync(tmrca, dt, P * 4, cudaMemcpyDeviceToHost, c->stream_gen));
    CU(c, cudaStreamSynchronize(c->stream_gen));
    return 0;
}

// Newick of a checked node table, no device: root last, every other node's parent above it, so the tree is walked with
// an explicit stack (no recursion: a caterpillar of any size is fine). Leaves are ind_<i>, children go in the order of
// their smallest leaf; put_length(v, put) writes the ":<length>" of non-root node v. Returns the text's length.
extern "C++" {
template <class Parent, class PutLength>
static size_t newick_write(uint32_t n_nodes, uint32_t n_leaves, Parent parent_of, PutLength put_length, char *out, size_t cap)
{
    const uint32_t root = n_nodes - 1;
    // smallest leaf below every node; the children of every node in that order (CSR)
    std::vector<uint32_t> minleaf(n_nodes, GEN_NONE), first(n_nodes + 1, 0), child(root);
    for (uint32_t k = 0; k < n_leaves; k++) minleaf[k] = k;
    for (uint32_t k = 0; k < root; k++) {
        minleaf[parent_of(k)] = std::min(minleaf[parent_of(k)], minleaf[k]);
        first[parent_of(k) + 1]++;
    }
    for (uint32_t k = 0; k < n_nodes; k++) first[k + 1] += first[k];
    std::vector<uint32_t> order(root), fill(first.begin(), first.end() - 1);
    for (uint32_t k = 0; k < root; k++) order[k] = k;
    std::sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return minleaf[x] != minleaf[y] ? minleaf[x] < minleaf[y] : x < y; });
    for (uint32_t k : order) child[fill[parent_of(k)]++] = k;
    size_t pos = 0;
    auto put = [&](const char *s, size_t n) {
        if (out && pos + n <= cap) memcpy(out + pos, s, n);
        pos += n;
    };
    auto enter = [&](uint32_t v) {
        if (v < n_leaves) {
            char b[24];
            const int n = snprintf(b, sizeof b, "ind_%u", v);
            put(b, (size_t)n);
        } else {
            put("(", 1);
        }
    };
    struct Frame { uint32_t node, next; };
    std::vector<Frame> stack{{root, 0}};
    enter(root);
    while (!stack.empty()) {
        const uint32_t v = stack.back().node, i = stack.back().next;
        if (v >= n_leaves && first[v] + i < first[v + 1]) {
            if (i) put(",", 1);
            const uint32_t ch = child[first[v] + i];
            stack.back().next++;
            enter(ch);
            stack.push_back({ch, 0});
            continue;
        }
        if (v >= n_leaves) put(")", 1);
        if (v != root) put_length(v, put);
        stack.pop_back();
    }
    put(";\n", 2);
    return pos;
}
}  // extern "C++"

// the text into out when it fits with its terminating NUL (out = NULL: only the length)
static int newick_finish(char *out, size_t cap, size_t pos, size_t *len)
{
    *len = pos;
    if (!out) return 0;
    if (cap < pos + 1) return PANSIM_ERR_INVALID;
    out[pos] = '\0';
    return 0;
}

int pansim_genealogy_newick(const pansim_genealogy_node *nodes, uint32_t n_nodes, uint32_t n_leaves, char *out,
                            size_t cap, size_t *len)
{
    if (!nodes || !len || n_leaves == 0 || n_nodes < n_leaves || (uint64_t)n_nodes > 2ull * n_leaves) return PANSIM_ERR_INVALID;
    const uint32_t root = n_nodes - 1;
    if (nodes[root].parent != GEN_NONE) return PANSIM_ERR_INVALID;
    for (uint32_t k = 0; k < root; k++) {
        const uint32_t p = nodes[k].parent;
        if (p <= k || p < n_leaves || p >= n_nodes || nodes[p].time < nodes[k].time) return PANSIM_ERR_INVALID;
    }
    const size_t pos = newick_write(
        n_nodes, n_leaves, [&](uint32_t k) { return nodes[k].parent; },
        [&](uint32_t v, auto &put) {
            char b[24];
            const int n = snprintf(b, sizeof b, ":%u", nodes[nodes[v].parent].time - nodes[v].time);
            put(b, (size_t)n);
        },
        out, cap);
    return newick_finish(out, cap, pos, len);
}

int pansim_tree_newick(const uint32_t *parent, const double *length, uint32_t n_nodes, uint32_t n_leaves, char *out,
                       size_t cap, size_t *len)
{
    if (!parent || !length || !len || n_leaves == 0 || !node_table_error(parent, n_nodes, n_leaves, nullptr).empty())
        return PANSIM_ERR_INVALID;
    const size_t pos = newick_write(
        n_nodes, n_leaves, [&](uint32_t k) { return parent[k]; },
        [&](uint32_t v, auto &put) {
            char b[40];
            const int n = snprintf(b, sizeof b, ":%.17g", length[v]);
            put(b, (size_t)n);
        },
        out, cap);
    return newick_finish(out, cap, pos, len);
}

// ---- split comparison (no device) -------------------------------------------------------------
// The leaves of a checked table in an order where every subtree is a contiguous run and leaf 0 comes first (at every
// node the child holding leaf 0 is laid out first). Then the side of a split without leaf 0 is a run too: the subtree
// [lo, hi] itself, or [hi + 1, N - 1] when the subtree holds leaf 0. sides = those runs with 2 .. N - 2 leaves, as
// lo << 32 | hi, sorted, distinct. pos[leaf] = its place in the order, order[place] = the leaf.
static void tree_sides(const uint32_t *parent, uint32_t n_nodes, uint32_t N, std::vector<uint32_t> &pos,
                       std::vector<uint32_t> &order, std::vector<uint64_t> &sides)
{
    const uint32_t root = n_nodes - 1;
    std::vector<uint32_t> cnt(n_nodes, 0), start(n_nodes, 0), off(n_nodes + 1, 0), child(root);
    std::vector<uint8_t> has0(n_nodes, 0);
    for (uint32_t k = 0; k < N; k++) cnt[k] = 1;
    has0[0] = 1;
    for (uint32_t k = 0; k < root; k++) {
        cnt[parent[k]] += cnt[k];
        has0[parent[k]] |= has0[k];
        off[parent[k] + 1]++;
    }
    for (uint32_t k = 0; k < n_nodes; k++) off[k + 1] += off[k];
    std::vector<uint32_t> fill(off.begin(), off.end() - 1);
    for (uint32_t k = 0; k < root; k++) child[fill[parent[k]]++] = k;
    for (uint32_t v = root + 1; v-- > N;) {                  // parents before children
        uint32_t run = start[v];
        for (int pass = 0; pass < 2; pass++)                 // the child holding leaf 0 first
            for (uint32_t e = off[v]; e < off[v + 1]; e++)
                if (has0[child[e]] == (pass == 0)) { start[child[e]] = run; run += cnt[child[e]]; }
    }
    pos.assign(N, 0);
    order.assign(N, 0);
    for (uint32_t k = 0; k < N; k++) { pos[k] = start[k]; order[start[k]] = k; }
    sides.clear();
    for (uint32_t v = 0; v < root; v++) {
        uint64_t lo = start[v], hi = (uint64_t)start[v] + cnt[v] - 1;
        if (lo == 0) { lo = hi + 1; hi = N - 1; }
        const uint64_t size = hi + 1 - lo;
        if (size >= 2 && size + 2 <= N) sides.push_back(lo << 32 | hi);
    }
    std::sort(sides.begin(), sides.end());
    sides.erase(std::unique(sides.begin(), sides.end()), sides.end());
}

// A side of B (a run of B's order) is a split of A iff its leaves occupy a run [m, M] of A's order (M - m + 1 = its
// size; min and max by a sparse table over A's places in B's order) and [m, M] is one of A's sides.
int pansim_tree_compare_splits(const uint32_t *parent_a, uint32_t n_a, const uint32_t *parent_b, uint32_t n_b,
                               uint32_t n_leaves, uint64_t out[3])
{
    if (!out || n_leaves == 0 || !node_table_error(parent_a, n_a, n_leaves, nullptr).empty() ||
        !node_table_error(parent_b, n_b, n_leaves, nullptr).empty())
        return PANSIM_ERR_INVALID;
    const uint32_t N = n_leaves;
    std::vector<uint32_t> pos_a, order_a, pos_b, order_b;
    std::vector<uint64_t> sides_a, sides_b;
    tree_sides(parent_a, n_a, N, pos_a, order_a, sides_a);
    tree_sides(parent_b, n_b, N, pos_b, order_b, sides_b);
    uint32_t levels = 1;
    while ((1ull << levels) <= N) levels++;
    std::vector<std::vector<uint32_t>> mn(levels), mx(levels);
    mn[0].resize(N);
    for (uint32_t i = 0; i < N; i++) mn[0][i] = pos_a[order_b[i]];
    mx[0] = mn[0];
    for (uint32_t l = 1; l < levels; l++) {
        const uint32_t w = 1u << (l - 1), n = N - (1u << l) + 1;
        mn[l].resize(n);
        mx[l].resize(n);
        for (uint32_t i = 0; i < n; i++) {
            mn[l][i] = std::min(mn[l - 1][i], mn[l - 1][i + w]);
            mx[l][i] = std::max(mx[l - 1][i], mx[l - 1][i + w]);
        }
    }
    uint64_t shared = 0;
    for (uint64_t s : sides_b) {
        const uint32_t lo = (uint32_t)(s >> 32), hi = (uint32_t)s, l = 31 - __builtin_clz(hi - lo + 1);
        const uint32_t m = std::min(mn[l][lo], mn[l][hi + 1 - (1u << l)]), M = std::max(mx[l][lo], mx[l][hi + 1 - (1u << l)]);
        if (M - m == hi - lo && std::binary_search(sides_a.begin(), sides_a.end(), (uint64_t)m << 32 | M)) shared++;
    }
    out[0] = sides_a.size();
    out[1] = sides_b.size();
    out[2] = shared;
    return 0;
}

// ---- communicator over column shards (one process per GPU) -------------------
int pansim_comm_unique_id(void *id_out)
{
    if (!id_out) return PANSIM_ERR_INVALID;
    NcclApi &api = nccl_api();
    if (!api.ok()) { g_create_error = api.error; return PANSIM_ERR_CUDA; }
    ncclUniqueId id;
    const ncclResult_t r = api.GetUniqueId(&id);
    if (r != ncclSuccess) { g_create_error = std::string("ncclGetUniqueId failed: ") + api.GetErrorString(r); return PANSIM_ERR_CUDA; }
    static_assert(sizeof(id) == PANSIM_COMM_ID_BYTES, "ncclUniqueId size");
    memcpy(id_out, &id, sizeof id);
    return 0;
}

int pansim_comm_init_rank(pansim_ctx *c, int n_ranks, int rank, const void *id)
{
    if (!c || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return PANSIM_ERR_INVALID;
    if (c->comm) FAIL(c, PANSIM_ERR_STATE, "context already has a communicator");
    NcclApi &api = nccl_api();
    if (!api.ok()) FAIL(c, PANSIM_ERR_CUDA, "%s", api.error.c_str());
    CU(c, cudaSetDevice(c->cfg.device));
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof uid);
    NCK(c, api.CommInitRank(&c->comm, n_ranks, uid, rank));
    c->comm_size = n_ranks; c->comm_rank = rank; c->comm_owned = true;
    return 0;
}

int pansim_comm_info(pansim_ctx *c, int *n_ranks, int *rank)
{
    if (!c) return PANSIM_ERR_INVALID;
    if (n_ranks) *n_ranks = c->comm ? c->comm_size : 1;
    if (rank) *rank = c->comm ? c->comm_rank : 0;
    return 0;
}

// ---- event dump -------------------------------------------------------------
int pansim_enable_event_dump(pansim_ctx *c, size_t max_core_events)
{
    if (!c || max_core_events == 0 || max_core_events > 0x7FFFFFFFull) return PANSIM_ERR_INVALID;
    CU(c, cudaSetDevice(c->cfg.device));
    if (c->dump_enabled) FAIL(c, PANSIM_ERR_STATE, "event dump already enabled");
    const size_t n = max_core_events;
    const size_t accw = (size_t)c->N * c->acc_stride_words * 4;
    struct Want { void **p; size_t bytes; };
    const Want want[] = {{(void **)&c->d_mut_row, n * 4}, {(void **)&c->d_mut_site, n * 4}, {(void **)&c->d_mut_seq, n * 4},
                         {(void **)&c->d_mut_allele, n}, {(void **)&c->d_hr_rec, n * 4}, {(void **)&c->d_hr_locus, n * 4},
                         {(void **)&c->d_hr_donor, n * 4}, {(void **)&c->d_hr_seq, n * 4}, {(void **)&c->d_hr_value, n},
                         {(void **)&c->d_dump_flip, accw}, {(void **)&c->d_dump_gain, accw}};
    for (const Want &w : want) {
        if (cudaMalloc(w.p, w.bytes) != cudaSuccess) {
            *w.p = nullptr;
            for (const Want &u : want) { if (*u.p) cudaFree(*u.p); *u.p = nullptr; }      // nothing stays half-allocated
            cudaGetLastError();
            FAIL(c, PANSIM_ERR_NOMEM, "cudaMalloc for the event dump (%zu events) failed", n);
        }
    }
    CU(c, cudaMemset(c->d_dump_flip, 0, accw)); CU(c, cudaMemset(c->d_dump_gain, 0, accw));
    c->dump_cap = (uint32_t)n;
    c->dump_enabled = true;
    return 0;
}

int pansim_fetch_event_dump(pansim_ctx *c, pansim_event_dump *o)
{
    if (!c || !o) return PANSIM_ERR_INVALID;
    if (!c->dump_enabled) FAIL(c, PANSIM_ERR_STATE, "event dump not enabled");
    CU(c, cudaSetDevice(c->cfg.device));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaStreamSynchronize(c->stream_core));
    memset(o, 0, sizeof *o);
    uint32_t cnt[2];
    CU(c, cudaMemcpy(cnt, c->d_dump_counters, sizeof cnt, cudaMemcpyDeviceToHost));
    if (cnt[0] > c->dump_cap || cnt[1] > c->dump_cap) FAIL(c, PANSIM_ERR_NOMEM, "event dump overflow: %u SNP / %u HR events, capacity %u", cnt[0], cnt[1], c->dump_cap);
    auto fetch = [&](const void *d, size_t bytes) -> void * {
        void *h = malloc(bytes ? bytes : 1);
        if (bytes) cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost);
        return h;
    };
    o->n_core_mut = cnt[0];
    o->core_mut_row = (uint32_t *)fetch(c->d_mut_row, cnt[0] * 4ul);
    o->core_mut_site = (uint32_t *)fetch(c->d_mut_site, cnt[0] * 4ul);
    o->core_mut_seq = (uint32_t *)fetch(c->d_mut_seq, cnt[0] * 4ul);
    o->core_mut_allele = (uint8_t *)fetch(c->d_mut_allele, cnt[0]);
    o->n_hr = cnt[1];
    o->hr_recipient = (uint32_t *)fetch(c->d_hr_rec, cnt[1] * 4ul);
    o->hr_locus = (uint32_t *)fetch(c->d_hr_locus, cnt[1] * 4ul);
    o->hr_donor = (uint32_t *)fetch(c->d_hr_donor, cnt[1] * 4ul);
    o->hr_seq = (uint32_t *)fetch(c->d_hr_seq, cnt[1] * 4ul);
    o->hr_value = (uint8_t *)fetch(c->d_hr_value, cnt[1]);
    const size_t words = (size_t)c->N * c->acc_stride_words;
    std::vector<uint32_t> tmp(words ? words : 1);
    for (int which = 0; which < 2; which++) {
        uint8_t *m = (uint8_t *)malloc(((size_t)c->N * c->G) > 0 ? (size_t)c->N * c->G : 1);
        CU(c, cudaMemcpy(tmp.data(), which ? c->d_dump_gain : c->d_dump_flip, words * 4, cudaMemcpyDeviceToHost));
        for (uint32_t r = 0; r < c->N; r++)
            for (uint32_t g = 0; g < c->G; g++)
                m[(size_t)r * c->G + g] = (uint8_t)((tmp[(size_t)r * c->acc_stride_words + (g >> 5)] >> (g & 31)) & 1u);
        if (which) o->acc_gain_mask = m; else o->acc_flip_mask = m;
    }
    CU(c, cudaGetLastError());
    return 0;
}

void pansim_free_event_dump(pansim_event_dump *d)
{
    if (!d) return;
    free(d->core_mut_row); free(d->core_mut_site); free(d->core_mut_seq); free(d->core_mut_allele);
    free(d->hr_recipient); free(d->hr_locus); free(d->hr_donor); free(d->hr_seq); free(d->hr_value);
    free(d->acc_flip_mask); free(d->acc_gain_mask);
    memset(d, 0, sizeof *d);
}

#include "group_api.inl"

}  // extern "C"
