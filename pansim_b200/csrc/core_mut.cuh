// core_mut.cuh -- K4a: gather-by-parent fused with SNP mutation (core genome).
//
// One pass over the 2-bit packed core alignment does, per output row i:
//   gather-by-parent   next[i,:] = pop[parents[i],:]      (population.rs:450-465)
//   SNP mutation       population.rs:512-539
// Homologous recombination (population.rs:544-751) needs the finished rows of
// ALL individuals (they are the snapshot of :693-695), so it cannot be applied
// while this pass is still writing them. It is DEFERRED instead: the rows this
// kernel writes are the pre-recombination snapshot of generation g, and the
// recombination events of generation g are applied by the NEXT launch to every
// region right after it has been loaded (a child inherits its parent's row
// *after* recombination). The donor cells are then read from the old buffer,
// which is read-only here, so there is no hazard and no second pass over the
// state; the events are recomputed from their counters (core_hr.cuh), and the
// donor words are fetched one item ahead of their use. A reader of the state
// (distances, downloads) first materialises the pending events with the
// stand-alone kernels of core_hr.cuh; both routes give identical states.
//
// Every output cell is a pure function of (old state, parents, Philox key):
// no races, no atomics, independent of grid size and of the column sharding.
//
// Exact thinning instead of the reference's per-row event loop (SURVEY.md 8a
// row M): per row the reference draws n ~ Poisson(lambda) events at uniform
// sites, each writing U{C,G,T} (core_vec[1 >> value] is always core_vec[0],
// population.rs:531). Restricted to a 256-site block that is a
// Poisson(256*lambda/L) number of events at uniform positions, one byte of
// Philox output each; later events overwrite earlier ones.
//
// The kernel is instruction-issue bound, not HBM bound (DESIGN.md section 7),
// so the event loop is written for instruction count:
//   * a position byte b addresses word (b & 15) of the lane's 16 words and
//     cell (b >> 4) of that word; the shared-memory address is one shift and
//     one LOP3 ((p >> k) & 0x780 | lane/stage base, stages 2 KiB aligned), the
//     cell mask one wrap-mode shift of a pre-masked copy of the position word;
//   * alleles: a uniform byte v < 243 carries base-3 digits; a 243-entry table
//     in shared memory maps v to four words, word j holding allele code
//     (digit j) + 1 replicated into all 16 cells, so the read-modify-write is
//     LDS, SHF, LOP3 (bit select), predicated STS;
//   * the five chunks (4 events each) of the first two Philox calls are
//     unrolled behind warp-uniform guards, positions are compile-time shifts.
//
// Data movement: warp-private TMA pipelines (cp.async.bulk global->shared with
// mbarrier completion from the PARENT's row, cp.async.bulk shared->global into
// the child's row), two 2 KiB stages per warp, no CTA-wide barrier in the
// steady state. One item keeps a warp busy far longer than a load takes, so a
// load issued one item ahead is hidden. Two stages and a 48-register budget
// (40 used) leave a quarter of each SM's registers and ~38 KB of its shared
// memory free at four resident CTAs: the selection chain of the next
// generation runs there beside the core kernel instead of waiting for core
// CTAs to retire (DESIGN.md section 5).
#pragma once
#include "common.cuh"
#include "core_hr.cuh"

namespace pansim {

#ifndef PANSIM_CM_WARPS
#define PANSIM_CM_WARPS 8
#endif
#ifndef PANSIM_CM_MAXREG
#define PANSIM_CM_MAXREG 0          // > 0: cap registers per thread with __maxnreg__ instead of the launch bound
#endif
constexpr int CM_WARPS = PANSIM_CM_WARPS;
// PANSIM_CM_STAGES=3 PANSIM_CM_CTAS=4 builds the earlier three-stage ring (58 registers) for comparison
#ifndef PANSIM_CM_STAGES
#define PANSIM_CM_STAGES 2
#endif
#ifndef PANSIM_CM_CTAS
#define PANSIM_CM_CTAS 5
#endif
#ifndef PANSIM_CM_RESIDENT
#define PANSIM_CM_RESIDENT 4
#endif
constexpr int CM_STAGES = PANSIM_CM_STAGES;       // 2 KiB stages per warp
constexpr int CM_CTAS_PER_SM = PANSIM_CM_CTAS;    // launch bound (register budget = 65536 / (256 * CTAs))
// CTAs resident per SM at most: the host sizes the dynamic shared memory of a CTA so that no more fit.
// At cfg2, 4 resident CTAs of the two-stage kernel: 143.8-144.3 us per generation; 5 (40 warps, the
// chain squeezed out of every scheduler): 152.3-152.5.
constexpr int CM_RESIDENT_CTAS = PANSIM_CM_RESIDENT;
// Two stages: the load of item j+1 is issued in item j, after its recombination apply, once the bulk
// store of item j-1 has finished reading the stage it reuses. Three stages: issued at the end of
// item j-1, two items ahead.
constexpr bool CM_LATE_LOAD = CM_STAGES == 2;
constexpr int CM_THREADS = CM_WARPS * 32;
constexpr uint32_t CM_GUIDE = 512;            // u16 guide entries (= 256 words)
constexpr uint32_t CM_GUIDE_SHIFT = 23;
constexpr uint32_t CM_GUIDE_WORDS = CM_GUIDE / 2;
constexpr uint32_t CM_LUT_ENTRIES = 243;
constexpr uint32_t CM_LUT_BYTES = 3904;       // 243 x 16, rounded up to 64
constexpr uint32_t CM_GROUP0 = 20;            // events carried by Philox calls 0 and 1
constexpr uint32_t CM_TAIL = 8;               // events carried by each later call

struct CoreMutArgs {
    const uint8_t *old_state;
    uint8_t *new_state;
    const uint32_t *parents;  // nullptr = identity gather
    uint32_t n_rows;
    uint32_t n_regions;       // regions per (local) row
    uint64_t row_stride;      // bytes
    uint32_t region0;         // global index of local region 0
    uint32_t items_per_warp;
    uint64_t site_limit;      // global site index one past the last valid site of this shard
    uint32_t last_greg, lim_last;   // the region that holds site_limit - 1 and its number of valid sites (1..8192)
    uint2 key;
    PhiloxKeys rk;            // round keys of `key`
    uint32_t gen;
    // constants of the launch, one contiguous device image copied into shared memory by a single bulk
    // copy: [243 x uint4 allele-digit table (CM_LUT_BYTES)][CM_GUIDE u16 guide][mut_size thresholds of the
    // SNP count per 256-site block][hr_size thresholds of the recombination count per region]
    const uint8_t *const_img;
    uint32_t mut_size, mut_nsub, mut_kmax;
    // recombination events of generation hr_gen still pending on old_state (hr_nsub = 0: none)
    uint32_t hr_size, hr_nsub, hr_kmax, hr_gen;
    const uint32_t *gen_dev;  // nullptr, or a device word added to gen / hr_gen (replayed CUDA graphs: the generation number of a
                              // captured launch is relative to a counter the graph advances itself)
    uint32_t hr_k0;           // first threshold of the 32-wide window hr_count_from_uniform_s tries first (<= hr_size - 32)
    uint32_t hr_lemire_t;     // 2^32 mod (n_rows - 1), see hr_event
    // optional event dump (parity instrumentation)
    uint32_t *dump_counters;  // [0] = SNP events
    uint32_t dump_cap;
    uint32_t *d_mut_row, *d_mut_site, *d_mut_seq;
    uint8_t *d_mut_allele;
};

__host__ __device__ static inline uint32_t core_mut_tab_words(uint32_t mut_size, uint32_t hr_size)
{
    return (CM_GUIDE_WORDS + mut_size + hr_size + 3u) & ~3u;     // bulk copies move multiples of 16 bytes
}

// bytes of the constant image (device and shared memory)
__host__ __device__ static inline uint32_t core_mut_const_bytes(uint32_t mut_size, uint32_t hr_size)
{
    return CM_LUT_BYTES + core_mut_tab_words(mut_size, hr_size) * 4u;
}

static inline size_t core_mut_smem_bytes(uint32_t mut_size, uint32_t hr_size)
{
    return 2048 /* alignment slack */ + (size_t)CM_WARPS * CM_STAGES * REGION_BYTES + core_mut_const_bytes(mut_size, hr_size) +
           (size_t)(CM_WARPS * CM_STAGES + 1) * sizeof(uint64_t);
}

// Poisson by CDF inversion (see common.cuh) with a 512-bin u16 guide: entry =
// 2*k0 + many, k0 = #{j : T[j] <= bin start}. A bin holding at most one
// threshold needs exactly one comparison; `many` marks the few tail bins that
// hold more and finish with a scan.
__device__ __forceinline__ uint32_t poisson_fast(const uint32_t *tab, uint32_t kmax, uint32_t u)
{
    const uint32_t g = reinterpret_cast<const uint16_t *>(tab)[u >> CM_GUIDE_SHIFT];
    const uint32_t *thr = tab + CM_GUIDE_WORDS;
    uint32_t k = g >> 1;
    k += thr[k] <= u ? 1u : 0u;
    if (g & 1u) {
        while (k < kmax && thr[k] <= u) k++;
    }
    return k;
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// the same sampler on a 32-bit shared-space address of the table image (hot path: no generic pointers)
__device__ __forceinline__ uint32_t poisson_fast_s(uint32_t tab_s, uint32_t kmax, uint32_t u)
{
    uint32_t g;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(g) : "r"(tab_s + (u >> CM_GUIDE_SHIFT) * 2u));
    const uint32_t thr_s = tab_s + CM_GUIDE_WORDS * 4u;
    uint32_t k = g >> 1;
    k += lds_u32(thr_s + k * 4u) <= u ? 1u : 0u;
    if (g & 1u) {
        while (k < kmax && lds_u32(thr_s + k * 4u) <= u) k++;
    }
    return k;
}

// hr_count_from_uniform (core_hr.cuh) on a shared-space address. k = #{j : T[j] <= u} with T
// non-decreasing: one ballot over the 32 thresholds T[k0 .. k0+31] that carry nearly all of the
// probability mass settles it (0 < c < 32 matches in the window means every earlier threshold is
// <= u and every later one is > u, so k = k0 + c); otherwise the whole table is scanned.
__device__ __forceinline__ uint32_t hr_count_from_uniform_s(uint32_t thr_s, uint32_t size, uint32_t kmax, uint32_t k0, uint32_t u,
                                                            uint32_t lane)
{
    const uint32_t c = (uint32_t)__popc(__ballot_sync(0xffffffffu, lds_u32(thr_s + (k0 + lane) * 4u) <= u));
    if (c - 1u < 31u) return min(k0 + c, kmax);
    uint32_t k = 0;
#pragma unroll 1
    for (uint32_t j0 = 0; j0 < size; j0 += 32) k += (uint32_t)__popc(__ballot_sync(0xffffffffu, lds_u32(thr_s + (j0 + lane) * 4u) <= u));
    return min(k, kmax);
}

// means above the table range: extra draws from dedicated count calls (exact by additivity)
__device__ __noinline__ uint32_t mut_count_extra(uint4 ctr, uint2 key, const uint32_t *tab, uint32_t nsub, uint32_t kmax)
{
    uint32_t k = 0;
    for (uint32_t s = 1; s < nsub; s++) {
        uint4 c = ctr;
        c.w |= 0x8000u | ((s - 1) >> 2);
        const uint4 r = philox_core(c, key);
        const uint32_t sel = (s - 1) & 3u;
        const uint32_t u = sel == 0 ? r.x : sel == 1 ? r.y : sel == 2 ? r.z : r.w;
        k += poisson_fast(tab, kmax, u);
    }
    return k;
}

// digit byte and its reserves were all >= 243 (p = 1e-4 per chunk): dedicated Philox word, bias 6e-8
__device__ __noinline__ uint32_t mut_digit_fallback(uint4 ctr, uint2 key, uint32_t tag)
{
    ctr.w |= 0x2000u;
    ctr.x ^= 0x5bd1e995u * (tag + 1u);
    return __umulhi(philox_core(ctr, key).x, 243u);
}

template <bool DUMP>
struct MutChunk {
    uint32_t base_s;          // shared-space address of the stage | lane * 4
    uint32_t lut_s;           // shared-space address of the digit table
    uint32_t k, lane, row, lim;
    uint64_t reg_site0;
    uint4 ctr;
    uint2 key;
    const CoreMutArgs *a;

    // events ev0 .. ev0+3 of this lane's stream: digit byte d (0..255), position bytes in p.
    // `res` = reserve digit bytes (consumed from the low end, 0xFF shifted in).
    __device__ __forceinline__ void run(uint32_t ev0, uint32_t d, uint32_t p, uint32_t &res) const
    {
        const bool rej = d >= 243u;
        uint32_t v = rej ? (res & 255u) : d;
        res = rej ? __funnelshift_r(res, 0xFFFFFFFFu, 8) : res;
        if (v >= 243u) {                              // a second reserve byte before the (costly) fallback call
            v = res & 255u;
            res = __funnelshift_r(res, 0xFFFFFFFFu, 8);
            if (v >= 243u) v = mut_digit_fallback(ctr, key, ev0 >> 2);
        }
        uint32_t c0, c1, c2, c3;
        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(c0), "=r"(c1), "=r"(c2), "=r"(c3) : "r"(lut_s + v * 16u));
        const uint32_t cc[4] = {c0, c1, c2, c3};
        const uint32_t psh = (p >> 3) & 0x1E1E1E1Eu;     // byte j: 2 * cell of event j (bit 0 clear)
        const int rem = (int)k - (int)ev0;               // events of this chunk that exist for this lane
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t fa = j == 0 ? (p << 7) : (p >> (8 * j - 7));
            const uint32_t addr = (fa & 0x780u) | base_s;                 // word (b & 15) * 32 + lane
            const uint32_t m = __funnelshift_l(0u, 3u, psh >> (8 * j));   // 3 << (2 * cell), shift taken mod 32
            uint32_t w;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(addr));
            w = (w & ~m) | (cc[j] & m);
            asm volatile("{\n\t.reg .pred q;\n\tsetp.gt.s32 q, %2, %3;\n\t@q st.shared.u32 [%0], %1;\n\t}"
                         ::"r"(addr), "r"(w), "r"(rem), "r"(j) : "memory");
            if (DUMP) {
                const uint32_t b = (p >> (8 * j)) & 255u;
                const uint32_t sir = (((b & 15u) << 5) + lane) * 16u + (b >> 4);
                if (j < rem && sir < lim) {
                    const uint32_t s = atomicAdd(&a->dump_counters[0], 1u);
                    if (s < a->dump_cap) {
                        a->d_mut_row[s] = row;
                        a->d_mut_site[s] = (uint32_t)(reg_site0 + sir);
                        a->d_mut_seq[s] = ev0 + j;
                        a->d_mut_allele[s] = (uint8_t)(1u << (cc[j] & 3u));
                    }
                }
            }
        }
    }
};

// ---- pending recombination events of the previous generation (see the header) ----------------
// One window = events base .. base+31 of item (parent row prow, local region reg), one per lane.
// K = event count of the item (computed here for base 0), pk = site | keep << 31 where `keep`
// marks the last event of its cell within the window (population.rs:745), dw = the donor's word.
struct HrWindow { uint32_t K, pk, dw; };

__device__ __forceinline__ HrWindow hr_window_fetch(const CoreMutArgs &a, uint32_t hr_gen, const uint32_t *hr_thr, uint32_t hr_thr_s, uint32_t prow,
                                                    uint32_t reg, uint32_t lane, uint32_t base, uint32_t K_known)
{
    const uint32_t greg = a.region0 + reg;
    const uint32_t lim = greg == a.last_greg ? a.lim_last : REGION_SITES;
    const HrEvent ev = hr_event(greg, prow, hr_gen, a.rk, base + lane, a.n_rows - 1u, a.hr_lemire_t);
    // lanes that drew the same site: asked for before the count is known (the match unit is slow and
    // the count needs a shared-memory round trip of its own), validity is folded in afterwards
    const uint32_t same = __match_any_sync(0xffffffffu, ev.pos);
    HrWindow h;
    h.K = K_known;
    if (base == 0u) {
        h.K = hr_count_from_uniform_s(hr_thr_s, a.hr_size, a.hr_kmax, a.hr_k0, __shfl_sync(0xffffffffu, ev.w, 0), lane);
        if (a.hr_nsub > 1) h.K += hr_count_extra(greg, prow, hr_gen, a.key, hr_thr, a.hr_size, a.hr_nsub, a.hr_kmax, lane);
    }
    // events base .. K-1 exist: they sit in the lanes below K - base. A site beyond the ragged end of the
    // alignment is thinned away (the same site in every lane of its match group, so the group drops as a whole).
    const uint32_t n_here = h.K - min(h.K, base);
    const uint32_t live = n_here >= 32u ? 0xffffffffu : ((1u << n_here) - 1u);
    const bool valid = ((live >> lane) & 1u) != 0u && ev.pos < lim;
    const bool keep = valid && (((same & live) >> lane) >> 1) == 0u;        // the last event of a cell wins (population.rs:745)
    h.pk = ev.pos | (keep ? 0x80000000u : 0u);
    h.dw = 0;
    if (keep)   // the old buffer is read-only during this launch: the snapshot the donor cell is taken from (:693-695)
        h.dw = __ldcg(reinterpret_cast<const uint32_t *>(a.old_state + (uint64_t)ev.donor * a.row_stride) +
                      (uint64_t)reg * REGION_WORDS + (ev.pos >> 4));
    return h;
}

// kept cells of one window are distinct, so the XOR of a lane touches bits no other lane reads or writes.
// sw_s = shared-space address of the stage (32-bit addressing: no generic-pointer conversion per item)
__device__ __forceinline__ void hr_window_apply(uint32_t sw_s, const HrWindow &h)
{
    if (h.pk & 0x80000000u) {
        const uint32_t pos = h.pk & 0x1FFFu;
        const uint32_t addr = sw_s + (pos >> 4) * 4u;
        uint32_t w;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(addr));
        const uint32_t delta = (w ^ h.dw) & (3u << ((pos & 15u) * 2u));
        if (delta) asm volatile("red.shared.xor.b32 [%0], %1;" ::"r"(addr), "r"(delta) : "memory");
    }
    __syncwarp();
}

// shared-memory carve-up of one CTA (dynamic shared memory, re-based to a 2 KiB boundary)
struct MutSmem {
    uint8_t *stages;     // CM_WARPS x CM_STAGES x 2 KiB
    uint8_t *lut;        // 243 x uint4
    uint32_t *tab;       // Poisson image (SNP count per 256-site block)
    uint32_t *hr_thr;    // Poisson thresholds (pending recombination events per region)
    uint64_t *bars;      // CM_WARPS x CM_STAGES mbarriers of the stage ring, then one for the constant image
};

__device__ __forceinline__ MutSmem mut_smem_carve(uint8_t *smem_dyn, uint32_t mut_size, uint32_t hr_size)
{
    // stages must sit on 2 KiB boundaries of the shared window (the slot address is an OR)
    const uint32_t pad = (2048u - (smem_u32(smem_dyn) & 2047u)) & 2047u;
    MutSmem m;
    m.stages = smem_dyn + pad;
    m.lut = m.stages + (size_t)CM_WARPS * CM_STAGES * REGION_BYTES;
    m.tab = reinterpret_cast<uint32_t *>(m.lut + CM_LUT_BYTES);
    m.hr_thr = m.tab + CM_GUIDE_WORDS + mut_size;
    m.bars = reinterpret_cast<uint64_t *>(m.tab + core_mut_tab_words(mut_size, hr_size));
    return m;
}

// CTA prologue: mbarriers initialised, bulk copy of the constant image started (completion on
// bars[CM_WARPS * CM_STAGES]; mut_const_wait before the first table access). Ends with __syncthreads().
template <bool RNG>
__device__ __forceinline__ void mut_cta_setup(const CoreMutArgs &a, const MutSmem &m)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        for (int s = 0; s < CM_STAGES; s++) mbar_init(&m.bars[warp * CM_STAGES + s], 1);
        if (warp == 0) mbar_init(&m.bars[CM_WARPS * CM_STAGES], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (RNG && threadIdx.x == 0) {
        const uint32_t bytes = core_mut_const_bytes(a.mut_size, a.hr_nsub ? a.hr_size : 0u);
        mbar_arrive_expect_tx(&m.bars[CM_WARPS * CM_STAGES], bytes);
        bulk_g2s(m.lut, a.const_img, bytes, &m.bars[CM_WARPS * CM_STAGES]);
    }
}

__device__ __forceinline__ void mut_const_wait(const MutSmem &m) { mbar_wait(&m.bars[CM_WARPS * CM_STAGES], 0u); }

// Items [item_begin, item_end) of a column block of `blk_regs` regions starting at local region
// `blk_reg0`: item t -> row t / blk_regs, region blk_reg0 + t % blk_regs. Warp w takes
// item_begin + w + 8j. Returns when all bulk stores of the calling warp have completed.
template <bool RNG, bool DUMP>
__device__ __forceinline__ void mut_cta_items(const CoreMutArgs &a, const MutSmem &m, uint32_t item_begin,
                                              uint32_t item_end, uint32_t blk_regs, uint32_t blk_reg0)
{
    // REDUX writes a uniform register: everything a warp derives from its index (item cursor, stage and
    // mbarrier addresses) can then live in uniform registers instead of taking one register per lane
    const uint32_t warp = __reduce_max_sync(0xffffffffu, threadIdx.x >> 5);
    uint32_t lane = threadIdx.x & 31;
    asm volatile("" : "+r"(lane));          // keep it in a register (otherwise %tid.x is re-read at every use)
    const uint32_t gen_off = a.gen_dev ? __ldg(a.gen_dev) : 0u;
    const uint32_t gen = a.gen + gen_off, hr_gen = a.hr_gen + gen_off;
    uint8_t *stages = m.stages + (size_t)warp * CM_STAGES * REGION_BYTES;
    uint64_t *bars = m.bars + warp * CM_STAGES;
    const uint32_t *tab = m.tab;
    const uint32_t gw = item_begin + warp;
    if (gw >= item_end) return;
    const uint32_t n_my = (item_end - gw + CM_WARPS - 1) / CM_WARPS;
    const uint32_t d_row = CM_WARPS / blk_regs, d_reg = CM_WARPS % blk_regs;

    // parent rows are kept in registers and re-read only when an item moves on to another row (a warp
    // stays on one row for many items when the row has more regions than the CTA has warps)
#define PANSIM_CM_PARENT(r_) (a.parents ? __ldg(a.parents + (r_)) : (r_))
    // shared-space addresses, computed once and made opaque so that they stay in registers (otherwise
    // they are re-derived from %cluster_ctaid and the carve-up arithmetic at every use)
    uint32_t stages_s = smem_u32(stages), bars_s = smem_u32(bars), lut_s = smem_u32(m.lut);
    asm volatile("" : "+r"(stages_s), "+r"(bars_s), "+r"(lut_s));
    const uint32_t tab_s = lut_s + CM_LUT_BYTES, hr_thr_s = tab_s + (CM_GUIDE_WORDS + a.mut_size) * 4u;
    const uint8_t *old_blk = a.old_state + (uint64_t)blk_reg0 * REGION_BYTES;
    // TMA load of (parent row p, block region r) into stage st (lane 0)
#define PANSIM_CM_LOAD(p_, r_, st_)                                                                          \
    do {                                                                                                     \
        const uint8_t *src_ = old_blk + (uint64_t)(p_) * a.row_stride + (r_) * REGION_BYTES;                \
        const uint32_t bar_ = bars_s + (st_) * 8u;                                                           \
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_), "n"(REGION_BYTES) : "memory"); \
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" \
                     ::"r"(stages_s + (st_) * REGION_BYTES), "l"(src_), "n"(REGION_BYTES), "r"(bar_) : "memory"); \
    } while (0)

    uint32_t row = gw / blk_regs, breg = gw % blk_regs;
    uint32_t prow = PANSIM_CM_PARENT(row);          // parent of `row`
    // Two stages: the load of item j+1 is issued by item j itself, from the (row, region, parent) it computes
    // for the next item anyway. Three stages: the load side runs two items ahead with its own cursor (lane 0).
    uint32_t l_row = row, l_reg = breg, l_prow = prow, l_stage = 0;
#define PANSIM_CM_ISSUE_LOAD()                                                                               \
    do {                                                                                                     \
        PANSIM_CM_LOAD(l_prow, l_reg, l_stage);                                                              \
        l_stage = l_stage == (uint32_t)(CM_STAGES - 1) ? 0u : l_stage + 1u;                                  \
        uint32_t nr_ = l_row + d_row;                                                                        \
        l_reg += d_reg;                                                                                      \
        if (l_reg >= blk_regs) { l_reg -= blk_regs; nr_++; }                                                 \
        if (nr_ != l_row) {          /* the parent of the next row, one load ahead of its use */             \
            l_row = nr_;                                                                                     \
            if (l_row < a.n_rows) l_prow = PANSIM_CM_PARENT(l_row);                                          \
        }                                                                                                    \
    } while (0)

    if (lane == 0) {
        if (CM_LATE_LOAD) {
            PANSIM_CM_LOAD(prow, breg, 0u);
        } else {
            const uint32_t pre = min(n_my, (uint32_t)(CM_STAGES - 1));
#pragma unroll 1
            for (uint32_t jj = 0; jj < pre; jj++) PANSIM_CM_ISSUE_LOAD();
        }
    }

    if (RNG) mut_const_wait(m);
    const bool hr_on = RNG && a.hr_nsub != 0u;
    HrWindow hw_cur{0u, 0u, 0u};
    if (hr_on) hw_cur = hr_window_fetch(a, hr_gen, m.hr_thr, hr_thr_s, prow, blk_reg0 + breg, lane, 0u, 0u);
    uint32_t s = 0, par = 0;                 // stage of item j and the phase parity of its mbarrier
    for (uint32_t j = 0; j < n_my; j++) {
        uint32_t *sw = reinterpret_cast<uint32_t *>(stages + s * REGION_BYTES);     // generic pointer: ragged edge only
        const uint32_t sw_s = stages_s + s * REGION_BYTES;
        const uint32_t reg = blk_reg0 + breg;

        // RNG work that does not need the data is done before waiting for the TMA load
        const uint32_t greg = a.region0 + reg;
        const uint64_t reg_site0 = (uint64_t)greg * REGION_SITES;          // event dump only
        const uint32_t lim = greg == a.last_greg ? a.lim_last : REGION_SITES;
        const uint4 mctr = make_ctr(greg * 32u + lane, row, gen, STREAM_CORE_MUT);
        uint4 c0 = make_uint4(0, 0, 0, 0), c1 = make_uint4(0, 0, 0, 0);
        uint32_t k = 0;
        if (RNG && a.mut_nsub) {
            c0 = philox_core(mctr, a.rk);
            uint4 t = mctr;
            t.w += 1u;
            c1 = philox_core(t, a.rk);
            k = poisson_fast_s(tab_s, a.mut_kmax, c0.x);
            if (a.mut_nsub > 1) k += mut_count_extra(mctr, a.key, tab, a.mut_nsub, a.mut_kmax);
        }
        mbar_wait_s(bars_s + s * 8u, par);

        if (hr_on && hw_cur.K) {
            // ---- recombination of the previous generation on the parent's row (population.rs:725-748):
            // windows in draw order, so a later event of a cell overwrites an earlier one ----
            hr_window_apply(sw_s, hw_cur);
#pragma unroll 1
            for (uint32_t base = 32u; base < hw_cur.K; base += 32u)
                hr_window_apply(sw_s, hr_window_fetch(a, hr_gen, m.hr_thr, hr_thr_s, prow, reg, lane, base, hw_cur.K));
        }
        // the next item: its row, region and parent
        const bool more = j + 1 < n_my;
        uint32_t nrow = row + d_row, nreg = breg + d_reg;
        if (nreg >= blk_regs) { nreg -= blk_regs; nrow++; }
        const uint32_t nprow = (!more || nrow == row) ? prow : PANSIM_CM_PARENT(nrow);
        if (CM_LATE_LOAD && lane == 0 && more) {
            // issued after the recombination apply rather than before the mbarrier wait: by now the bulk store
            // of item j-1 has long left the stage item j+1 goes into, so lane 0 does not wait for it to drain
            bulk_wait_read<0>();
            PANSIM_CM_LOAD(nprow, nreg, s ^ 1u);
        }
        // first recombination window of the next item, fetched into the registers just consumed: its donor
        // loads are in flight while this item's SNP events are applied
        if (hr_on && more) hw_cur = hr_window_fetch(a, hr_gen, m.hr_thr, hr_thr_s, nprow, blk_reg0 + nreg, lane, 0u, 0u);

        if (RNG && a.mut_nsub) {
            // ---- SNP mutation (population.rs:512-539) ----
            const uint32_t kw = __reduce_max_sync(0xffffffffu, k);      // warp-uniform trip counts
            const MutChunk<DUMP> f{sw_s | (lane * 4u), lut_s, k, lane, row, lim, reg_site0, mctr, a.key, &a};
            // calls 0,1:  c0.x count | c0.y digit bytes of chunks 0-3 | c0.z digit byte of chunk 4 + 3 reserve bytes |
            //             c0.w, c1.x, c1.y, c1.z, c1.w position bytes of events 0..19
            if (kw > 0u) {
                uint32_t res = (c0.z >> 8) | 0xFF000000u;
                f.run(0u, c0.y & 255u, c0.w, res);
                if (kw > 4u) f.run(4u, (c0.y >> 8) & 255u, c1.x, res);
                if (kw > 8u) f.run(8u, (c0.y >> 16) & 255u, c1.y, res);
                if (kw > 12u) f.run(12u, c0.y >> 24, c1.z, res);
                if (kw > 16u) f.run(16u, c0.z & 255u, c1.w, res);
            }
            // later calls carry 8 events each: x = 2 digit bytes + 2 reserve bytes, y, z = position bytes
#pragma unroll 1
            for (uint32_t base = CM_GROUP0, call = 2u; base < kw; base += CM_TAIL, call++) {
                uint4 t = mctr;
                t.w += call;
                const uint4 c = philox_core(t, a.rk);
                uint32_t res = (c.x >> 16) | 0xFFFF0000u;
                f.run(base, c.x & 255u, c.y, res);
                if (kw > base + 4u) f.run(base + 4u, (c.x >> 8) & 255u, c.z, res);
            }
            // ragged last region: clear whatever the events wrote beyond the end of the alignment
            if (lim < REGION_SITES) {
#pragma unroll 1
                for (uint32_t kk = 0; kk < WORDS_PER_LANE; kk++) {
                    const uint32_t site0 = (kk * 32u + lane) * 16u;
                    const uint32_t nv = site0 >= lim ? 0u : min(16u, lim - site0);
                    if (nv < 16u) sw[kk * 32u + lane] &= (1u << (2u * nv)) - 1u;
                }
            }
        }
        if (RNG && (a.mut_nsub || hr_on)) fence_proxy_async();     // generic-proxy writes -> visible to the bulk store
        __syncwarp();

        if (lane == 0) {
            uint8_t *dst = a.new_state + (uint64_t)row * a.row_stride + (uint64_t)reg * REGION_BYTES;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(sw_s), "n"(REGION_BYTES) : "memory");
            bulk_commit();
            if (!CM_LATE_LOAD && j + CM_STAGES - 1 < n_my) {
                bulk_wait_read<1>();      // the store that last used stage (j-1)%S has left smem
                PANSIM_CM_ISSUE_LOAD();
            }
        }
        __syncwarp();
        row = nrow; breg = nreg; prow = nprow;
        if (++s == (uint32_t)CM_STAGES) { s = 0; par ^= 1u; }
    }
    if (lane == 0) bulk_wait<0>();
#undef PANSIM_CM_ISSUE_LOAD
#undef PANSIM_CM_LOAD
#undef PANSIM_CM_PARENT
}

// Stand-alone launch: CTA b covers items [b*C, (b+1)*C) of the whole shard, C = CM_WARPS*items_per_warp.
// CTAs are short-lived on purpose: SM slots turn over every few tens of microseconds, so the
// (higher-priority) accessory/selection kernels of the next generation can slip in between.
template <bool RNG, bool DUMP>
#if PANSIM_CM_MAXREG
__global__ void __maxnreg__(PANSIM_CM_MAXREG) core_mut_kernel(const CoreMutArgs a)
#else
__global__ void __launch_bounds__(CM_THREADS, CM_CTAS_PER_SM) core_mut_kernel(const CoreMutArgs a)
#endif
{
    extern __shared__ uint8_t smem_dyn[];
    const MutSmem m = mut_smem_carve(smem_dyn, a.mut_size, a.hr_nsub ? a.hr_size : 0u);
    mut_cta_setup<RNG>(a, m);
    const uint32_t total = a.n_rows * a.n_regions;
    const uint32_t cta_items = CM_WARPS * a.items_per_warp;
    const uint32_t cta_base = blockIdx.x * cta_items;
    mut_cta_items<RNG, DUMP>(a, m, cta_base, min(total, cta_base + cta_items), a.n_regions, 0u);
}

}  // namespace pansim
