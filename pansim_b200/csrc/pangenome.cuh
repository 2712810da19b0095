// pangenome.cuh -- pangenome accumulation curves and the gene frequency spectrum (DESIGN.md section 16).
//
// Order draw: pg_order_kernel draws P permutations of the N rows by Fisher-Yates, one CTA per order. The N - 1
// swap indices j_i do not depend on the swaps, so the threads draw them in parallel (Philox4x32-10, counter
// {i, p, 0, PG_ORDER_TAG}); thread 0 then runs the swap chain. The order and the indices live in shared memory when
// 8 N bytes fit, otherwise in global memory (the same code on other pointers, so the orders do not depend on it).
//
// Walk: per order, the rows are visited in order and every thread keeps three bit sets of one accessory word in
// registers: S1 (seen in >= 1 row), S2 (seen in >= 2 rows), C (seen in every row). Per step and word x:
//   new += popc(x & ~S1), lost core += popc(C & ~x) (not at step 1), left unique += popc(x & S1 & ~S2),
// then S2 |= S1 & x, S1 |= x, C &= x. A warp sums the three counts of a step with two redux.sync (new and lost core
// packed in 16-bit halves), lane s keeps step s of a batch of 32, and after each batch the CTA adds its warps'
// sums in shared memory and makes one integer atomic per (order, step, count) that is not zero. Grid: word slices of
// 128 words x row chunks x orders. With one chunk each CTA walks every step. With more (too few CTAs to fill the
// SMs), pg_summary_kernel first forms each chunk's (S1, S2, C), and a walking CTA combines the summaries of the
// chunks before its own into its incoming state:
//   S1 = a.S1 | b.S1, S2 = a.S2 | b.S2 | (a.S1 & b.S1), C = a.C & b.C.
// Row words are loaded 32 steps at a time (the 32 row indices of a batch are one coalesced load, broadcast by
// shuffles), all 32 loads in flight before the batch is processed. Bits at or past G are masked off.
//
// Curves: pg_curves_kernel scans each order's deltas over k (one CTA per order, tiles of 256 steps) into
// pan = c0 + sum new, core = c0 + new(1) - sum lost, new (+ c0 at k = 1), unique = sum new - sum left (+ c0 at
// k = 1). Everything is an integer: the grid, the chunking and the shard count change no bit.
//
// Spectrum: pg_spectrum_kernel bins the presence counts of acc_gene_counts_kernel (K8), one atomic per distinct
// count of a warp.
#pragma once
#include "common.cuh"

namespace pansim {

// Counter word 3 of the order draw (PANSIM_GENE_ACC_ORDER_TAG). The simulation's streams use (stream << 16) | q with
// stream <= 8 and q < 2^16 (common.cuh, core_mut.cuh, core_hr.cuh, acc_step.cuh, select.cuh: below 0x00090000) and
// 0x01000000 + e for the recombination events of core_hr.cuh; this word is neither.
constexpr uint32_t PG_ORDER_TAG = 0x00A00000u;
constexpr uint32_t PG_ORDER_THREADS = 256;
constexpr uint32_t PG_WARPS = 4;                       // walk / summary CTA: one word per thread
constexpr uint32_t PG_SLICE_WORDS = PG_WARPS * 32;     // words per CTA
constexpr uint32_t PG_BATCH = 32;                      // steps per batch (one per lane)
constexpr uint32_t PG_SCAN_THREADS = 256;
constexpr uint32_t PG_STATS = 3;                       // deltas per step: new, lost core, left unique

struct PgOrderArgs {
    PhiloxKeys rk;                  // key (lo32(seed), hi32(seed))
    uint32_t n_rows;
    uint32_t *orders;               // [P][n_rows]
    uint32_t *scratch;              // [P][n_rows] swap indices (global path only)
};

__device__ __forceinline__ uint32_t pg_swap_index(const PhiloxKeys &rk, uint32_t i, uint32_t p)
{
    const uint4 r = philox4x32_10(make_uint4(i, p, 0u, PG_ORDER_TAG), rk);
    return (uint32_t)(((uint64_t)r.x * (i + 1u)) >> 32);
}

template <bool SMEM>
__global__ void __launch_bounds__(PG_ORDER_THREADS) pg_order_kernel(PgOrderArgs a)
{
    extern __shared__ uint32_t s_ord[];
    const uint32_t n = a.n_rows, p = blockIdx.x;
    uint32_t *o = SMEM ? s_ord : a.orders + (size_t)p * n;
    uint32_t *js = SMEM ? s_ord + n : a.scratch + (size_t)p * n;
    for (uint32_t i = threadIdx.x; i < n; i += PG_ORDER_THREADS) {
        o[i] = i;
        if (i) js[i] = pg_swap_index(a.rk, i, p);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t *__restrict__ jr = js;
        for (uint32_t i = n - 1; i >= 1 && i < n; i--) {
            const uint32_t j = jr[i];
            const uint32_t t = o[i];
            o[i] = o[j];
            o[j] = t;
        }
    }
    if (SMEM) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n; i += PG_ORDER_THREADS) a.orders[(size_t)p * n + i] = o[i];
    }
}

struct PgWalkArgs {
    const uint32_t *state;          // accessory rows
    uint32_t stride_words, n_words, n_genes, n_rows;
    const uint32_t *orders;         // [P][n_rows]
    uint32_t chunk_rows, n_chunks;  // steps per chunk (a multiple of PG_BATCH), chunks per order
    uint32_t *summary;              // [P][n_chunks][3][n_words]: S1, S2, C of each chunk (n_chunks > 1)
    uint32_t *delta;                // [P][n_rows][3]: new, lost core, left unique of each step (zeroed)
};

// valid gene bits of word w: padding past G and words past the row are never counted
__device__ __forceinline__ uint32_t pg_word_mask(const PgWalkArgs &a, uint32_t w)
{
    if (w >= a.n_words) return 0u;
    const uint32_t rem = a.n_genes & 31u;
    return (w == a.n_words - 1 && rem) ? (1u << rem) - 1u : ~0u;
}

// word w of the rows of steps k0 .. k0 + 31 (0 at or past k1)
__device__ __forceinline__ void pg_load_batch(const PgWalkArgs &a, const uint32_t *ord, uint32_t k0, uint32_t k1, uint32_t w,
                                              uint32_t mask, uint32_t lane, uint32_t (&x)[PG_BATCH])
{
    const uint32_t idx = k0 + lane < k1 ? __ldg(ord + k0 + lane) : 0u;
#pragma unroll
    for (uint32_t s = 0; s < PG_BATCH; s++) {
        const uint32_t r = __shfl_sync(0xffffffffu, idx, s);
        x[s] = (mask && k0 + s < k1) ? __ldg(a.state + (uint64_t)r * a.stride_words + w) & mask : 0u;
    }
}

// (S1, S2, C) of the rows of chunk blockIdx.y (grid.y = n_chunks - 1: the last chunk's summary is never read)
__global__ void __launch_bounds__(PG_SLICE_WORDS) pg_summary_kernel(PgWalkArgs a)
{
    const uint32_t lane = threadIdx.x & 31u, w = blockIdx.x * PG_SLICE_WORDS + threadIdx.x;
    const uint32_t chunk = blockIdx.y, p = blockIdx.z;
    const uint32_t k_begin = chunk * a.chunk_rows, k_end = min(a.n_rows, k_begin + a.chunk_rows);
    const uint32_t mask = pg_word_mask(a, w);
    const uint32_t *ord = a.orders + (size_t)p * a.n_rows;
    uint32_t S1 = 0u, S2 = 0u, C = mask;
#pragma unroll 1
    for (uint32_t k0 = k_begin; k0 < k_end; k0 += PG_BATCH) {
        uint32_t x[PG_BATCH];
        pg_load_batch(a, ord, k0, k_end, w, mask, lane, x);
#pragma unroll
        for (uint32_t s = 0; s < PG_BATCH; s++) {
            if (k0 + s < k_end) {
                S2 |= S1 & x[s];
                S1 |= x[s];
                C &= x[s];
            }
        }
    }
    if (w < a.n_words) {
        uint32_t *sm = a.summary + ((size_t)p * a.n_chunks + chunk) * 3 * a.n_words + w;
        sm[0] = S1;
        sm[a.n_words] = S2;
        sm[2 * (size_t)a.n_words] = C;
    }
}

__global__ void __launch_bounds__(PG_SLICE_WORDS) pg_walk_kernel(PgWalkArgs a)
{
    __shared__ uint32_t s_red[2][PG_WARPS][2][32];      // double-buffered by batch parity
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, w = blockIdx.x * PG_SLICE_WORDS + threadIdx.x;
    const uint32_t chunk = blockIdx.y, p = blockIdx.z;
    const uint32_t k_begin = chunk * a.chunk_rows, k_end = min(a.n_rows, k_begin + a.chunk_rows);
    const uint32_t mask = pg_word_mask(a, w);
    // incoming state: the summaries of the chunks before this one, combined in order (C is set at step 0)
    uint32_t S1 = 0u, S2 = 0u, C = chunk ? mask : 0u;
    if (mask) {
        const uint32_t *sm = a.summary + (size_t)p * a.n_chunks * 3 * a.n_words + w;
        for (uint32_t q = 0; q < chunk; q++, sm += 3 * (size_t)a.n_words) {
            const uint32_t s1 = __ldg(sm), s2 = __ldg(sm + a.n_words), c = __ldg(sm + 2 * (size_t)a.n_words);
            S2 |= s2 | (S1 & s1);
            S1 |= s1;
            C &= c;
        }
    }
    const uint32_t *ord = a.orders + (size_t)p * a.n_rows;
    uint32_t *delta = a.delta + (size_t)p * a.n_rows * PG_STATS;
    uint32_t buf = 0;
#pragma unroll 1
    for (uint32_t k0 = k_begin; k0 < k_end; k0 += PG_BATCH, buf ^= 1u) {
        uint32_t x[PG_BATCH];
        pg_load_batch(a, ord, k0, k_end, w, mask, lane, x);
        uint32_t keep_nl = 0u, keep_u = 0u;
#pragma unroll
        for (uint32_t s = 0; s < PG_BATCH; s++) {
            const uint32_t k = k0 + s;
            if (k < k_end) {                                // uniform over the CTA
                const uint32_t nw = __popc(x[s] & ~S1), ls = k ? __popc(C & ~x[s]) : 0u, lu = __popc(x[s] & S1 & ~S2);
                S2 |= S1 & x[s];
                S1 |= x[s];
                C = k ? C & x[s] : x[s];
                // per warp at most 32 x 32 = 1 024 per count: new and lost core share one word
                const uint32_t nl = __reduce_add_sync(0xffffffffu, nw | ls << 16), u = __reduce_add_sync(0xffffffffu, lu);
                if (lane == s) { keep_nl = nl; keep_u = u; }
            }
        }
        s_red[buf][warp][0][lane] = keep_nl;
        s_red[buf][warp][1][lane] = keep_u;
        __syncthreads();
        if (warp == 0 && k0 + lane < k_end) {
            uint32_t n = 0u, l = 0u, u = 0u;
#pragma unroll
            for (uint32_t q = 0; q < PG_WARPS; q++) {
                const uint32_t v = s_red[buf][q][0][lane];
                n += v & 0xFFFFu;
                l += v >> 16;
                u += s_red[buf][q][1][lane];
            }
            uint32_t *d = delta + (size_t)(k0 + lane) * PG_STATS;
            if (n) atomicAdd(d, n);
            if (l) atomicAdd(d + 1, l);
            if (u) atomicAdd(d + 2, u);
        }
        // the next batch writes the other buffer; the one after it passes the barrier above only once warp 0 is done
    }
}

struct PgCurveArgs {
    const uint32_t *delta;          // [P][n_rows][3]
    uint32_t n_rows, c0;
    uint32_t *pan, *core, *new_genes, *unique;   // [P][n_rows] each
};

// inclusive sums over the CTA of three counts per thread; *tot = the CTA's totals
__device__ __forceinline__ void pg_block_scan3(uint32_t (&v)[3], uint32_t (&tot)[3], uint32_t (*s_warp)[PG_SCAN_THREADS / 32])
{
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 3; q++) {
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, v[q], d);
            if (lane >= d) v[q] += t;
        }
        if (lane == 31) s_warp[q][warp] = v[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 3; q++) {
        uint32_t before = 0u, all = 0u;
#pragma unroll
        for (uint32_t j = 0; j < PG_SCAN_THREADS / 32; j++) {
            const uint32_t t = s_warp[q][j];
            before += j < warp ? t : 0u;
            all += t;
        }
        v[q] += before;
        tot[q] = all;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(PG_SCAN_THREADS) pg_curves_kernel(PgCurveArgs a)
{
    __shared__ uint32_t s_warp[3][PG_SCAN_THREADS / 32];
    const uint32_t n = a.n_rows, p = blockIdx.x;
    const uint32_t *d = a.delta + (size_t)p * n * PG_STATS;
    const uint32_t first_new = __ldg(d);
    uint32_t carry[3] = {0u, 0u, 0u};
    for (uint32_t k0 = 0; k0 < n; k0 += PG_SCAN_THREADS) {
        const uint32_t k = k0 + threadIdx.x;
        uint32_t v[3] = {0u, 0u, 0u}, tot[3];
        if (k < n) {
            v[0] = __ldg(d + (size_t)k * PG_STATS);
            v[1] = __ldg(d + (size_t)k * PG_STATS + 1);
            v[2] = __ldg(d + (size_t)k * PG_STATS + 2);
        }
        const uint32_t nw = v[0];
        pg_block_scan3(v, tot, s_warp);
        if (k < n) {
            const uint32_t sum_new = carry[0] + v[0], sum_lost = carry[1] + v[1], sum_left = carry[2] + v[2];
            const uint32_t first = k == 0 ? a.c0 : 0u;
            const size_t o = (size_t)p * n + k;
            a.pan[o] = a.c0 + sum_new;
            a.core[o] = a.c0 + first_new - sum_lost;
            a.new_genes[o] = nw + first;
            a.unique[o] = sum_new - sum_left + first;
        }
#pragma unroll
        for (int q = 0; q < 3; q++) carry[q] += tot[q];
    }
}

// spectrum[a_g] += 1 for every gene (spectrum zeroed, [n_rows + 1]); lanes with the same count add once
__global__ void __launch_bounds__(256) pg_spectrum_kernel(const uint32_t *counts, uint32_t n_genes, unsigned long long *spectrum)
{
    const uint32_t g = blockIdx.x * 256u + threadIdx.x;
    const uint32_t c = g < n_genes ? __ldg(counts + g) : 0xFFFFFFFFu;
    const uint32_t peers = __match_any_sync(0xffffffffu, c);
    if (g < n_genes && (threadIdx.x & 31u) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(spectrum + c, (unsigned long long)__popc(peers));
}

}  // namespace pansim
