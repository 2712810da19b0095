// distance.cuh -- K7: pairwise core Hamming / accessory Jaccard counts
// (population.rs:787-837 with distances.rs:22-77) on the packed layouts.
//
// Core: the reference XORs one-hot bytes and halves the popcount
// (population.rs:817) = number of differing sites. On 2-bit codes a site
// differs iff either bit of the XOR is set:
//   d = a ^ b;  m = (d | d >> 1) & 0x5555...;  differing sites = popc(m)
// The pair kernels compare the bit-plane form of the rows (core_planes_kernel),
// where the mask is one OR of two XORs. Row padding is zero in every row, so it
// never contributes.
#pragma once
#include <cuda.h>          // CUtensorMap (the encoder is fetched through cudaGetDriverEntryPoint: no libcuda link)

#include "common.cuh"

namespace pansim {

__device__ __forceinline__ uint4 ld_stream(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

constexpr int PAIR_THREADS = 256;

// Row-stationary groups. Pairs are sorted by their first row on the host (plan
// cached while the pair list is unchanged, as in the reference where the pairs are
// fixed for the whole run, main.rs:413-427). A CTA handles one group = one row i and up
// to PAIR_GROUP partner rows j: row i's words are loaded once per thread and compared
// against every partner, which almost halves the L2 traffic of one CTA per pair.
constexpr int PAIR_GROUP = 8;

struct PairGroup {
    uint32_t row_i;
    uint32_t first;      // index into the sorted partner / original-index arrays
    uint32_t count;      // 1..PAIR_GROUP
};

// Exact all-pairs mode: the pair list of a row block [row_begin, row_end) -- every (i, j) with
// i < j < N, ordered by i then j -- and its row-stationary groups are generated on the device, so
// nothing but a small offset table crosses the bus. off[r] = number of pairs of the rows before
// row_begin + r, goff[r] = number of groups before it (both with nr + 1 entries).
__device__ __forceinline__ uint32_t upper_row(const uint32_t *off, uint32_t nr, uint32_t k)
{
    uint32_t lo = 0, hi = nr;            // last r with off[r] <= k
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (off[mid] <= k) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void rows_pairs_kernel(const uint32_t *off, uint32_t nr, uint32_t row_begin, uint32_t n_pairs,
                                  uint32_t *range1, uint32_t *range2, uint32_t *partner, uint32_t *orig_index)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_pairs) return;
    const uint32_t r = upper_row(off, nr, k);
    const uint32_t i = row_begin + r, j = i + 1u + (k - off[r]);
    range1[k] = i; range2[k] = j; partner[k] = j; orig_index[k] = k;
}

// groups of the pairs (i, j) of the row block with j in [jb0, jb1): goff[r] = groups of this
// column block before row row_begin + r
__global__ void rows_groups_kernel(const uint32_t *off, const uint32_t *goff, uint32_t nr, uint32_t row_begin,
                                   uint32_t jb0, uint32_t jb1, uint32_t n_groups, PairGroup *groups)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    const uint32_t r = upper_row(goff, nr, g);
    const uint32_t i = row_begin + r;
    const uint32_t j_lo = max(i + 1u, jb0);                                      // first partner of row i in this block
    const uint32_t j = j_lo + (uint32_t)PAIR_GROUP * (g - goff[r]);
    groups[g] = PairGroup{i, off[r] + (j - (i + 1u)), min((uint32_t)PAIR_GROUP, jb1 - j)};
}

struct TileBatch {
    uint32_t block_a, block_b;         // 64-row blocks (block_a <= block_b)
    uint32_t first, count;             // range in the tile pair arrays
    uint32_t col_begin, col_end;       // column range in units of 512-byte chunks
};

// ===========================================================================
// K7 on bit planes (round 2).
//
// The XOR-popcount on 2-bit cells costs three logic operations per 32-bit word before the POPC
// ((a ^ b), >> 1, (x | s) & 0x5555...), all on the ALU pipe the POPC shares (64 lanes/clk/SM, POPC a
// quarter of that): 12 ALU slots per 32 sites, which is what bounded a row-stationary kernel on 2-bit cells at
// 4.3e7 pairs/s. A site differs iff its low bits differ OR its high bits differ, so with the low bits
// and the high bits of 32 sites in two separate words the mask is two operations:
//     m = (aL ^ bL) | (aH ^ bH)            (LOP3, LOP3)           -> 7 slots per 32 sites with the POPC
// The packed state stays 2 bits per site (the generation step writes cells); a pre-pass over the rows
// makes the plane form once per distance pass (4 logic ops per 32 sites, HBM-bound, ~0.1 ms at cfg1).
// Any bijection of the sites works as long as both planes use the same one: for the two words (w0, w1)
// of 32 sites
//     L = (w0 & 0x5555..) | ((w1 & 0x5555..) << 1)      H = ((w0 >> 1) & 0x5555..) | (w1 & 0xAAAA..)
// (site k of w0 -> bit 2k of L and H, site k of w1 -> bit 2k+1), so a 16-byte piece (64 sites) becomes
// the 16-byte piece {L01, H01, L23, H23} at the same offset: same geometry, padding stays zero.
// ===========================================================================
__global__ void __launch_bounds__(256) core_planes_kernel(const uint4 *__restrict__ state, uint4 *__restrict__ planes, uint64_t n_vec4)
{
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec4; v += (uint64_t)gridDim.x * blockDim.x) {
        const uint4 w = ld_stream(state + v);
        uint4 o;
        o.x = (w.x & 0x55555555u) | ((w.y & 0x55555555u) << 1);
        o.y = ((w.x >> 1) & 0x55555555u) | (w.y & 0xAAAAAAAAu);
        o.z = (w.z & 0x55555555u) | ((w.w & 0x55555555u) << 1);
        o.w = ((w.z >> 1) & 0x55555555u) | (w.w & 0xAAAAAAAAu);
        planes[v] = o;
    }
}

// differing sites of two 16-byte plane pieces (64 sites)
__device__ __forceinline__ uint32_t diff_planes(const uint4 a, const uint4 b)
{
    const uint32_t m0 = (a.x ^ b.x) | (a.y ^ b.y);
    const uint32_t m1 = (a.z ^ b.z) | (a.w ^ b.w);
    return __popc(m0) + __popc(m1);
}

// row-stationary groups (PairGroup) on the plane form: the sparse remainder of a
// sampled pair list and the exact all-pairs row blocks
__global__ void __launch_bounds__(PAIR_THREADS, 4) pair_planes_grouped_kernel(
    const uint8_t *planes, uint64_t row_stride, uint32_t chunk_vec4, uint32_t row_vec4, const PairGroup *groups,
    uint32_t n_groups, const uint32_t *partner, const uint32_t *orig_index, uint32_t *core_diff)
{
    __shared__ uint32_t wsum[PAIR_THREADS / 32][PAIR_GROUP];
    const uint32_t chunk = blockIdx.y;
    const uint32_t v_lo = chunk * chunk_vec4;
    const uint32_t v_hi = min(row_vec4, v_lo + chunk_vec4);
    for (uint32_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const PairGroup grp = groups[g];
        const uint4 *ra = reinterpret_cast<const uint4 *>(planes + (uint64_t)grp.row_i * row_stride);
        const uint4 *rb[PAIR_GROUP];
#pragma unroll
        for (int q = 0; q < PAIR_GROUP; q++) {
            const uint32_t j = partner[grp.first + (q < (int)grp.count ? q : 0)];
            rb[q] = reinterpret_cast<const uint4 *>(planes + (uint64_t)j * row_stride);
        }
        // carry-save counting as in the tile kernel: `ones` absorbs the two masks of a piece, the carries are POPCounted
        uint32_t acc[PAIR_GROUP], ones[PAIR_GROUP];
#pragma unroll
        for (int q = 0; q < PAIR_GROUP; q++) { acc[q] = 0; ones[q] = 0; }
        for (uint32_t v = v_lo + threadIdx.x; v < v_hi; v += PAIR_THREADS) {
            const uint4 a = ld_stream(ra + v);
            uint4 b[PAIR_GROUP];
#pragma unroll
            for (int q = 0; q < PAIR_GROUP; q++) b[q] = ld_stream(rb[q] + v);
#pragma unroll
            for (int q = 0; q < PAIR_GROUP; q++) {
                const uint32_t m0 = (a.x ^ b[q].x) | (a.y ^ b[q].y);
                const uint32_t m1 = (a.z ^ b[q].z) | (a.w ^ b[q].w);
                const uint32_t o = ones[q];
                ones[q] = o ^ m0 ^ m1;
                acc[q] += __popc((o & m0) | (m1 & (o | m0)));
            }
        }
#pragma unroll
        for (int q = 0; q < PAIR_GROUP; q++) {
            acc[q] = 2u * acc[q] + __popc(ones[q]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
        }
        if ((threadIdx.x & 31) == 0) {
#pragma unroll
            for (int q = 0; q < PAIR_GROUP; q++) wsum[threadIdx.x >> 5][q] = acc[q];
        }
        __syncthreads();
        if (threadIdx.x < grp.count) {
            uint32_t t = 0;
            for (int w = 0; w < PAIR_THREADS / 32; w++) t += wsum[w][threadIdx.x];
            atomicAdd(&core_diff[orig_index[grp.first + threadIdx.x]], t);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// TMA-staged shared-memory tiles (north_star: "128-bit vectorised XOR/popcount over TMA-staged
// shared-memory tiles"). The host buckets the pairs by the pair of 64-row blocks their endpoints fall
// in and cuts every bucket into batches of up to T2_BATCH pairs. A work item = (batch, column range).
// Persistent CTAs (one per SM) take work items from a counter. Per 512-byte column chunk one elected
// producer thread issues TWO instructions -- cp.async.bulk.tensor.2d with a 64-row x 512-byte box per
// row block, mbarrier complete_tx -- into a 3-stage ring (3 x 64 KB); fifteen consumer warps wait on
// the stage's `full` barrier, each compares its pairs (one 16-byte piece per lane per row, first row
// kept in registers while it repeats) and arrives on the stage's `empty` barrier. Every staged row
// serves all pairs of the batch that touch it (~6 at cfg1), which takes the L2 -> SM traffic from
// 337 KB to ~50 KB per pair; DRAM sees each row about once per pass because the work items of one
// column range run at the same time on all SMs.
// ---------------------------------------------------------------------------
constexpr int T2_BLOCK_ROWS = 64;
constexpr int T2_CHUNK_BYTES = 512;
constexpr int T2_STAGES = 3;
constexpr int T2_WARPS = 15;                        // consumer warps (+ the producer warp = 512 threads: 128 registers each)
constexpr int T2_THREADS = (T2_WARPS + 1) * 32;     // + one producer warp
constexpr int T2_PPW = 20;                          // pairs per consumer warp
constexpr int T2_BATCH = T2_WARPS * T2_PPW;         // 300
constexpr uint32_t T2_STAGE_BYTES = 2 * T2_BLOCK_ROWS * T2_CHUNK_BYTES;   // 65536

static inline size_t tile2_smem_bytes()
{
    return 1024 /* alignment slack */ + (size_t)T2_STAGES * T2_STAGE_BYTES + 2 * T2_STAGES * sizeof(uint64_t) + T2_BATCH * sizeof(uint32_t) + 16;
}

__device__ __forceinline__ void tma_load_2d(void *smem_dst, const void *tmap, uint32_t x, uint32_t y, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(T2_THREADS, 1) pair_tile2_kernel(
    const __grid_constant__ CUtensorMap tmap, const TileBatch *batches, uint32_t n_work, uint32_t *work_counter,
    const uint16_t *tile_slots, const uint32_t *tile_orig, uint32_t *core_diff)
{
    extern __shared__ uint8_t t2_raw[];
    uint8_t *base = t2_raw + ((1024u - (smem_u32(t2_raw) & 1023u)) & 1023u);      // TMA destinations: 128-byte aligned at least
    uint8_t *stages = base;
    uint64_t *full = reinterpret_cast<uint64_t *>(base + (size_t)T2_STAGES * T2_STAGE_BYTES);
    uint64_t *empty = full + T2_STAGES;
    uint32_t *meta = reinterpret_cast<uint32_t *>(empty + T2_STAGES);
    uint32_t *work_s = meta + T2_BATCH;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < T2_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], T2_WARPS); }
        fence_mbar_init();
    }
    __syncthreads();

    uint32_t it = 0;                 // chunks handled so far by this CTA (all work items): stage = it % 3, phase = (it / 3) & 1
    for (;;) {
        if (threadIdx.x == 0) *work_s = atomicAdd(work_counter, 1u);
        __syncthreads();
        const uint32_t w = *work_s;
        if (w >= n_work) break;
        const TileBatch bt = batches[w];
        const uint32_t n_chunks = bt.col_end - bt.col_begin;
        const bool diag = bt.block_a == bt.block_b;
        for (uint32_t i = threadIdx.x; i < (uint32_t)T2_BATCH; i += T2_THREADS)
            meta[i] = i < bt.count ? (uint32_t)tile_slots[bt.first + i] : 0xFFFFu;
        __syncthreads();

        if (warp == T2_WARPS) {
            // ---- producer: one elected thread ----
            if (lane == 0) {
                for (uint32_t c = 0; c < n_chunks; c++) {
                    const uint32_t k = it + c, s = k % T2_STAGES, ph = (k / T2_STAGES) & 1u;
                    mbar_wait(&empty[s], ph ^ 1u);                      // all consumer warps have left the stage (fresh barrier: passes)
                    mbar_arrive_expect_tx(&full[s], diag ? T2_STAGE_BYTES / 2 : T2_STAGE_BYTES);
                    uint8_t *dst = stages + (size_t)s * T2_STAGE_BYTES;
                    const uint32_t x = (bt.col_begin + c) * (T2_CHUNK_BYTES / 4);
                    tma_load_2d(dst, &tmap, x, bt.block_a * T2_BLOCK_ROWS, &full[s]);
                    if (!diag) tma_load_2d(dst + T2_STAGE_BYTES / 2, &tmap, x, bt.block_b * T2_BLOCK_ROWS, &full[s]);
                }
            }
        } else {
            // ---- consumers: pairs [warp * PPW, warp * PPW + PPW) of the batch ----
            // Branch-free over the PPW slots of the warp (a slot without a pair compares row slot 0 with
            // itself and is not written back), so the shared-memory loads of later pairs are issued
            // while earlier ones are being counted. offb[q] = byte offset of the second row's piece in a
            // stage; the first row's offsets are packed two per register and read only where the first
            // row changes (`reload`, warp-uniform: the pairs of a batch are sorted by first row).
            // Counting is carry-save: per pair one `ones` word absorbs the two 32-site masks of a chunk,
            // only the carries are POPCounted (weight 2), so a chunk costs one POPC per pair instead of two.
            uint32_t offb[T2_PPW], offa2[T2_PPW / 2];
            uint32_t acc[T2_PPW], ones[T2_PPW];
            uint32_t reload = 0;
            {
                uint32_t prev = 0xFFFFFFFFu;
#pragma unroll
                for (int q = 0; q < T2_PPW; q++) {
                    uint32_t m = meta[warp * T2_PPW + q];
                    if (m == 0xFFFFu) m = 0u;
                    const uint32_t sa = m & 0xFFu, sb = (m >> 8) & 0xFFu;
                    offb[q] = sb * T2_CHUNK_BYTES + lane * 16u;
                    const uint32_t oa = sa * T2_CHUNK_BYTES + lane * 16u;                 // < 65536
                    if (q & 1) offa2[q >> 1] |= oa << 16; else offa2[q >> 1] = oa;
                    acc[q] = 0; ones[q] = 0;
                    if (sa != prev) reload |= 1u << q;
                    prev = sa;
                }
            }
            for (uint32_t c = 0; c < n_chunks; c++) {
                const uint32_t k = it + c, s = k % T2_STAGES, ph = (k / T2_STAGES) & 1u;
                mbar_wait(&full[s], ph);
                const uint32_t st_s = smem_u32(stages) + s * T2_STAGE_BYTES;
                uint4 a = make_uint4(0, 0, 0, 0);
#pragma unroll
                for (int q = 0; q < T2_PPW; q++) {
                    uint4 b;
                    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "r"(st_s + offb[q]));
                    if ((reload >> q) & 1u) {
                        const uint32_t oa = (q & 1) ? (offa2[q >> 1] >> 16) : (offa2[q >> 1] & 0xFFFFu);
                        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w) : "r"(st_s + oa));
                    }
                    const uint32_t m0 = (a.x ^ b.x) | (a.y ^ b.y);
                    const uint32_t m1 = (a.z ^ b.z) | (a.w ^ b.w);
                    const uint32_t o = ones[q];
                    ones[q] = o ^ m0 ^ m1;
                    acc[q] += __popc((o & m0) | (m1 & (o | m0)));       // carries of the three-input add
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
            }
#pragma unroll
            for (int q = 0; q < T2_PPW; q++) {
                uint32_t v = 2u * acc[q] + __popc(ones[q]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                const uint32_t idx = warp * T2_PPW + q;
                if (lane == 0 && idx < bt.count) atomicAdd(&core_diff[tile_orig[bt.first + idx]], v);
            }
        }
        it += n_chunks;
        __syncthreads();                 // meta[] and *work_s are rewritten by the next work item
    }
}

// accessory: one warp per pair; intersection and union popcounts (distances.rs:62-68)
__global__ void __launch_bounds__(256) pair_acc_kernel(const uint32_t *acc, uint32_t stride_words,
                                                       uint32_t n_words, const uint32_t *range1,
                                                       const uint32_t *range2, uint32_t n_pairs,
                                                       uint32_t *inter, uint32_t *uni)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t wpb = blockDim.x >> 5;
    for (uint32_t p = blockIdx.x * wpb + (threadIdx.x >> 5); p < n_pairs; p += gridDim.x * wpb) {
        const uint32_t *ra = acc + (uint64_t)range1[p] * stride_words;
        const uint32_t *rb = acc + (uint64_t)range2[p] * stride_words;
        uint32_t in = 0, un = 0;
        for (uint32_t w = lane; w < n_words; w += 32) {
            const uint32_t x = ra[w], y = rb[w];
            in += __popc(x & y);
            un += __popc(x | y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            in += __shfl_xor_sync(0xffffffffu, in, o);
            un += __shfl_xor_sync(0xffffffffu, un, o);
        }
        if (lane == 0) {
            if (inter) inter[p] = in;
            if (uni) uni[p] = un;
        }
    }
}

// --print_dist statistics (main.rs:502-519): standard_deviation (population.rs:87-94) of the two
// distance vectors of one pass, on the device, so 32 bytes leave the GPU per generation instead of
// the three count vectors. The reference sums with `iter().sum::<f64>()`, i.e. strictly left to
// right, and the result is printed with 17 significant digits, so the summation ORDER is part of
// the result: each of the four sums (two means, then two sums of squared deviations) is one chain
// of dependent f64 additions made by a single thread in index order. Everything that is not the
// chain -- the divisions of population.rs:822 / :828-830, x - mean, the square -- is done by a
// producer warp one 1024-element chunk ahead, through shared memory. No fused multiply-add can
// form: the products are rounded into shared memory before they are added (Rust has no contraction).
// out[4] = { avg_core, std_core, avg_acc, std_acc } (the column order of _per_gen.tsv, main.rs:546).
constexpr int STATS_CHUNK = 1024;
constexpr int STATS_PROD_WARPS = 4;     // producer warps per vector: a chunk is 8 loads deep per lane, well under the chain's 8.4k cycles
constexpr int STATS_THREADS = (2 * STATS_PROD_WARPS + 2) * 32;   // warps 0-3: core producers, 4-7: accessory producers, 8: core chain, 9: accessory chain

struct PairStatsArgs {
    const uint32_t *core_diff, *inter, *uni;
    uint32_t n_pairs;
    double core_size, core_genes;
    double *out;
};

__global__ void __launch_bounds__(STATS_THREADS) pair_stats_kernel(const PairStatsArgs a)
{
    __shared__ double buf[2][2][STATS_CHUNK];      // [vector][stage][element]
    __shared__ double mean_s[2];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool producer = warp < 2u * STATS_PROD_WARPS;
    const uint32_t vec = producer ? warp / STATS_PROD_WARPS : warp - 2u * STATS_PROD_WARPS;     // 0 = core distances, 1 = accessory distances
    const uint32_t plane = (warp % STATS_PROD_WARPS) * 32u + lane;                               // producer lane within its vector
    const uint32_t n = a.n_pairs;
    const uint32_t n_chunks = (n + STATS_CHUNK - 1) / STATS_CHUNK;
    const double dn = (double)n;

    auto produce = [&](uint32_t c, int pass, double mean) {
        double *dst = buf[vec][c & 1u];
        const uint32_t k0 = c * STATS_CHUNK, k1 = min(n, k0 + STATS_CHUNK);
#pragma unroll 4
        for (uint32_t k = k0 + plane; k < k1; k += 32u * STATS_PROD_WARPS) {
            double d;
            if (vec == 0) {
                d = __ddiv_rn((double)a.core_diff[k], a.core_size);                                          // population.rs:822
            } else {
                const double num = __dadd_rn((double)a.inter[k], a.core_genes), den = __dadd_rn((double)a.uni[k], a.core_genes);
                d = __dsub_rn(1.0, __ddiv_rn(num, den));                                                     // :828-830
            }
            if (pass == 1) {
                const double diff = __dsub_rn(d, mean);                                                      // :90
                d = __dmul_rn(diff, diff);
            }
            dst[k - k0] = d;
        }
    };

    double sum = 0.0;
    for (int pass = 0; pass < 2; pass++) {
        const double mean = pass ? mean_s[vec] : 0.0;
        if (producer && n_chunks) produce(0, pass, mean);
        __syncthreads();
        sum = 0.0;
        for (uint32_t c = 0; c < n_chunks; c++) {
            if (producer) {
                if (c + 1 < n_chunks) produce(c + 1, pass, mean);
            } else if (lane == 0) {
                const double *src = buf[vec][c & 1u];
                const uint32_t len = min((uint32_t)STATS_CHUNK, n - c * STATS_CHUNK);
                // the chain: one dependent DADD per element (8.2 cycles each); the shared-memory loads of the
                // next eight elements are issued before the current eight are added, so only the adds remain
                uint32_t i = 0;
                if (len >= 8) {
                    double v[8], w[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) v[j] = src[j];
                    for (i = 8; i + 8 <= len; i += 8) {
#pragma unroll
                        for (int j = 0; j < 8; j++) w[j] = src[i + j];
#pragma unroll
                        for (int j = 0; j < 8; j++) sum = __dadd_rn(sum, v[j]);
#pragma unroll
                        for (int j = 0; j < 8; j++) v[j] = w[j];
                    }
#pragma unroll
                    for (int j = 0; j < 8; j++) sum = __dadd_rn(sum, v[j]);
                }
                for (; i < len; i++) sum = __dadd_rn(sum, src[i]);
            }
            __syncthreads();
        }
        if (!producer && lane == 0) {
            if (pass == 0) {
                const double mean0 = __ddiv_rn(sum, dn);                                                     // :83-85
                mean_s[vec] = mean0;
                a.out[vec * 2] = mean0;
            } else {
                a.out[vec * 2 + 1] = __dsqrt_rn(__ddiv_rn(sum, dn));                                         // :92-93
            }
        }
        __syncthreads();
    }
}

}  // namespace pansim
