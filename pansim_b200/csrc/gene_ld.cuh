// gene_ld.cuh -- linkage of the accessory genes: r^2, associated, dissociated and four-gamete gene pairs by
// compartment class, the joint presence counts of gene pairs on the tensor cores (DESIGN.md section 15).
//
// Gene pass: from the per-gene presence counts a (acc_gene_counts_kernel, K8), gene_ld_mark_kernel counts the used
// genes of every 2048-gene block (min_minor <= min(a, n - a)); vcf_scan_blocks_kernel scans the block totals, and
// gene_ld_compact_kernel gives every used gene its compact index (rank, ascending gene order) and writes a,
// inv = 1 / (a (n - a)) and its group (1 = the second compartment). Integer scans: deterministic.
//
// Transpose: gene_ld_transpose_kernel turns the accessory rows (one bit per gene) into gene-major bit rows X[k][kw]
// of the used genes (bit r of row k: row r carries used gene k), kw = ld_row_words(n), zero past row n. A warp owns
// one accessory word (32 genes) and 64 rows: a lane loads one row's word, and 32 __ballot_sync give each gene's
// 32 row bits.
//
// Pair kernel: all tile pairs I <= J over tiles of 128 used genes, the tile pair of a CTA found by binary search
// over the closed form of ld_pair_kernel's tile-pair offsets (tile I pairs with every J >= I). The operand pipeline
// of bitmma.cuh (u8 expansion, tcgen05.mma.kind::i8, tcgen05.ld) puts c = the rows carrying both genes in tensor
// memory. The epilogue forms D, r^2 and q per pair and keeps the class totals in registers while the
// class does not change along a thread's columns (groups are one contiguous gene range, so at most twice), then in
// shared memory; the r^2 histogram is counted in shared u32 counters. At CTA exit both go to global u64 counters
// (r^2 as a 128-bit sum).
#pragma once
#include "common.cuh"
#include "ld.cuh"

namespace pansim {

constexpr uint32_t GL_MAX_BINS = 1024;                  // largest r2_bins
constexpr uint32_t GL_CLASS_WORDS = 6;                  // pansim_gene_ld_class: pairs, four_gamete, r2_hi, r2_lo, associated, dissociated
constexpr uint32_t GL_OUT_CLASSES = 3 * GL_CLASS_WORDS; // output words before the histogram
constexpr uint32_t GT_WARPS = 8;                        // transpose: warps per CTA, 64 rows each

struct GeneLdArgs {
    const uint32_t *counts;         // [n_genes] rows carrying each gene
    uint32_t n_genes, n_rows, min_minor;
    uint32_t lo1, hi1;              // genes of group 1: [lo1, hi1) (empty unless there are two compartments)
    unsigned long long *block;      // [n_blocks + 1] used genes per block, then their exclusive scan (+ total)
    uint32_t *rank;                 // [n_genes] compact index of a used gene, ~0u otherwise
    uint32_t *a, *grp;              // [used] presence count, group
    double *inv;                    // [used] 1 / (a (n - a))
    unsigned long long *used1;      // used genes of group 1
};

__device__ __forceinline__ bool gene_ld_used(const GeneLdArgs &a, uint32_t g)
{
    const uint32_t c = a.counts[g];
    return a.min_minor <= min(c, a.n_rows - c);
}

// used genes per block; thread t of block b takes genes b*VS_SITES + 8t .. 8t+7
__global__ void __launch_bounds__(VS_THREADS) gene_ld_mark_kernel(GeneLdArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t g0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    unsigned long long used = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++)
        if (g0 + i < a.n_genes && gene_ld_used(a, (uint32_t)(g0 + i))) used++;
    unsigned long long total;
    vcf_block_scan(used, s_warp, &total);
    if (threadIdx.x == 0) a.block[blockIdx.x] = total;
}

// rank, presence count, inverse and group of every used gene (block base + scan inside the block)
__global__ void __launch_bounds__(VS_THREADS) gene_ld_compact_kernel(GeneLdArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t g0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    uint32_t used = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++)
        if (g0 + i < a.n_genes && gene_ld_used(a, (uint32_t)(g0 + i))) used |= 1u << i;
    unsigned long long total;
    uint32_t k = (uint32_t)(a.block[blockIdx.x] + vcf_block_scan(__popc(used), s_warp, &total));
    uint32_t used1 = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        const uint64_t g = g0 + i;
        if (g >= a.n_genes) break;
        if (used >> i & 1u) {
            const uint32_t c = a.counts[g];
            const uint32_t grp = g >= a.lo1 && g < a.hi1 ? 1u : 0u;
            a.rank[g] = k;
            a.a[k] = c;
            a.grp[k] = grp;
            a.inv[k] = __ddiv_rn(1.0, (double)((unsigned long long)c * (a.n_rows - c)));
            used1 += grp;
            k++;
        } else {
            a.rank[g] = ~0u;
        }
    }
    used1 = __reduce_add_sync(~0u, used1);
    if ((threadIdx.x & 31u) == 0 && used1) atomicAdd(a.used1, (unsigned long long)used1);
}

struct GeneLdTransposeArgs {
    const uint32_t *state;          // accessory rows, bit g & 31 of word g >> 5 = gene g
    uint32_t stride_words;          // row pitch
    uint32_t n_rows, n_genes;
    const uint32_t *rank;
    uint32_t kw;                    // words per row of x
    uint32_t *x;                    // [used][kw]
};

// grid: x = accessory words, y = blocks of GT_WARPS * 64 rows covering kw * 32 rows
__global__ void __launch_bounds__(GT_WARPS * 32) gene_ld_transpose_kernel(GeneLdTransposeArgs a)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t w = blockIdx.x;
    const uint32_t xw = (blockIdx.y * GT_WARPS + warp) * 2u;          // the warp's two words of x (kw is even)
    if (xw >= a.kw) return;
    const uint32_t g = w * 32u + lane;
    const uint32_t k = g < a.n_genes ? a.rank[g] : ~0u;
    if (!__ballot_sync(~0u, k != ~0u)) return;
    uint32_t out[2];
#pragma unroll
    for (uint32_t h = 0; h < 2; h++) {
        const uint32_t r = (xw + h) * 32u + lane;
        const uint32_t v = r < a.n_rows ? __ldg(a.state + (uint64_t)r * a.stride_words + w) : 0u;
        uint32_t mine = 0;
#pragma unroll
        for (uint32_t b = 0; b < 32; b++) {
            const uint32_t m = __ballot_sync(~0u, (v >> b) & 1u);        // bit l: row xw*32 + 32h + l carries gene 32w + b
            if (lane == b) mine = m;
        }
        out[h] = mine;
    }
    if (k != ~0u) *reinterpret_cast<uint2 *>(a.x + (uint64_t)k * a.kw + xw) = make_uint2(out[0], out[1]);
}

struct GeneLdPairArgs {
    const uint32_t *x;              // [n_used][kw] presence bit rows
    uint32_t kw, k_iters;           // k_iters = kw * 32 / LD_KB
    const uint32_t *a, *grp;
    const double *inv;
    uint32_t n_used, n_rows, n_tiles, r2_bins;
    unsigned long long *out;        // [3][GL_CLASS_WORDS] class totals, then the histogram [3][r2_bins]
};

// tile pairs before tile I when tile I pairs with J = I .. n_tiles - 1
__device__ __forceinline__ uint64_t gene_ld_tile_off(uint64_t I, uint64_t n_tiles) { return I * n_tiles - I * (I - 1) / 2; }

static inline size_t gene_ld_pair_smem_bytes(uint32_t r2_bins) { return LD_OPERAND_SMEM + 3 * (size_t)r2_bins * sizeof(uint32_t); }

__global__ void __launch_bounds__(LD_THREADS, 3) gene_ld_pair_kernel(const GeneLdPairArgs p)
{
    extern __shared__ uint8_t um_smem[];
    __shared__ uint32_t s_a[LD_TILE], s_grp[LD_TILE];
    __shared__ double s_inv[LD_TILE];
    __shared__ unsigned long long s_cls[3][GL_CLASS_WORDS - 1];      // pairs, four-gamete, sum of q, associated, dissociated
    __shared__ uint32_t s_ij[2];
    const BitMma m = bitmma_smem<LD_KB>(um_smem);
    uint32_t *s_hist = reinterpret_cast<uint32_t *>(um_smem + LD_OPERAND_SMEM);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        // tile pair blockIdx.x: the largest I with tile_off(I) <= blockIdx.x
        uint32_t lo = 0, hi = p.n_tiles - 1;
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo + 1) / 2;
            if (gene_ld_tile_off(mid, p.n_tiles) <= blockIdx.x) lo = mid;
            else hi = mid - 1;
        }
        s_ij[0] = lo;
        s_ij[1] = lo + (uint32_t)(blockIdx.x - gene_ld_tile_off(lo, p.n_tiles));
        bitmma_init<LD_KB>(m);
    }
    for (uint32_t b = threadIdx.x; b < 3 * p.r2_bins; b += LD_THREADS) s_hist[b] = 0;
    if (threadIdx.x < 3 * (GL_CLASS_WORDS - 1)) (&s_cls[0][0])[threadIdx.x] = 0;
    if (warp == UB_EXP_WARPS) bitmma_alloc(m);
    const uint32_t tmem = bitmma_tmem(m);
    const uint32_t bi = s_ij[0], bj = s_ij[1];
    if (threadIdx.x < LD_TILE) {
        const uint32_t j = bj * LD_TILE + threadIdx.x;
        const bool ok = j < p.n_used;
        s_a[threadIdx.x] = ok ? p.a[j] : 0u;
        s_grp[threadIdx.x] = ok ? p.grp[j] : 0u;
        s_inv[threadIdx.x] = ok ? p.inv[j] : 0.0;
    }

    bitmma_mainloop<LD_KB>(m, tmem, p.x, p.kw, p.n_used, p.k_iters, bi, bj, warp, lane);
    __syncthreads();                                   // s_a / s_grp / s_inv / s_cls / s_hist written

    // ---- epilogue: warps w and w + 4 share the accumulator lanes 32 * (w % 4) .. + 31 (genes i of the I tile)
    //      and split the 128 columns (genes j of the J tile) ----
    if (warp < UB_EXP_WARPS) {
        bitmma_wait(m);
        const uint32_t quad = warp & 3u;
        const uint32_t ci = bi * LD_TILE + quad * 32u + lane;
        const bool i_ok = ci < p.n_used;
        const long long ai = i_ok ? (long long)p.a[ci] : 0ll;
        const double inv_i = i_ok ? p.inv[ci] : 0.0;
        const uint32_t gi = i_ok ? p.grp[ci] : 0u;
        const long long n = p.n_rows;
        uint32_t cur = ~0u;
        unsigned long long np = 0, nf = 0, sq = 0, nas = 0, nds = 0;
        auto flush = [&]() {
            if (!np) return;
            atomicAdd(&s_cls[cur][0], np);
            if (nf) atomicAdd(&s_cls[cur][1], nf);
            atomicAdd(&s_cls[cur][2], sq);
            if (nas) atomicAdd(&s_cls[cur][3], nas);
            if (nds) atomicAdd(&s_cls[cur][4], nds);
            np = nf = sq = nas = nds = 0;
        };
#pragma unroll 1
        for (uint32_t c0 = (warp >> 2) * 64u; c0 < (warp >> 2) * 64u + 64u; c0 += 16) {
            uint32_t v[16];
            bitmma_load16(tmem, quad, c0, v);
            if (!i_ok) continue;
#pragma unroll
            for (uint32_t q = 0; q < 16; q++) {
                const uint32_t jl = c0 + q, cj = bj * LD_TILE + jl;
                if (cj <= ci || cj >= p.n_used) continue;
                const uint32_t cls = gi + s_grp[jl];
                if (cls != cur) { flush(); cur = cls; }
                const long long c = v[q], aj = s_a[jl];
                const long long Di = n * c - ai * aj;
                const double D = (double)Di;
                const double r2 = __dmul_rn(__dmul_rn(__dmul_rn(D, D), inv_i), s_inv[jl]);
                const unsigned long long qv = __double2ull_rn(__dmul_rn(r2, 4294967296.0));
                np++;
                nf += (c > 0) & (ai > c) & (aj > c) & (n - ai - aj + c > 0);
                sq += qv;
                nas += Di > 0;
                nds += Di < 0;
                const uint32_t b = (uint32_t)min((qv * p.r2_bins) >> 32, (unsigned long long)(p.r2_bins - 1));
                atomicAdd(&s_hist[cls * p.r2_bins + b], 1u);
            }
        }
        flush();
    }
    bitmma_free(tmem, warp);
    if (threadIdx.x < 3 && s_cls[threadIdx.x][0]) {
        unsigned long long *g = p.out + GL_CLASS_WORDS * threadIdx.x;
        atomicAdd(g, s_cls[threadIdx.x][0]);
        if (s_cls[threadIdx.x][1]) atomicAdd(g + 1, s_cls[threadIdx.x][1]);
        ld_add128(g + 2, g + 3, s_cls[threadIdx.x][2]);
        if (s_cls[threadIdx.x][3]) atomicAdd(g + 4, s_cls[threadIdx.x][3]);
        if (s_cls[threadIdx.x][4]) atomicAdd(g + 5, s_cls[threadIdx.x][4]);
    }
    for (uint32_t b = threadIdx.x; b < 3 * p.r2_bins; b += LD_THREADS)
        if (s_hist[b]) atomicAdd(p.out + GL_OUT_CLASSES + b, (unsigned long long)s_hist[b]);
}

}  // namespace pansim
