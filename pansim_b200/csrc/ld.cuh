// ld.cuh -- linkage disequilibrium of the core alignment: r^2 and four-gamete pairs binned by site distance,
// the joint derived counts of site pairs on the tensor cores (DESIGN.md section 12).
//
// Site pass: from the per-site allele counts (diversity_kernel<true, false>) and the packed ancestral row,
// ld_site_kernel counts the used sites of every 2048-site block (derived count a with min_minor <= min(a, n - a));
// vcf_scan_blocks_kernel scans the block totals, and ld_compact_kernel gives every used site its compact index
// (rank) and writes its global position, a, and inv = 1 / (a (n - a)). Integer scans: deterministic.
//
// Transpose: ld_transpose_kernel turns the packed row-major 2-bit rows into site-major bit rows X[k][kw] of the
// used sites (bit r of row k: row r is derived at used site k), kw = ceil(n / 64) * 2 words, zero past row n.
// A CTA owns 128 sites (8 packed words) x 128 rows; 16 x 16 blocks of 2-bit codes are transposed in registers as
// in vcf_expand_kernel, compared with the ancestral code and squeezed to 16-bit masks in shared memory.
//
// Tile list: used sites in tiles of 128. Tile I pairs with J = I .. the tile of the last used site within max_dist
// of I's last site (ld_tiles_kernel: a binary search per I), scanned into tile-pair offsets.
//
// Pair kernel: one CTA per tile pair on the operand pipeline of bitmma.cuh with 64-byte swizzled rows: eight warps
// expand the bit rows of both tiles into the swizzled K-major u8 operand layout, one thread issues
// tcgen05.mma.kind::i8 into a 128 x 128 s32 accumulator in tensor memory, which holds c = the rows derived at both
// sites. The same eight warps then read it with tcgen05.ld and form D, r^2, q and the four-gamete test per pair,
// accumulating in registers while the bin does not change (j ascending, so d ascending); per-CTA bins in shared
// memory, then global u64 adds (r^2 as a 128-bit sum: lo with carry into hi). About 50 KB of shared memory and
// 128 tensor-memory columns per CTA, so several CTAs share an SM and one's epilogue overlaps another's MMAs.
#pragma once
#include "bitmma.cuh"
#include "common.cuh"
#include "vcf.cuh"

namespace pansim {

constexpr uint32_t LD_KB = 64;                          // K bits per pipeline stage (UbCfg<64>: 64-byte swizzle)
constexpr uint32_t LD_TILE = UM_TILE;                   // 128 used sites per tile
constexpr uint32_t LT_SITES = 128;                      // transpose: sites per CTA (8 packed words)
constexpr uint32_t LT_ROWS = 128;                       // transpose: rows per CTA (4 output words)
constexpr uint32_t LT_THREADS = 128;
constexpr uint32_t LD_SMEM_BINS = 256;                  // bins kept in shared memory per CTA; more go to global directly
constexpr uint32_t LD_THREADS = UB_THREADS;             // 8 expansion / epilogue warps + the MMA warp

// kw: 32-bit words per site row of X (whole MMA K steps of 64 rows)
__host__ __device__ inline uint32_t ld_row_words(uint32_t n_rows) { return (n_rows + LD_KB - 1) / LD_KB * (LD_KB / 32); }

struct LdSiteArgs {
    const uint4 *counts;            // [n_sites] (n_A, n_C, n_G, n_T)
    const uint32_t *anc;            // packed ancestral row of the local sites
    uint64_t n_sites;               // sites of the pass; everything at or past it is never used
    uint32_t n_rows;
    uint32_t min_minor;
    uint32_t pos0;                  // global index of local site 0
    unsigned long long *block;      // [n_blocks + 1] used sites per block, then their exclusive scan (+ total)
    uint32_t *rank;                 // [n_sites] compact index of a used site, ~0u otherwise
    uint32_t *pos, *a;              // [used] global index, derived count
    double *inv;                    // [used] 1 / (a (n - a))
};

// derived count of local site s and whether the site is used
__device__ __forceinline__ bool ld_site_used(const LdSiteArgs &a, uint64_t s, uint32_t *derived)
{
    const uint4 n = a.counts[s];
    const uint32_t ref = (__ldg(a.anc + (s >> 4)) >> (2 * (s & 15u))) & 3u;
    const uint32_t n_anc = ref == 0 ? n.x : ref == 1 ? n.y : ref == 2 ? n.z : n.w;
    const uint32_t d = a.n_rows - n_anc;
    *derived = d;
    return a.min_minor <= min(d, n_anc);
}

// used sites per block; thread t of block b takes sites b*VS_SITES + 8t .. 8t+7
__global__ void __launch_bounds__(VS_THREADS) ld_site_kernel(LdSiteArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t s0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    unsigned long long used = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        uint32_t d;
        if (s0 + i < a.n_sites && ld_site_used(a, s0 + i, &d)) used++;
    }
    unsigned long long total;
    vcf_block_scan(used, s_warp, &total);
    if (threadIdx.x == 0) a.block[blockIdx.x] = total;
}

// rank, position, derived count and inverse of every used site (block base + scan inside the block)
__global__ void __launch_bounds__(VS_THREADS) ld_compact_kernel(LdSiteArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t s0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    uint32_t dv[VS_PER_THREAD];
    uint32_t used = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        dv[i] = 0;
        if (s0 + i < a.n_sites && ld_site_used(a, s0 + i, &dv[i])) used |= 1u << i;
    }
    unsigned long long total;
    uint32_t k = (uint32_t)(a.block[blockIdx.x] + vcf_block_scan(__popc(used), s_warp, &total));
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        const uint64_t s = s0 + i;
        if (s >= a.n_sites) break;
        if (used >> i & 1u) {
            a.rank[s] = k;
            a.pos[k] = a.pos0 + (uint32_t)s;
            a.a[k] = dv[i];
            a.inv[k] = __ddiv_rn(1.0, (double)((unsigned long long)dv[i] * (a.n_rows - dv[i])));
            k++;
        } else {
            a.rank[s] = ~0u;
        }
    }
}

struct LdTransposeArgs {
    const uint32_t *state;          // packed rows (16 sites per word), row pitch row_words
    uint64_t row_words;
    uint32_t n_rows;
    uint64_t n_sites;
    const uint32_t *anc;
    const uint32_t *rank;
    uint32_t kw;                    // words per row of x
    uint32_t *x;                    // [used][kw]
};

// grid: x = 128-site tiles, y = 128-row blocks covering kw * 32 rows
__global__ void __launch_bounds__(LT_THREADS) ld_transpose_kernel(LdTransposeArgs a)
{
    __shared__ uint16_t s_m[LT_SITES][LT_ROWS / 16 + 2];    // derived mask of 16 rows per (site, row group)
    __shared__ uint32_t s_rank[LT_SITES];
    __shared__ int s_any;
    const uint32_t tid = threadIdx.x;
    const uint64_t tile = blockIdx.x;
    const uint32_t r0 = blockIdx.y * LT_ROWS;
    if (tid == 0) s_any = 0;
    __syncthreads();
    {
        const uint64_t s = tile * LT_SITES + tid;
        const uint32_t k = s < a.n_sites ? a.rank[s] : ~0u;
        s_rank[tid] = k;
        if (k != ~0u) s_any = 1;
    }
    __syncthreads();
    if (!s_any) return;

    // thread = (packed word w of the tile, row group j of 16 rows)
    if (tid < 8 * (LT_ROWS / 16)) {
        const uint32_t w = tid & 7u, j = tid >> 3;
        const uint32_t *src = a.state + tile * (LT_SITES / 16) + w;
        uint32_t x[16];
#pragma unroll
        for (uint32_t k = 0; k < 16; k++) {
            const uint32_t r = r0 + 16 * j + k;
            x[k] = r < a.n_rows ? __ldg(src + (uint64_t)r * a.row_words) : 0u;
        }
        vcf_transpose_stage<8>(x, 0x0000FFFFu);
        vcf_transpose_stage<4>(x, 0x00FF00FFu);
        vcf_transpose_stage<2>(x, 0x0F0F0F0Fu);
        vcf_transpose_stage<1>(x, 0x33333333u);
        // x[i] = codes of the group's 16 rows at site 16w + i, row k in bits 2k
        const uint32_t ancw = __ldg(a.anc + tile * (LT_SITES / 16) + w);
        const uint32_t rg = r0 + 16 * j;
        const uint32_t valid = rg >= a.n_rows ? 0u : a.n_rows - rg >= 16 ? 0xFFFFu : (1u << (a.n_rows - rg)) - 1u;
#pragma unroll
        for (uint32_t i = 0; i < 16; i++) {
            const uint32_t diff = x[i] ^ (((ancw >> (2 * i)) & 3u) * 0x55555555u);
            uint32_t m = (diff | (diff >> 1)) & 0x55555555u;      // bit 2k: row k differs from the ancestral code
            m = (m | (m >> 1)) & 0x33333333u;
            m = (m | (m >> 2)) & 0x0F0F0F0Fu;
            m = (m | (m >> 4)) & 0x00FF00FFu;
            m = (m | (m >> 8)) & 0x0000FFFFu;
            s_m[16 * w + i][j] = (uint16_t)(m & valid);
        }
    }
    __syncthreads();

    // thread = site: its 4 words of rows r0 .. r0 + 127 (two 8-byte stores; kw is even)
    const uint32_t k = s_rank[tid];
    if (k == ~0u) return;
    uint32_t *dst = a.x + (uint64_t)k * a.kw + r0 / 32;
#pragma unroll
    for (uint32_t q = 0; q < LT_ROWS / 64; q++) {
        if (r0 / 32 + 2 * q >= a.kw) break;
        const uint32_t w0 = s_m[tid][4 * q] | (uint32_t)s_m[tid][4 * q + 1] << 16;
        const uint32_t w1 = s_m[tid][4 * q + 2] | (uint32_t)s_m[tid][4 * q + 3] << 16;
        *reinterpret_cast<uint2 *>(dst + 2 * q) = make_uint2(w0, w1);
    }
}

// tile-pair count of every I tile: J = I .. the tile of the last used site with pos <= pos(last of I) + max_dist
__global__ void __launch_bounds__(256) ld_tiles_kernel(const uint32_t *pos, uint32_t n_own, uint32_t n_all, uint32_t max_dist,
                                                       unsigned long long *cnt)
{
    const uint32_t I = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_i = (n_own + LD_TILE - 1) / LD_TILE;
    if (I >= n_i) return;
    const uint32_t last = min((I + 1) * LD_TILE, n_own) - 1;
    const uint64_t lim = (uint64_t)pos[last] + max_dist;
    uint32_t lo = last, hi = n_all - 1;                   // the largest e with pos[e] <= lim lies in [lo, hi]
    while (lo < hi) {
        const uint32_t mid = lo + (hi - lo + 1) / 2;
        if ((uint64_t)pos[mid] <= lim) lo = mid;
        else hi = mid - 1;
    }
    cnt[I] = lo / LD_TILE - I + 1;
}

struct LdPairArgs {
    const uint32_t *x;              // [n_all][kw] derived bit rows
    uint32_t kw, k_iters;           // k_iters = kw * 32 / LD_KB
    const uint32_t *pos, *a;
    const double *inv;
    uint32_t n_own, n_all, n_rows;  // I rows: compact sites < n_own; J rows: < n_all (own + halo)
    uint32_t max_dist, bin_width, n_bins;
    const unsigned long long *tile_off;   // [n_i + 1] exclusive scan of the tile-pair counts
    uint32_t n_i;
    unsigned long long *bins;       // [n_bins][4]: pairs, four_gamete, r2_hi, r2_lo (pansim_ld_bin)
};

// exact 128-bit sum in (hi, lo): lo wraps at most once per add
__device__ __forceinline__ void ld_add128(unsigned long long *hi, unsigned long long *lo, unsigned long long x)
{
    const unsigned long long old = atomicAdd(lo, x);
    if (old + x < old) atomicAdd(hi, 1ull);
}

// operand stages and barriers, then the per-CTA bins when they fit
constexpr uint32_t LD_OPERAND_SMEM = (uint32_t)UbCfg<LD_KB>::smem_bytes();
static_assert(LD_OPERAND_SMEM % 8 == 0, "per-CTA bins are 8-byte words");

static inline size_t ld_pair_smem_bytes(uint32_t n_bins)
{
    return LD_OPERAND_SMEM + (n_bins <= LD_SMEM_BINS ? 3 * (size_t)n_bins * sizeof(unsigned long long) : 0);
}

__global__ void __launch_bounds__(LD_THREADS, 3) ld_pair_kernel(const LdPairArgs p)
{
    extern __shared__ uint8_t um_smem[];
    __shared__ uint32_t s_pos[LD_TILE], s_a[LD_TILE];
    __shared__ double s_inv[LD_TILE];
    __shared__ uint32_t s_ij[2];
    const BitMma m = bitmma_smem<LD_KB>(um_smem);
    // per-CTA bins after the operand stages and barriers: pairs, four-gamete, sum of q
    unsigned long long *s_bins = reinterpret_cast<unsigned long long *>(um_smem + LD_OPERAND_SMEM);
    const bool smem_bins = p.n_bins <= LD_SMEM_BINS;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        // tile pair blockIdx.x: the largest I with tile_off[I] <= blockIdx.x
        uint32_t lo = 0, hi = p.n_i - 1;
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo + 1) / 2;
            if (p.tile_off[mid] <= blockIdx.x) lo = mid;
            else hi = mid - 1;
        }
        s_ij[0] = lo;
        s_ij[1] = lo + (uint32_t)(blockIdx.x - p.tile_off[lo]);
        bitmma_init<LD_KB>(m);
    }
    if (smem_bins)
        for (uint32_t b = threadIdx.x; b < 3 * p.n_bins; b += LD_THREADS) s_bins[b] = 0;
    if (warp == UB_EXP_WARPS) bitmma_alloc(m);
    const uint32_t tmem = bitmma_tmem(m);
    const uint32_t bi = s_ij[0], bj = s_ij[1];
    if (threadIdx.x < LD_TILE) {
        const uint32_t j = bj * LD_TILE + threadIdx.x;
        const bool ok = j < p.n_all;
        s_pos[threadIdx.x] = ok ? p.pos[j] : 0u;
        s_a[threadIdx.x] = ok ? p.a[j] : 0u;
        s_inv[threadIdx.x] = ok ? p.inv[j] : 0.0;
    }

    bitmma_mainloop<LD_KB>(m, tmem, p.x, p.kw, p.n_all, p.k_iters, bi, bj, warp, lane);
    __syncthreads();                                   // s_pos / s_a / s_inv written

    // ---- epilogue: warps w and w + 4 share the accumulator lanes 32 * (w % 4) .. + 31 (sites i of the I tile)
    //      and split the 128 columns (sites j of the J tile) ----
    if (warp < UB_EXP_WARPS) {
        bitmma_wait(m);
        const uint32_t quad = warp & 3u;
        const uint32_t ci = bi * LD_TILE + quad * 32u + lane;
        const bool i_ok = ci < p.n_own;
        const uint32_t pi = i_ok ? p.pos[ci] : 0u;
        const long long ai = i_ok ? (long long)p.a[ci] : 0ll;
        const double inv_i = i_ok ? p.inv[ci] : 0.0;
        const long long n = p.n_rows;
        uint32_t cur = ~0u;
        unsigned long long np = 0, nf = 0, sq = 0;
        auto flush = [&]() {
            if (!np) return;
            if (smem_bins) {
                atomicAdd(&s_bins[cur], np);
                atomicAdd(&s_bins[p.n_bins + cur], nf);
                atomicAdd(&s_bins[2 * p.n_bins + cur], sq);
            } else {
                unsigned long long *g = p.bins + 4ull * cur;
                atomicAdd(g, np);
                if (nf) atomicAdd(g + 1, nf);
                ld_add128(g + 2, g + 3, sq);
            }
            np = nf = sq = 0;
        };
#pragma unroll 1
        for (uint32_t c0 = (warp >> 2) * 64u; c0 < (warp >> 2) * 64u + 64u; c0 += 16) {
            uint32_t v[16];
            bitmma_load16(tmem, quad, c0, v);
            if (!i_ok) continue;
#pragma unroll
            for (uint32_t q = 0; q < 16; q++) {
                const uint32_t jl = c0 + q, cj = bj * LD_TILE + jl;
                if (cj <= ci || cj >= p.n_all) continue;
                const uint32_t d = s_pos[jl] - pi;
                if (d > p.max_dist) continue;
                const uint32_t b = (d - 1u) / p.bin_width;
                if (b != cur) { flush(); cur = b; }
                const long long c = v[q], aj = s_a[jl];
                const double D = (double)(n * c - ai * aj);
                const double r2 = __dmul_rn(__dmul_rn(__dmul_rn(D, D), inv_i), s_inv[jl]);
                np++;
                nf += (c > 0) & (ai > c) & (aj > c) & (n - ai - aj + c > 0);
                sq += __double2ull_rn(__dmul_rn(r2, 4294967296.0));
            }
        }
        flush();
    }
    bitmma_free(tmem, warp);
    if (smem_bins)
        for (uint32_t b = threadIdx.x; b < p.n_bins; b += LD_THREADS) {
            const unsigned long long np = s_bins[b];
            if (!np) continue;
            unsigned long long *g = p.bins + 4ull * b;
            atomicAdd(g, np);
            if (s_bins[p.n_bins + b]) atomicAdd(g + 1, s_bins[p.n_bins + b]);
            ld_add128(g + 2, g + 3, s_bins[2 * p.n_bins + b]);
        }
}

}  // namespace pansim
