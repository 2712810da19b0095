// diversity.cuh -- one column reduction of the packed core alignment: per-site allele counts
// n_A..n_T and, from them, the population-genetic summaries (segregating / multiallelic sites,
// sum over sites of the pairwise differences, site frequency spectrum against the ancestral row).
//
// Layout (DESIGN.md section 10). A CTA owns a slab of 64 packed words = 1024 sites of every row; each
// of its 8 warps walks 1/8 of the rows, lane l loading words 2l, 2l+1 of the slab (256 contiguous
// bytes per warp and row). Per row nothing is decoded: the packed word itself is added to bit-sliced
// vertical counters (Harley-Seal carry-save adders, 8 inputs at a time), so bit 2s counts the rows whose
// site s has its low code bit set (C or T) and bit 2s+1 those with the high bit set (G or T). The T
// count comes from a second counter over v & (v >> 1), two rows packed into one word. Every 128 rows
// the counters (8 bit-planes, so at most 255 per position) are turned into byte lanes and added to the
// CTA's per-site counts in shared memory; after the last row the CTA derives the per-site outputs and
// adds its integer partials into global memory with atomics. All outputs are integers: the grid shape
// cannot change a result.
#pragma once
#include "common.cuh"

namespace pansim {

constexpr uint32_t DV_WARPS = 8;
constexpr uint32_t DV_THREADS = DV_WARPS * 32;
constexpr uint32_t DV_WORDS = 64;                 // packed words per CTA slab (two per lane)
constexpr uint32_t DV_SITES = DV_WORDS * 16;      // 1024
constexpr uint32_t DV_CHUNK = 128;                // rows between two flushes of the 8-plane counters (max 255)
constexpr uint32_t DV_PITCH = DV_WORDS + 1;       // shared count arrays [site in word][slab column], padded
constexpr uint32_t DV_SFS_BINS = 4096;            // SFS bins histogrammed in shared memory; larger k go to global

struct DiversityArgs {
    const uint32_t *state;          // packed rows (16 sites per word), row pitch row_words
    uint64_t row_words;
    uint64_t n_sites;               // local sites: positions at or beyond it are padding and never counted
    uint32_t n_rows;
    const uint32_t *anc;            // packed ancestral row (SFS only)
    unsigned long long *out;        // [0] segregating, [1] multiallelic, [2] sum over sites of sum_{a<b} n_a n_b
    uint4 *counts;                  // [n_sites] (n_A, n_C, n_G, n_T), or null
    unsigned long long *sfs;        // [n_rows + 1], or null
};

__device__ __forceinline__ void dv_csa(uint32_t &h, uint32_t &l, uint32_t a, uint32_t b, uint32_t c)
{
    const uint32_t u = a ^ b;
    h = (a & b) | (u & c);
    l = u ^ c;
}

// add eight 1-bit inputs per bit position into the vertical counter c (plane i has weight 2^i)
__device__ __forceinline__ void dv_add8(uint32_t (&c)[8], uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t x4,
                                        uint32_t x5, uint32_t x6, uint32_t x7)
{
    uint32_t tA, tB, fA, fB, e;
    dv_csa(tA, c[0], c[0], x0, x1);
    dv_csa(tB, c[0], c[0], x2, x3);
    dv_csa(fA, c[1], c[1], tA, tB);
    dv_csa(tA, c[0], c[0], x4, x5);
    dv_csa(tB, c[0], c[0], x6, x7);
    dv_csa(fB, c[1], c[1], tA, tB);
    dv_csa(e, c[2], c[2], fA, fB);
#pragma unroll
    for (int i = 3; i < 8; i++) {
        const uint32_t t = c[i] & e;
        c[i] ^= e;
        e = t;
    }
}

// counts of bit positions p, p+8, p+16, p+24 as four byte lanes
__device__ __forceinline__ uint32_t dv_lanes(const uint32_t (&c)[8], int p)
{
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r += ((c[i] >> p) & 0x01010101u) << i;
    return r;
}

// T bits of two rows in one word: bit 2s = row a has T at site s, bit 2s+1 = row b has
__device__ __forceinline__ uint32_t dv_t_pair(uint32_t a, uint32_t b)
{
    return (a & (a >> 1) & 0x55555555u) | (b & (b << 1) & 0xAAAAAAAAu);
}

template <bool COUNTS, bool SFS>
__global__ void __launch_bounds__(DV_THREADS, 2) diversity_kernel(DiversityArgs a)
{
    __shared__ uint32_t s_lo[16 * DV_PITCH], s_hi[16 * DV_PITCH], s_t[16 * DV_PITCH];
    __shared__ unsigned long long s_red[DV_WARPS][4];
    extern __shared__ uint32_t s_sfs[];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t n_bins = SFS ? min(a.n_rows + 1u, DV_SFS_BINS) : 1u;   // only read where SFS
    for (uint32_t i = tid; i < 16 * DV_PITCH; i += DV_THREADS) s_lo[i] = s_hi[i] = s_t[i] = 0;
    if (SFS)
        for (uint32_t i = tid; i < n_bins; i += DV_THREADS) s_sfs[i] = 0;
    __syncthreads();

    const uint64_t slab = blockIdx.x;
    const uint2 *col = reinterpret_cast<const uint2 *>(a.state + slab * DV_WORDS) + lane;
    const uint64_t pitch2 = a.row_words / 2;
    const uint32_t rows_per_warp = (a.n_rows + DV_WARPS - 1) / DV_WARPS;
    const uint32_t r_begin = min(a.n_rows, warp * rows_per_warp), r_end = min(a.n_rows, r_begin + rows_per_warp);

    for (uint32_t c0 = r_begin; c0 < r_end; c0 += DV_CHUNK) {
        const uint32_t c1 = min(r_end, c0 + DV_CHUNK);
        uint32_t v0[8], v1[8], t0[8], t1[8];          // vertical counters: words 2l, 2l+1; all bits / T pairs
#pragma unroll
        for (int i = 0; i < 8; i++) v0[i] = v1[i] = t0[i] = t1[i] = 0;
        for (uint32_t r = c0; r < c1; r += 16) {
            uint2 x[16];
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = (r + k < c1) ? __ldg(col + (uint64_t)(r + k) * pitch2) : make_uint2(0, 0);
            dv_add8(v0, x[0].x, x[1].x, x[2].x, x[3].x, x[4].x, x[5].x, x[6].x, x[7].x);
            dv_add8(v0, x[8].x, x[9].x, x[10].x, x[11].x, x[12].x, x[13].x, x[14].x, x[15].x);
            dv_add8(v1, x[0].y, x[1].y, x[2].y, x[3].y, x[4].y, x[5].y, x[6].y, x[7].y);
            dv_add8(v1, x[8].y, x[9].y, x[10].y, x[11].y, x[12].y, x[13].y, x[14].y, x[15].y);
            dv_add8(t0, dv_t_pair(x[0].x, x[1].x), dv_t_pair(x[2].x, x[3].x), dv_t_pair(x[4].x, x[5].x), dv_t_pair(x[6].x, x[7].x),
                    dv_t_pair(x[8].x, x[9].x), dv_t_pair(x[10].x, x[11].x), dv_t_pair(x[12].x, x[13].x), dv_t_pair(x[14].x, x[15].x));
            dv_add8(t1, dv_t_pair(x[0].y, x[1].y), dv_t_pair(x[2].y, x[3].y), dv_t_pair(x[4].y, x[5].y), dv_t_pair(x[6].y, x[7].y),
                    dv_t_pair(x[8].y, x[9].y), dv_t_pair(x[10].y, x[11].y), dv_t_pair(x[12].y, x[13].y), dv_t_pair(x[14].y, x[15].y));
        }
        // flush: bit position p + 8j of a word is site p/2 + 4j (low code bit for even p, high for odd p).
        // Shared column of word 2l + w is w*32 + l, so the 32 lanes of a warp hit 32 banks.
#pragma unroll
        for (int w = 0; w < 2; w++) {
            const uint32_t(&v)[8] = w ? v1 : v0;
            const uint32_t(&t)[8] = w ? t1 : t0;
            const uint32_t colw = w * 32u + lane;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t lo = dv_lanes(v, 2 * q), hi = dv_lanes(v, 2 * q + 1);
                const uint32_t tt = dv_lanes(t, 2 * q) + dv_lanes(t, 2 * q + 1);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const uint32_t idx = (uint32_t)(q + 4 * j) * DV_PITCH + colw;
                    atomicAdd(&s_lo[idx], (lo >> (8 * j)) & 0xFFu);
                    atomicAdd(&s_hi[idx], (hi >> (8 * j)) & 0xFFu);
                    atomicAdd(&s_t[idx], (tt >> (8 * j)) & 0xFFu);
                }
            }
        }
    }
    __syncthreads();

    // per-site outputs: thread tid takes sites tid, tid + 256, ... of the slab
    const unsigned long long N = a.n_rows;
    unsigned long long seg = 0, multi = 0, pd = 0, k0 = 0;
#pragma unroll
    for (uint32_t i = 0; i < DV_SITES / DV_THREADS; i++) {
        const uint32_t e = tid + i * DV_THREADS;
        const uint64_t gs = slab * DV_SITES + e;
        if (gs >= a.n_sites) break;
        const uint32_t word = e >> 4, idx = (e & 15u) * DV_PITCH + (word & 1u) * 32u + (word >> 1);
        const uint32_t nT = s_t[idx], nC = s_lo[idx] - nT, nG = s_hi[idx] - nT;
        const uint32_t nA = a.n_rows - nC - nG - nT;
        const uint32_t present = (nA > 0) + (nC > 0) + (nG > 0) + (nT > 0);
        seg += present >= 2;
        multi += present >= 3;
        const unsigned long long sq = (unsigned long long)nA * nA + (unsigned long long)nC * nC + (unsigned long long)nG * nG +
                                      (unsigned long long)nT * nT;
        pd += (N * N - sq) >> 1;
        if (COUNTS) a.counts[gs] = make_uint4(nA, nC, nG, nT);
        if (SFS) {
            const uint32_t code = (__ldg(a.anc + (gs >> 4)) >> (2 * (gs & 15u))) & 3u;
            const uint32_t n_anc = code == 0 ? nA : code == 1 ? nC : code == 2 ? nG : nT;
            const uint32_t k = a.n_rows - n_anc;
            if (k == 0) k0++;
            else if (k < n_bins) atomicAdd(&s_sfs[k], 1u);
            else atomicAdd(&a.sfs[k], 1ull);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        seg += __shfl_xor_sync(0xFFFFFFFFu, seg, o);
        multi += __shfl_xor_sync(0xFFFFFFFFu, multi, o);
        pd += __shfl_xor_sync(0xFFFFFFFFu, pd, o);
        k0 += __shfl_xor_sync(0xFFFFFFFFu, k0, o);
    }
    if (lane == 0) { s_red[warp][0] = seg; s_red[warp][1] = multi; s_red[warp][2] = pd; s_red[warp][3] = k0; }
    __syncthreads();
    if (tid < 4) {
        unsigned long long s = 0;
        for (uint32_t w = 0; w < DV_WARPS; w++) s += s_red[w][tid];
        if (tid < 3) {
            if (s) atomicAdd(&a.out[tid], s);
        } else if (SFS && s) {
            atomicAdd(&a.sfs[0], s);
        }
    }
    if (SFS)
        for (uint32_t b = 1 + tid; b < n_bins; b += DV_THREADS)
            if (s_sfs[b]) atomicAdd(&a.sfs[b], (unsigned long long)s_sfs[b]);
}

}  // namespace pansim
