// select.cuh -- K1/K2/K3: fitness, competition term and parent resampling.
//   K1 fitness           population.rs:282-322  (f64 sum in column order -> bit-exact)
//   K2 average_distance  population.rs:753-784 + get_distance :114-151 (bit-exact)
//   K3 weights + draw    population.rs:325-447
#pragma once
#include <cfloat>
#include "bitmma.cuh"
#include "common.cuh"

namespace pansim {

// ---------------------------------------------------------------------------
// K1: log-fitness l_i = sum_j ln(1 + s_j * x_ij) and gene counts.
// x_ij in {0,1}, so a term is either ln(1) = +0.0 (adding it never changes the
// running sum) or lw_j = ln(1 + s_j), precomputed on the host with the same
// libm expression the reference evaluates. One thread per row adds the present
// genes in increasing column order, reproducing the reference's sequential f64
// sum bit for bit (population.rs:303-317). A present gene with lw_j = -inf
// (s_j = -1) sets l_i := 0.0 (population.rs:312-318).
// ---------------------------------------------------------------------------
constexpr int FIT_WARPS = 4;                      // rows per CTA of the blocked / count-only kernels
constexpr int FIT_ROWS = 2;                       // rows per CTA of the sequential kernel (two warps per row)
constexpr int FIT_CHUNK_WORDS = 32;               // 1024 genes per compaction round
constexpr int FIT_BATCH = 8;                      // chain elements loaded ahead of the additions

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t threads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t threads)
{
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// every selection coefficient is 0 (neutral run: lw_j = ln(1) = +0.0 for all j): the sum is +0.0
// whatever the genome; only the row popcounts are needed
__global__ void __launch_bounds__(FIT_WARPS * 32) fitness_count_kernel(const uint32_t *acc, uint32_t n_rows,
                                                                       uint32_t n_genes, uint32_t stride_words,
                                                                       double *logfit, int32_t *num_genes)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t row = blockIdx.x * FIT_WARPS + warp;
    if (row >= n_rows) return;
    const uint32_t *r = acc + (uint64_t)row * stride_words;
    const uint32_t n_words = (n_genes + 31u) / 32u;
    int32_t cnt = 0;
    for (uint32_t w = lane; w < n_words; w += 32) cnt += __popc(r[w]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) { logfit[row] = 0.0; num_genes[row] = cnt; }
}

// Terms of absent genes are ln(1 + s*0) = +0.0: adding them never changes the running sum, so
// only present genes are added -- in increasing column order, by a single sequential f64 chain
// per row (bit-exact vs population.rs:303-317). Two warps per row: the PRODUCER compacts the lw
// values of the present genes of each 1024-gene chunk into one of two shared-memory lists (padded
// with +0.0 to whole batches: the running sum starts at +0.0 and can never become -0.0, so
// x + (+0.0) = x); the CONSUMER runs the chain, its loads one batch ahead of the additions, so it
// advances at the latency of a dependent DADD (8.2 cycles on B200) while the producer prepares
// the next chunk. Full/empty hand-over through named barriers.
__global__ void __launch_bounds__(FIT_ROWS * 64) fitness_kernel(const uint32_t *acc, uint32_t n_rows,
                                                                uint32_t n_genes, uint32_t stride_words,
                                                                const double *lw, double *logfit,
                                                                int32_t *num_genes)
{
    constexpr int LIST = FIT_CHUNK_WORDS * 32 + 2 * FIT_BATCH;
    __shared__ double list[FIT_ROWS][2][LIST];
    __shared__ uint32_t tot_s[FIT_ROWS][2];
    __shared__ int32_t fin_s[FIT_ROWS][2];           // gene count, -inf seen
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t r_in_cta = warp >> 1;
    const bool producer = (warp & 1u) != 0u;
    const uint32_t row = blockIdx.x * FIT_ROWS + r_in_cta;
    if (row >= n_rows) return;                        // both warps of the row leave together
    const uint32_t n_words = (n_genes + 31u) / 32u;
    const uint32_t n_chunks = (n_words + FIT_CHUNK_WORDS - 1) / FIT_CHUNK_WORDS;
    const uint32_t bar_full = 1u + r_in_cta * 5u, bar_empty = 3u + r_in_cta * 5u, bar_done = 5u + r_in_cta * 5u;
    if (producer) {
        const uint32_t *r = acc + (uint64_t)row * stride_words;
        bool neg_inf = false;
        int32_t cnt = 0;
        for (uint32_t ch = 0; ch < n_chunks; ch++) {
            const uint32_t b = ch & 1u;
            if (ch >= 2) named_bar_sync(bar_empty + b, 64);          // the consumer is done with this list
            double *mine = list[r_in_cta][b];
            const uint32_t w = ch * FIT_CHUNK_WORDS + lane;
            uint32_t bits = (w < n_words) ? r[w] : 0u;
            const uint32_t c = __popc(bits);
            uint32_t incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if ((int)lane >= o) incl += v;
            }
            uint32_t off = incl - c;
            const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
            cnt += (int32_t)tot;
            if (lane < 2 * FIT_BATCH) mine[tot + lane] = 0.0;        // padding behind the last value
            if (lane == 0) tot_s[r_in_cta][b] = tot;
            while (bits) {
                const uint32_t bb = __ffs(bits) - 1;
                bits &= bits - 1;
                const double v = lw[w * 32u + bb];
                neg_inf |= (v == -INFINITY);
                mine[off++] = v;
            }
            named_bar_arrive(bar_full + b, 64);
        }
        neg_inf = __any_sync(0xffffffffu, neg_inf);
        if (lane == 0) { fin_s[r_in_cta][0] = cnt; fin_s[r_in_cta][1] = neg_inf ? 1 : 0; }
        named_bar_arrive(bar_done, 64);
    } else {
        double sum = 0.0;
        for (uint32_t ch = 0; ch < n_chunks; ch++) {
            const uint32_t b = ch & 1u;
            named_bar_sync(bar_full + b, 64);
            const double *mine = list[r_in_cta][b];
            const uint32_t tot = tot_s[r_in_cta][b];
            // every lane runs the same chain
            double nx[FIT_BATCH];
#pragma unroll
            for (int q = 0; q < FIT_BATCH; q++) nx[q] = mine[q];
            for (uint32_t t = 0; t < tot; t += FIT_BATCH) {
                double cu[FIT_BATCH];
#pragma unroll
                for (int q = 0; q < FIT_BATCH; q++) cu[q] = nx[q];
#pragma unroll
                for (int q = 0; q < FIT_BATCH; q++) nx[q] = mine[t + FIT_BATCH + q];
#pragma unroll
                for (int q = 0; q < FIT_BATCH; q++) sum += cu[q];
            }
            if (ch + 2 < n_chunks) named_bar_arrive(bar_empty + b, 64);
        }
        named_bar_sync(bar_done, 64);
        if (lane == 0) {
            logfit[row] = (n_genes > 0) ? (fin_s[r_in_cta][1] ? 0.0 : sum) : 0.0;
            num_genes[row] = fin_s[r_in_cta][0];
        }
    }
}

// The same sequential sum with ONE LANE PER ROW: every lane walks the set bits of its own row in
// column order and runs its own dependent f64 chain, so a warp advances 32 rows per DADD instead
// of one. The kernel needs 1/32 of the warps of the row-per-warp-pair kernel above and therefore
// hardly takes SM slots away from the core kernel it runs beside (measured: the row-per-warp-pair
// kernel holds ~500 CTAs for ~30 us each and costs the concurrent core kernel 6 %). The warp steps
// through ALL gene positions (G dependent DADD issues, each predicated on the lane's own bit) with
// the lw values of a 1024-gene chunk in shared memory. Genes with lw = -inf (s = -1) are given as
// a bit mask: they are left out of the chain and any of them present sets the result to 0.0
// (population.rs:312-318).
constexpr int FITL_THREADS = 128;

// sum += x iff (bits & mask). Written as the fused multiply-add sum = x * b + sum with b = 1.0 or +0.0
// built from the bit (one select for the high word of b; the low word is zero): x * 1.0 = x and
// x * 0.0 = +-0.0 are exact, so the single rounding of the FMA is the rounding of the plain addition,
// and sum + (+-0.0) = sum because the running sum starts at +0.0 and can never become -0.0. The
// operand selection is off the dependent chain (x and bits are known ahead): one DFMA per position.
__device__ __forceinline__ void add_if_bit(double &sum, double x, uint32_t bits, uint32_t mask)
{
    int hi;
    asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\tselp.b32 %0, 0x3FF00000, 0, p;\n\t}"
        : "=r"(hi) : "r"(bits), "r"(mask));
    sum = fma(x, __hiloint2double(hi, 0), sum);
}

__global__ void __launch_bounds__(FITL_THREADS, 4) fitness_lane_kernel(const uint32_t *acc, uint32_t n_rows,
                                                                    uint32_t n_genes, uint32_t stride_words,
                                                                    const double *lw, const uint32_t *lethal,
                                                                    double *logfit, int32_t *num_genes)
{
    __shared__ double lw_s[FIT_CHUNK_WORDS * 32];
    __shared__ uint32_t lethal_s[FIT_CHUNK_WORDS];
    // the lane's own 32 row words of the chunk (transposed: conflict-free), fetched with eight 16-byte loads before the
    // chain starts -- read one by one from global memory they cost an L2 round trip per word (2.5 x the chain itself)
    __shared__ uint32_t bits_s[FIT_CHUNK_WORDS][FITL_THREADS];
    const uint32_t row = blockIdx.x * FITL_THREADS + threadIdx.x;
    const bool live = row < n_rows;
    const uint32_t *r = acc + (uint64_t)(live ? row : 0u) * stride_words;
    const uint32_t n_words = (n_genes + 31u) / 32u;
    double sum = 0.0;
    bool neg_inf = false;
    int32_t cnt = 0;
    // the chunk's inputs travel through registers: those of chunk k + 1 are requested before the chain of chunk k starts
    // and land while it runs, so only the first chunk waits for global memory
    uint4 rw[FIT_CHUNK_WORDS / 4];
    double lwr[FIT_CHUNK_WORDS * 32 / FITL_THREADS];
    uint32_t lethal_r = 0;
    auto fetch = [&](uint32_t w0) {
#pragma unroll
        for (uint32_t q = 0; q < FIT_CHUNK_WORDS / 4; q++)      // rows are padded with zero words to a multiple of four (16-byte aligned)
            rw[q] = (live && w0 + 4u * q < stride_words) ? __ldg(reinterpret_cast<const uint4 *>(r + w0) + q) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (uint32_t q = 0; q < FIT_CHUNK_WORDS * 32 / FITL_THREADS; q++) {
            const uint32_t g = w0 * 32u + q * FITL_THREADS + threadIdx.x;
            lwr[q] = g < n_genes ? __ldg(lw + g) : 0.0;
        }
        if (threadIdx.x < FIT_CHUNK_WORDS) lethal_r = (w0 + threadIdx.x < n_words) ? __ldg(lethal + w0 + threadIdx.x) : 0u;
    };
    fetch(0u);
    for (uint32_t w0 = 0; w0 < n_words; w0 += FIT_CHUNK_WORDS) {
        __syncthreads();                                        // the previous chunk's chain has left shared memory
#pragma unroll
        for (uint32_t q = 0; q < FIT_CHUNK_WORDS * 32 / FITL_THREADS; q++)
            lw_s[q * FITL_THREADS + threadIdx.x] = (lwr[q] == -INFINITY) ? 0.0 : lwr[q];
        if (threadIdx.x < FIT_CHUNK_WORDS) lethal_s[threadIdx.x] = lethal_r;
        __syncthreads();
#pragma unroll
        for (uint32_t q = 0; q < FIT_CHUNK_WORDS / 4; q++) {
            const uint32_t wq[4] = {rw[q].x, rw[q].y, rw[q].z, rw[q].w};
#pragma unroll
            for (uint32_t i = 0; i < 4; i++) {
                const uint32_t dead = wq[i] & lethal_s[4u * q + i];        // present genes with s = -1 (population.rs:312-318)
                cnt += __popc(wq[i]);
                neg_inf |= dead != 0u;
                bits_s[4u * q + i][threadIdx.x] = wq[i] ^ dead;
            }
        }
        if (w0 + FIT_CHUNK_WORDS < n_words) fetch(w0 + FIT_CHUNK_WORDS);
        const uint32_t nw = min((uint32_t)FIT_CHUNK_WORDS, n_words - w0);
        // The additions of 16 gene positions (one half word) run while the lw values of the next
        // half word are already on their way from shared memory (same address for every lane:
        // broadcast; unconditional volatile loads so that they stay ahead of the chain), so the
        // chain advances at the DFMA latency (8.4 cycles, tools/experiments/fp64_latency.cu).
        const uint32_t lw_sa = smem_u32(lw_s);
        double xa[16], xb[16];
        auto load_half = [&](double (&x)[16], uint32_t half) {       // half = 2 * word + (0 | 1)
#pragma unroll
            for (int q = 0; q < 8; q++)
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x[2 * q]), "=d"(x[2 * q + 1])
                             : "r"(lw_sa + half * 128u + q * 16u));
        };
        uint32_t bits_next = bits_s[0][threadIdx.x];
        load_half(xa, 0u);
#pragma unroll 1
        for (uint32_t w = 0; w < nw; w++) {
            const uint32_t bits = bits_next;
            bits_next = bits_s[min(w + 1u, (uint32_t)FIT_CHUNK_WORDS - 1u)][threadIdx.x];
            load_half(xb, 2u * w + 1u);
#pragma unroll
            for (int b = 0; b < 16; b++) add_if_bit(sum, xa[b], bits, 1u << b);
            load_half(xa, min(2u * w + 2u, 2u * FIT_CHUNK_WORDS - 1u));
#pragma unroll
            for (int b = 0; b < 16; b++) add_if_bit(sum, xb[b], bits, 1u << (16 + b));
        }
    }
    if (live) {
        logfit[row] = (n_genes > 0) ? (neg_inf ? 0.0 : sum) : 0.0;
        num_genes[row] = cnt;
    }
}

// Large shapes (N x G above FITNESS_EXACT_CELLS): the strictly sequential chain above costs one
// issue slot per addition per row and dominates the accessory/selection chain (0.6 ms at
// N = 10 000, G = 18 000). The blocked variant adds, per row, the present genes of each 32-gene
// word in column order (one lane per word), then the word sums of each 1024-gene chunk in word
// order, then the chunk sums in chunk order: a fixed association, independent of grid shape and
// GPU count, within a few ulp (|rel| < 1e-13) of the reference's flat left-to-right sum.
__global__ void __launch_bounds__(FIT_WARPS * 32) fitness_blocked_kernel(const uint32_t *acc, uint32_t n_rows,
                                                                         uint32_t n_genes, uint32_t stride_words,
                                                                         const double *lw, double *logfit,
                                                                         int32_t *num_genes)
{
    __shared__ double lwc[1024];                       // lw of the current 1024-gene chunk (shared by the CTA's rows)
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t row = blockIdx.x * FIT_WARPS + warp;
    const bool live = row < n_rows;
    const uint32_t *r = acc + (uint64_t)(live ? row : 0) * stride_words;
    const uint32_t n_words = (n_genes + 31u) / 32u;
    double sum = 0.0;
    bool neg_inf = false;
    int32_t cnt = 0;
    for (uint32_t w0 = 0; w0 < n_words; w0 += 32) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < 1024; i += FIT_WARPS * 32) {
            const uint32_t g = w0 * 32u + i;
            lwc[i] = g < n_genes ? lw[g] : 0.0;
        }
        __syncthreads();
        const uint32_t w = w0 + lane;
        uint32_t bits = (live && w < n_words) ? r[w] : 0u;
        cnt += __popc(bits);
        double ws = 0.0;
        const double *lww = lwc + lane * 32u;
        while (bits) {
            const uint32_t b = __ffs(bits) - 1;
            bits &= bits - 1;
            const double v = lww[b];
            neg_inf |= (v == -INFINITY);
            ws += v;
        }
        double cs = 0.0;
#pragma unroll
        for (int t = 0; t < 32; t++) cs += __shfl_sync(0xffffffffu, ws, t);      // word order
        sum += cs;                                                               // chunk order
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    neg_inf = __any_sync(0xffffffffu, neg_inf);
    if (lane == 0 && live) {
        logfit[row] = (n_genes > 0) ? (neg_inf ? 0.0 : sum) : 0.0;
        num_genes[row] = cnt;
    }
}

// ---------------------------------------------------------------------------
// K2a: all-vs-all intersection counts I[i][j] = popc(row_i & row_j), the dense contraction X * X^T of the 0/1
// presence matrix on the tensor cores (bitmma.cuh). One CTA per upper-triangle tile of 128 x 128 pairs, mirrored on
// store. The diagonal I[i][i] = |row_i| is also written as a compact vector: the distance kernel takes its gene
// counts from there, so it does not have to wait for the (much longer) fitness kernel.
// Rows are zero-padded to stride_words = a multiple of 4 words (at least 4), so k_iters = ceil(max(G, 1) / 128)
// stages of 4 words never read past a row (the pipeline's precondition).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(UB_THREADS, 1) acc_inter_umma_bits_kernel(const uint32_t *__restrict__ acc, uint32_t n_rows,
                                                                           uint32_t stride_words, uint32_t k_iters,
                                                                           uint32_t *inter, int32_t *diag)
{
    extern __shared__ uint8_t um_smem[];
    const BitMma m = bitmma_smem<128>(um_smem);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // blockIdx.x enumerates the upper-triangle tiles row by row: (0,0..nb-1), (1,1..nb-1), ...
    const uint32_t nb = (n_rows + UM_TILE - 1) / UM_TILE;
    uint32_t t_lin = blockIdx.x, bi = 0;
    while (t_lin >= nb - bi) { t_lin -= nb - bi; bi++; }
    const uint32_t bj = bi + t_lin;

    if (threadIdx.x == 0) bitmma_init<128>(m);
    if (warp == UB_EXP_WARPS) bitmma_alloc(m);
    const uint32_t tmem = bitmma_tmem(m);
    bitmma_mainloop<128>(m, tmem, acc, stride_words, n_rows, k_iters, bi, bj, warp, lane);

    // ---- epilogue: warps w and w + 4 share the accumulator lanes 32 * (w % 4) .. + 31 and split the columns ----
    if (warp < UB_EXP_WARPS) {
        bitmma_wait(m);
        const uint32_t quad = warp & 3u;
        const uint32_t i = bi * UM_TILE + quad * 32u + lane;
        const bool vec_ok = (n_rows & 3u) == 0u;
#pragma unroll 1
        for (uint32_t c0 = (warp >> 2) * 64u; c0 < (warp >> 2) * 64u + 64u; c0 += 16) {
            uint32_t v[16];
            bitmma_load16(tmem, quad, c0, v);
            const uint32_t j0 = bj * UM_TILE + c0;
            if (i < n_rows) {
                uint32_t *dst = inter + (uint64_t)i * n_rows + j0;
                if (vec_ok && j0 + 16u <= n_rows) {
#pragma unroll
                    for (int q = 0; q < 16; q += 4) *reinterpret_cast<uint4 *>(dst + q) = make_uint4(v[q], v[q + 1], v[q + 2], v[q + 3]);
                } else {
#pragma unroll
                    for (int q = 0; q < 16; q++)
                        if (j0 + q < n_rows) dst[q] = v[q];
                }
#pragma unroll
                for (int q = 0; q < 16; q++) {
                    const uint32_t j = j0 + q;
                    if (j < n_rows) {
                        if (bi != bj) inter[(uint64_t)j * n_rows + i] = v[q];      // lanes = consecutive i: coalesced
                        else if (i == j) diag[i] = (int32_t)v[q];                  // |row_i|: the gene count the distances need
                    }
                }
            }
        }
    }
    bitmma_free(tmem, warp);
}

// K2b: mean Jaccard distance of individual i to all j != i, summed in j order
// exactly like get_distance + the fold of population.rs:770-771.
constexpr int AVG_WARPS = 8;
constexpr int AVG_RING = 256;       // distances evaluated per round (8 per lane)
constexpr int AVG_BATCH = 8;

__global__ void __launch_bounds__(AVG_WARPS * 32) avg_distance_kernel(const uint32_t *inter,
                                                                      const int32_t *num_genes, uint32_t n_rows,
                                                                      uint32_t core_genes, double *avgdist)
{
    // One warp per individual. Per round the 32 lanes evaluate 256 distances in parallel (the
    // f64 divisions are independent) into shared memory, then the values are added one by one in
    // j order -- the same sequential chain as the fold of population.rs:770 -- with the loads one
    // batch ahead of the additions. Entries with j == i or j >= N are +0.0, which never changes
    // the (non-negative) sum.
    __shared__ double ring[AVG_WARPS][AVG_RING + 2 * AVG_BATCH];
    pdl_launch_dependents();       // the parent-selection CTA may take its SM slot now (it waits for this grid)
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t i = blockIdx.x * AVG_WARPS + warp;
    if (i >= n_rows) return;
    double *mine = ring[warp];
    if (lane < 2 * AVG_BATCH) mine[AVG_RING + lane] = 0.0;
    const double cg = (double)core_genes;
    const uint32_t ki = (uint32_t)num_genes[i];
    const uint32_t *irow = inter + (uint64_t)i * n_rows;
    double sum = 0.0;
    for (uint32_t j0 = 0; j0 < n_rows; j0 += AVG_RING) {
        // all loads of the round first (one latency), then the divisions
        uint32_t in[AVG_RING / 32], kj[AVG_RING / 32];
#pragma unroll
        for (int q = 0; q < AVG_RING / 32; q++) {
            const uint32_t j = min(j0 + q * 32 + lane, n_rows - 1u);
            in[q] = irow[j];
            kj[q] = (uint32_t)num_genes[j];
        }
#pragma unroll
        for (int q = 0; q < AVG_RING / 32; q++) {
            const uint32_t j = j0 + q * 32 + lane;
            const uint32_t un = ki + kj[q] - in[q];
            const double d = 1.0 - (((double)in[q] + 0.0 + cg) / ((double)un + 0.0 + cg));   // :144-145
            mine[q * 32 + lane] = (j < n_rows && j != i) ? d : 0.0;
        }
        __syncwarp();
        const uint32_t tot = min((uint32_t)AVG_RING, n_rows - j0);
        double nx[AVG_BATCH];
#pragma unroll
        for (int q = 0; q < AVG_BATCH; q++) nx[q] = mine[q];
        for (uint32_t t = 0; t < tot; t += AVG_BATCH) {
            double cu[AVG_BATCH];
#pragma unroll
            for (int q = 0; q < AVG_BATCH; q++) cu[q] = nx[q];
#pragma unroll
            for (int q = 0; q < AVG_BATCH; q++) nx[q] = mine[t + AVG_BATCH + q];
#pragma unroll
            for (int q = 0; q < AVG_BATCH; q++) sum += cu[q];
        }
        __syncwarp();
    }
    if (lane == 0) {
        double fd = sum / (double)(n_rows - 1u);
        if (fd == 0.0) fd = DBL_MIN;                                  // :774-776
        avgdist[i] = fd;
    }
}

// The same mean distance for shapes with G + core_genes <= AVG_RCP_MAX. The quotient a / b of the two small integers
// a = |i & j| + core_genes <= b = |i | j| + core_genes is formed from the correctly rounded reciprocal r = RN(1 / b)
// (host table indexed by b) instead of the ~100-instruction IEEE division sequence:
//     q0 = RN(a * r);  e = a - q0 * b (exact, one FMA);  q = RN(q0 + e * r)
// which is the correctly rounded quotient RN(a / b) (Markstein's division step; checked exhaustively for every
// 0 <= a <= b <= 131072 by tools/check_recip_division.c), i.e. bit for bit what the division of population.rs:144-145
// returns; b = 0 (two empty genomes, no core genes) gives r = inf and a NaN, as 0.0 / 0.0 does.
// The kernel is software-pipelined over the rounds, for the generation pipeline where the warp shares its scheduler
// with eight core-kernel warps and every exposed global-load latency is paid in full: while the chain of round r runs
// over one half of a double-buffered ring,
//   * the reciprocals of round r + 1 are fetched (their addresses come from intersection counts loaded a round earlier),
//   * its quotients are evaluated into the other half of the ring between the two halves of the chain,
//   * the intersection counts and gene counts of round r + 2 are requested.
// The loads are volatile asm so that they are issued where they are written; two values per shared-memory load in the
// chain. Same additions in the same order: same bits.
constexpr uint32_t AVG_RCP_MAX = 131072;        // largest denominator the table may serve (range of the exhaustive check)

__device__ __forceinline__ uint32_t ldg_u32_v(const void *p)
{
    uint32_t v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ldg_f64_v(const void *p)
{
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

__global__ void __launch_bounds__(AVG_WARPS * 32, 4) avg_distance_pipe_kernel(const uint32_t *inter, const int32_t *num_genes,
                                                                             uint32_t n_rows, uint32_t core_genes,
                                                                             const double *__restrict__ rcp, double *avgdist)
{
    constexpr int PER = AVG_RING / 32;               // distances per lane per round
    __shared__ __align__(16) double ring[AVG_WARPS][2][AVG_RING];
    pdl_launch_dependents();       // the parent-selection CTA may take its SM slot now (it waits for this grid)
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t i = blockIdx.x * AVG_WARPS + warp;
    if (i >= n_rows) return;
    const uint32_t ki = (uint32_t)num_genes[i] + core_genes;
    const uint32_t *irow = inter + (uint64_t)i * n_rows;
    uint32_t in[PER], kj[PER];
    double rr[PER];
    auto load_counts = [&](uint32_t j0) {            // past the end: clamped (the values become +0.0 below)
#pragma unroll
        for (int q = 0; q < PER; q++) {
            const uint32_t j = min(j0 + q * 32 + lane, n_rows - 1u);
            in[q] = ldg_u32_v(irow + j);
            kj[q] = ldg_u32_v(num_genes + j);
        }
    };
    auto load_rcp = [&]() {
#pragma unroll
        for (int q = 0; q < PER; q++) rr[q] = ldg_f64_v(rcp + (ki + kj[q] - in[q]));
    };
    auto quotients = [&](uint32_t j0, double *buf) {
#pragma unroll
        for (int q = 0; q < PER; q++) {
            const uint32_t j = j0 + q * 32 + lane;
            const double da = (double)(in[q] + core_genes), db = (double)(ki + kj[q] - in[q]);
            const double q0 = da * rr[q];
            const double d = 1.0 - fma(fma(-q0, db, da), rr[q], q0);                  // population.rs:144-145
            buf[q * 32 + lane] = (j < n_rows && j != i) ? d : 0.0;                    // +0.0 never changes the (non-negative) sum
        }
    };
    double sum = 0.0;
    auto chain = [&](uint32_t base_s) {              // AVG_RING / 2 values, in order
#pragma unroll
        for (int c = 0; c < AVG_RING / 2; c += 2) {
            double x0, x1;
            asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x0), "=d"(x1) : "r"(base_s + c * 8u));
            sum += x0;
            sum += x1;
        }
    };
    load_counts(0u);
    load_rcp();
    quotients(0u, ring[warp][0]);
    load_counts(AVG_RING);
    __syncwarp();
    uint32_t b = 0;
    for (uint32_t j0 = 0; j0 < n_rows; j0 += AVG_RING, b ^= 1u) {
        const uint32_t cur = smem_u32(ring[warp][b]);
        load_rcp();                                              // round r + 1
        chain(cur);
        quotients(j0 + AVG_RING, ring[warp][b ^ 1u]);
        load_counts(j0 + 2 * AVG_RING);                          // round r + 2
        chain(cur + (AVG_RING / 2) * 8u);
        __syncwarp();
    }
    if (lane == 0) {
        double fd = sum / (double)(n_rows - 1u);
        if (fd == 0.0) fd = DBL_MIN;                                  // :774-776
        avgdist[i] = fd;
    }
}

// ---------------------------------------------------------------------------
// K3: weights (three softmaxes multiplied, population.rs:325-393), the all-zero
// rule (:403,435-437), WeightedIndex<f64> (cumulative + binary search, :440)
// and N draws from Philox(seed, gen, individual). Single CTA: N is small and
// the whole thing is a chain of reductions.
// ---------------------------------------------------------------------------
constexpr int SEL_THREADS = 256;      // one CTA slot of an SM: the kernel has to squeeze in beside the core step
constexpr int SEL_WARPS = SEL_THREADS / 32;

// block-wide reduction of three values at once (fixed order: shuffle tree, then the warp results
// in warp order), result in every thread
template <bool IS_MAX, int WARPS = SEL_WARPS>
__device__ __forceinline__ void block_reduce3(double &x, double &y, double &z, double (*scratch)[3])
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double tx = __shfl_xor_sync(0xffffffffu, x, o), ty = __shfl_xor_sync(0xffffffffu, y, o),
                     tz = __shfl_xor_sync(0xffffffffu, z, o);
        x = IS_MAX ? fmax(x, tx) : x + tx;
        y = IS_MAX ? fmax(y, ty) : y + ty;
        z = IS_MAX ? fmax(z, tz) : z + tz;
    }
    __syncthreads();
    if (lane == 0) { scratch[warp][0] = x; scratch[warp][1] = y; scratch[warp][2] = z; }
    __syncthreads();
    x = scratch[0][0]; y = scratch[0][1]; z = scratch[0][2];
#pragma unroll
    for (int q = 1; q < WARPS; q++) {
        x = IS_MAX ? fmax(x, scratch[q][0]) : x + scratch[q][0];
        y = IS_MAX ? fmax(y, scratch[q][1]) : y + scratch[q][1];
        z = IS_MAX ? fmax(z, scratch[q][2]) : z + scratch[q][2];
    }
}

struct SelectArgs {
    const double *logfit;
    const int32_t *num_genes;
    const double *avgdist;        // nullptr = all 1.0 (main.rs:435)
    uint32_t n_rows, n_genes;
    int32_t avg_gene_num;
    int32_t no_control_genome_size;
    double log_penalty;           // ln(genome_size_penalty), host libm
    double competition_strength;
    uint2 key;
    uint32_t gen;
    const uint32_t *gen_dev;      // nullptr, or a device word added to gen (replayed CUDA graphs)
    double *tmp_a, *tmp_b;        // [N] scratch
    double *weights;              // [N] out: final weights (population.rs:389-437)
    double *cumulative;           // [N] out
    uint32_t *parents;            // [N + 1] out: the parents, then a status word (1 = WeightedIndex::new would fail)
    int *err_flag;                // set to 1 if WeightedIndex::new would fail
};

// N <= 1024: the same computation with every per-individual value in registers (4 per thread) and
// the cumulative table in shared memory -- the kernel is a chain of dependent passes, so keeping
// them out of global memory is what makes it short.
constexpr int SEL_PER = 4;
constexpr uint32_t SEL_SMALL_MAX = SEL_THREADS * SEL_PER;

__global__ void __launch_bounds__(SEL_THREADS, 4) select_parents_small_kernel(const SelectArgs a)
{
    __shared__ double scratch[SEL_WARPS][3];
    __shared__ double warp_excl[SEL_WARPS + 1];
    __shared__ double w_s[SEL_SMALL_MAX];
    __shared__ double cum_s[SEL_SMALL_MAX];
    __shared__ int bad;
    const uint32_t n = a.n_rows, tid = threadIdx.x;
    const bool use_a = a.n_genes > 0, use_b = !a.no_control_genome_size;
    if (tid == 0) bad = 0;
    pdl_wait();                    // mean distances of avg_distance_kernel
    double xa[SEL_PER], xb[SEL_PER], xc[SEL_PER];
    double ma = -INFINITY, mb = -INFINITY, mc = -INFINITY;
#pragma unroll
    for (int k = 0; k < SEL_PER; k++) {
        const uint32_t i = tid + k * SEL_THREADS;
        const bool ok = i < n;
        const uint32_t ii = ok ? i : 0u;
        const double lf = a.logfit[ii];
        const int32_t ng = a.num_genes[ii];
        const double ad = a.avgdist ? a.avgdist[ii] : 1.0;
        xa[k] = ok ? (use_a ? lf : 0.0) : -INFINITY;
        xb[k] = ok ? (use_b ? (double)(ng - a.avg_gene_num) * a.log_penalty : 0.0) : -INFINITY;     // :350,355
        xc[k] = ok ? a.competition_strength * log(ad) : -INFINITY;                                  // :375
        ma = fmax(ma, xa[k]); mb = fmax(mb, xb[k]); mc = fmax(mc, xc[k]);
    }
    block_reduce3<true>(ma, mb, mc, scratch);
    double sa = 0.0, sb = 0.0, sc = 0.0;
#pragma unroll
    for (int k = 0; k < SEL_PER; k++) {        // entries beyond n are -inf: exp(-inf - m) = 0
        sa += exp(xa[k] - ma); sb += exp(xb[k] - mb); sc += exp(xc[k] - mc);
    }
    block_reduce3<false>(sa, sb, sc, scratch);
    const double la = (ma == -INFINITY) ? -INFINITY : ma + log(sa);
    const double lb = (mb == -INFINITY) ? -INFINITY : mb + log(sb);
    const double lc = (mc == -INFINITY) ? -INFINITY : mc + log(sc);
    double ta = 0.0, tb = 0.0, tc = 0.0;
#pragma unroll
    for (int k = 0; k < SEL_PER; k++) {
        xa[k] = exp(xa[k] - la); xb[k] = exp(xb[k] - lb); xc[k] = exp(xc[k] - lc);
        ta += xa[k]; tb += xb[k]; tc += xc[k];
    }
    block_reduce3<false>(ta, tb, tc, scratch);
    double w[SEL_PER];
    double mx = -INFINITY, dummy0 = -INFINITY, dummy1 = -INFINITY;
#pragma unroll
    for (int k = 0; k < SEL_PER; k++) {
        const double wa = use_a ? xa[k] / ta : 1.0;                 // a_i = 1 without an accessory genome (:293-296)
        const double w0 = use_b ? (xb[k] / tb) * wa : wa;           // :368 / :371
        w[k] = w0 * (xc[k] / tc);                                   // :391
        if (tid + k * SEL_THREADS < n) mx = fmax(mx, w[k]);
    }
    block_reduce3<true>(mx, dummy0, dummy1, scratch);
#pragma unroll
    for (int k = 0; k < SEL_PER; k++) {
        const uint32_t i = tid + k * SEL_THREADS;
        if (mx == 0.0) w[k] = 1.0;                                  // :435-437
        if (i < n) { w_s[i] = w[k]; a.weights[i] = w[k]; }
    }
    __syncthreads();
    // WeightedIndex::new: cumulative sums over contiguous chunks of 4, then a scan of the chunk totals
    const uint32_t lo = min(n, tid * SEL_PER), hi = min(n, lo + SEL_PER);
    double s = 0.0;
    bool mybad = false;
    for (uint32_t i = lo; i < hi; i++) {
        const double wi = w_s[i];
        if (!(wi >= 0.0)) mybad = true;
        s += wi;
    }
    if (mybad) bad = 1;
    const uint32_t lane = tid & 31, warp = tid >> 5;
    double v = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, v, o);
        if ((int)lane >= o) v += t;
    }
    if (lane == 31) scratch[warp][0] = v;
    __syncthreads();
    if (tid == 0) {
        double run = 0.0;
        for (int q = 0; q < SEL_WARPS; q++) { warp_excl[q] = run; run += scratch[q][0]; }
        warp_excl[SEL_WARPS] = run;
        if (!(run > 0.0) || isinf(run)) bad = 1;
    }
    __syncthreads();
    const double total = warp_excl[SEL_WARPS];
    double run = warp_excl[warp] + (v - s);
    for (uint32_t i = lo; i < hi; i++) {
        run += w_s[i];
        cum_s[i] = run;
        a.cumulative[i] = run;
    }
    __syncthreads();
    if (tid == 0) a.parents[n] = bad ? 1u : 0u;       // status word behind the vector: one read-back serves both
    if (bad) {
        if (tid == 0) *a.err_flag = 1;
        for (uint32_t i = tid; i < n; i += SEL_THREADS) a.parents[i] = i;
        return;
    }
    // N draws: u ~ U[0,total), index = #cumulative[0..n-1) <= u
#pragma unroll
    for (int k = 0; k < SEL_PER; k++) {
        const uint32_t i = tid + k * SEL_THREADS;
        const uint4 r = philox4x32_10(make_ctr(i, 0u, a.gen + (a.gen_dev ? __ldg(a.gen_dev) : 0u), STREAM_PARENTS), a.key);
        const uint64_t bits = (((uint64_t)r.x << 32) | r.y) >> 11;
        const double u = (double)bits * 0x1.0p-53 * total;
        uint32_t l = 0, h = n - 1;
        while (l < h) {
            const uint32_t mid = l + ((h - l) >> 1);
            if (cum_s[mid] <= u) l = mid + 1; else h = mid;
        }
        if (i < n) a.parents[i] = l;
    }
}

// The three softmaxes of population.rs:325-382 (fitness a, genome size b, competition c) are
// independent of each other, so each of their passes is made once for all three:
//   m = max v; s = sum exp(v - m); lse = m + ln s; e_i = exp(v_i - lse); out_i = e_i / sum e
// THREADS = 1024 for large populations: four times the lanes for the transcendental passes and the
// binary searches, and a CTA that owns its SM (nothing else fits beside 1024 threads), so the kernel
// is not slowed by the core step's CTAs once it has got its slot.
template <int THREADS>
__global__ void __launch_bounds__(THREADS) select_parents_kernel(const SelectArgs a)
{
    constexpr int WARPS = THREADS / 32;
    __shared__ double scratch[WARPS][3];
    __shared__ double warp_excl[WARPS + 1];
    __shared__ int bad;
    const uint32_t n = a.n_rows, tid = threadIdx.x;
    const bool use_a = a.n_genes > 0, use_b = !a.no_control_genome_size;
    double *va = a.tmp_a, *vb = a.tmp_b, *vc = a.cumulative;      // vc: scratch until the cumulative sums are written
    if (tid == 0) bad = 0;
    pdl_wait();                    // mean distances of avg_distance_kernel

    // pass 0: the three arguments and their maxima
    double ma = -INFINITY, mb = -INFINITY, mc = -INFINITY;
    for (uint32_t i = tid; i < n; i += THREADS) {
        const double xa = use_a ? a.logfit[i] : 0.0;
        const double xb = use_b ? (double)(a.num_genes[i] - a.avg_gene_num) * a.log_penalty : 0.0;     // :350,355
        const double xc = a.competition_strength * log(a.avgdist ? a.avgdist[i] : 1.0);                // :375
        vb[i] = xb; vc[i] = xc;
        ma = fmax(ma, xa); mb = fmax(mb, xb); mc = fmax(mc, xc);
    }
    block_reduce3<true, WARPS>(ma, mb, mc, scratch);
    // pass 1: log-sum-exp
    double sa = 0.0, sb = 0.0, sc = 0.0;
    for (uint32_t i = tid; i < n; i += THREADS) {
        if (use_a) sa += exp(a.logfit[i] - ma);
        if (use_b) sb += exp(vb[i] - mb);
        sc += exp(vc[i] - mc);
    }
    block_reduce3<false, WARPS>(sa, sb, sc, scratch);
    const double la = (ma == -INFINITY) ? -INFINITY : ma + log(sa);
    const double lb = (mb == -INFINITY) ? -INFINITY : mb + log(sb);
    const double lc = (mc == -INFINITY) ? -INFINITY : mc + log(sc);
    // pass 2: exp(v - lse) and their totals
    double ta = 0.0, tb = 0.0, tc = 0.0;
    for (uint32_t i = tid; i < n; i += THREADS) {
        const double ea = use_a ? exp(a.logfit[i] - la) : 1.0;
        const double eb = use_b ? exp(vb[i] - lb) : 1.0;
        const double ec = exp(vc[i] - lc);
        va[i] = ea; vb[i] = eb; vc[i] = ec;
        ta += ea; tb += eb; tc += ec;
    }
    block_reduce3<false, WARPS>(ta, tb, tc, scratch);
    // pass 3: weights (population.rs:365-393) and their maximum
    double mx = -INFINITY, dummy0 = -INFINITY, dummy1 = -INFINITY;
    for (uint32_t i = tid; i < n; i += THREADS) {
        const double wa = use_a ? va[i] / ta : 1.0;                 // a_i = 1 without an accessory genome (:293-296)
        const double w0 = use_b ? (vb[i] / tb) * wa : wa;           // :368 / :371
        const double w = w0 * (vc[i] / tc);                         // :391
        a.weights[i] = w;
        mx = fmax(mx, w);
    }
    block_reduce3<true, WARPS>(mx, dummy0, dummy1, scratch);
    if (mx == 0.0)                                                                       // :435-437
        for (uint32_t i = tid; i < n; i += THREADS) a.weights[i] = 1.0;
    __syncthreads();

    // WeightedIndex::new: cumulative sums; contiguous chunk per thread, then a scan of the chunk totals
    const uint32_t per = (n + THREADS - 1) / THREADS;
    const uint32_t lo = min(n, tid * per), hi = min(n, lo + per);
    double s = 0.0;
    bool mybad = false;
    for (uint32_t i = lo; i < hi; i++) {
        const double w = a.weights[i];
        if (!(w >= 0.0)) mybad = true;
        s += w;
    }
    if (mybad) bad = 1;
    const uint32_t lane = tid & 31, warp = tid >> 5;
    double v = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, v, o);
        if ((int)lane >= o) v += t;
    }
    if (lane == 31) scratch[warp][0] = v;
    __syncthreads();
    if (tid == 0) {
        double run = 0.0;
        for (int q = 0; q < WARPS; q++) { warp_excl[q] = run; run += scratch[q][0]; }
        warp_excl[WARPS] = run;
        if (!(run > 0.0) || isinf(run)) bad = 1;
    }
    __syncthreads();
    const double total = warp_excl[WARPS];
    double run = warp_excl[warp] + (v - s);
    for (uint32_t i = lo; i < hi; i++) {
        run += a.weights[i];
        a.cumulative[i] = run;
    }
    __syncthreads();
    if (tid == 0) a.parents[n] = bad ? 1u : 0u;       // status word behind the vector: one read-back serves both
    if (bad) {
        if (tid == 0) *a.err_flag = 1;
        for (uint32_t i = tid; i < n; i += THREADS) a.parents[i] = i;
        return;
    }
    // N draws: u ~ U[0,total), index = #cumulative[0..n-1) <= u
    for (uint32_t i = tid; i < n; i += THREADS) {
        const uint4 r = philox4x32_10(make_ctr(i, 0u, a.gen + (a.gen_dev ? __ldg(a.gen_dev) : 0u), STREAM_PARENTS), a.key);
        const uint64_t bits = (((uint64_t)r.x << 32) | r.y) >> 11;
        const double u = (double)bits * 0x1.0p-53 * total;
        uint32_t l = 0, h = n - 1;
        while (l < h) {
            const uint32_t mid = l + ((h - l) >> 1);
            if (a.cumulative[mid] <= u) l = mid + 1; else h = mid;
        }
        a.parents[i] = l;
    }
}

}  // namespace pansim
