// fasta.cuh -- the core alignment as FASTA text, expanded on the device (DESIGN.md section 14).
//
// Site pass (SNP mode only): from the per-site allele counts (diversity_kernel<true, false>),
// fasta_site_kernel marks the polymorphic sites (two or more letters present) of every 2048-site block,
// counts them per block and adds the letters of the constant sites into const_counts[4] (integer atomics,
// deterministic). vcf_scan_blocks_kernel scans the block totals and fasta_compact_kernel writes the
// polymorphic sites, ascending, into the column list. Padding sites (past n_sites) are never columns.
//
// Expansion: fasta_expand_kernel writes the records of a block of rows, row-major. A CTA owns FX_COLS columns
// of FX_ROWS rows. It first turns its columns (plus the next 16, see below) into (packed word, kept-site mask,
// first column) triples in shared memory: the mask is the same for every row, so each row loads each packed
// word it needs once. Whole mode is the identity column map (no list). A warp then takes one row at a time:
// its lanes load the row's words and place the kept letters in a per-warp row buffer, then write the row's
// text as aligned 16-byte words. A word belongs to the chunk that holds its first letter; it is stored whole
// when it holds letters only (the staged 16 columns past the chunk cover its tail), byte by byte where the
// letters begin or end. The CTAs of column chunk 0 also write the header `>ind_<i>\n` and the newline.
// Without framing (the letters-only export) row i's letters start at (i - row0) * columns.
#pragma once
#include "common.cuh"
#include "vcf.cuh"

namespace pansim {

constexpr uint32_t FX_COLS = 1024;                      // columns per CTA
constexpr uint32_t FX_STAGE = FX_COLS + 16;             // staged columns: the tail of the chunk's last word
constexpr uint32_t FX_ROWS = 64;                        // rows per CTA
constexpr uint32_t FX_THREADS = 256;
constexpr uint32_t FX_WARPS = FX_THREADS / 32;
constexpr uint32_t FX_BUF_WORDS = (FX_STAGE + 16) / 4;  // per-warp row buffer: the staged letters and a word of slack

// byte offset of record i when every record holds `cols` letters: sum over j < i of 7 + digits(j) + cols
__host__ __device__ inline uint64_t fasta_record_offset(uint64_t i, uint64_t cols)
{
    uint64_t o = i * (7 + cols) + i;                     // one digit each
    for (uint64_t p = 10; p <= i; p *= 10) o += i - p;   // one more for every j >= 10, 100, ...
    return o;
}

__device__ __forceinline__ bool fasta_polymorphic(uint4 n)
{
    return (n.x > 0) + (n.y > 0) + (n.z > 0) + (n.w > 0) >= 2;
}

struct FastaSiteArgs {
    const uint4 *counts;            // [n_sites] (n_A, n_C, n_G, n_T)
    uint64_t n_sites;
    unsigned long long *block;      // [n_blocks + 1] polymorphic sites per block, then their exclusive scan (+ total)
    unsigned long long *consts;     // [4] constant sites by letter (zeroed by the caller)
    uint32_t *cols;                 // [polymorphic sites] local site index of every column
};

// polymorphic sites per block and the letters of the constant ones; thread t of block b takes sites b*VS_SITES + 8t .. 8t+7
__global__ void __launch_bounds__(VS_THREADS) fasta_site_kernel(FastaSiteArgs a)
{
    __shared__ unsigned long long s_sum[5];
    if (threadIdx.x < 5) s_sum[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t s0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    uint32_t v[5] = {0, 0, 0, 0, 0};                     // constant A, C, G, T; polymorphic
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        if (s0 + i >= a.n_sites) break;
        const uint4 n = a.counts[s0 + i];
        if (fasta_polymorphic(n)) v[4]++;
        else if (n.x) v[0]++;
        else if (n.y) v[1]++;
        else if (n.z) v[2]++;
        else if (n.w) v[3]++;
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {
        const uint32_t w = __reduce_add_sync(0xFFFFFFFFu, v[k]);
        if ((threadIdx.x & 31u) == 0 && w) atomicAdd(&s_sum[k], (unsigned long long)w);
    }
    __syncthreads();
    if (threadIdx.x < 4 && s_sum[threadIdx.x]) atomicAdd(&a.consts[threadIdx.x], s_sum[threadIdx.x]);
    if (threadIdx.x == 4) a.block[blockIdx.x] = s_sum[4];
}

// the column list: every polymorphic site at the block's scanned base plus its rank inside the block
__global__ void __launch_bounds__(VS_THREADS) fasta_compact_kernel(FastaSiteArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t s0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    uint32_t poly = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++)
        if (s0 + i < a.n_sites && fasta_polymorphic(a.counts[s0 + i])) poly |= 1u << i;
    unsigned long long total;
    uint64_t k = a.block[blockIdx.x] + vcf_block_scan(__popc(poly), s_warp, &total);
    for (; poly; poly &= poly - 1) a.cols[k++] = (uint32_t)(s0 + __ffs(poly) - 1);
}

struct FastaExpandArgs {
    const uint32_t *state;          // packed rows (16 sites per word), row pitch row_words
    uint64_t row_words;
    const uint32_t *cols;           // [n_cols] local site of every column, or null: column k is site k
    uint64_t n_cols;
    uint32_t row0, row1;            // the rows of the chunk; row0's record (or letters) starts at byte 0 of `out`
    uint32_t framed;                // 1: records `>ind_<i>\n` letters `\n`; 0: letters only
    char *out;
};

__device__ __forceinline__ uint32_t fasta_letter(uint32_t code) { return (0x54474341u >> (8 * code)) & 0xFFu; }   // "ACGT"

// grid: x = column chunks (at least one), y = row blocks
__global__ void __launch_bounds__(FX_THREADS) fasta_expand_kernel(FastaExpandArgs a)
{
    __shared__ uint32_t s_word[FX_STAGE], s_mask[FX_STAGE], s_k0[FX_STAGE];
    __shared__ uint32_t s_lut[256];                      // a byte of four codes -> their four letters
    __shared__ __align__(16) uint32_t s_buf[FX_WARPS][FX_BUF_WORDS];
    __shared__ uint32_t s_wn[FX_WARPS];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint64_t C = a.n_cols, c0 = (uint64_t)blockIdx.x * FX_COLS;
    const uint64_t ce = min(C, c0 + FX_COLS);
    const uint32_t n_stage = (uint32_t)(min(C, c0 + FX_STAGE) - min(C, c0));

    s_lut[tid] = fasta_letter(tid & 3u) | fasta_letter((tid >> 2) & 3u) << 8 | fasta_letter((tid >> 4) & 3u) << 16 |
                 fasta_letter(tid >> 6) << 24;
    __syncthreads();
    // the staged columns as (word, mask, first column) triples: a column opens a triple when its word differs from
    // the previous column's; ballots and a scan over the warps number the triples
    uint32_t n_pairs = 0;
    for (uint32_t b = 0; b < n_stage; b += FX_THREADS) {
        const uint32_t k = b + tid;
        uint32_t site = 0;
        bool open = false;
        if (k < n_stage) {
            const uint64_t q = c0 + k;
            site = a.cols ? a.cols[q] : (uint32_t)q;
            open = k == 0 || (site >> 4) != ((a.cols ? a.cols[q - 1] : (uint32_t)(q - 1)) >> 4);
        }
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, open);
        if (lane == 0) s_wn[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = n_pairs, total = n_pairs;
        for (uint32_t w = 0; w < FX_WARPS; w++) {
            before += w < warp ? s_wn[w] : 0u;
            total += s_wn[w];
        }
        const uint32_t p = before + __popc(bal & (0xFFFFFFFFu >> (31 - lane))) - 1;   // the triple of column k
        if (open) { s_word[p] = site >> 4; s_mask[p] = 0; s_k0[p] = k; }
        __syncthreads();
        if (k < n_stage) atomicOr(&s_mask[p], 1u << (site & 15u));
        n_pairs = total;
        __syncthreads();
    }

    uint8_t *buf = reinterpret_cast<uint8_t *>(s_buf[warp]);
    const uint32_t r_end = min(a.row1, a.row0 + (blockIdx.y + 1) * FX_ROWS);
    const uint64_t rec0 = a.framed ? fasta_record_offset(a.row0, C) : 0;
    for (uint32_t r = a.row0 + blockIdx.y * FX_ROWS + warp; r < r_end; r += FX_WARPS) {
        const uint32_t *row = a.state + (uint64_t)r * a.row_words;
        for (uint32_t j = lane; j < n_pairs; j += 32) {
            const uint32_t x = __ldg(row + s_word[j]);
            uint32_t m = s_mask[j], k = s_k0[j];
            if (m == 0xFFFFu && !(k & 15u)) {
                *reinterpret_cast<uint4 *>(buf + k) = make_uint4(s_lut[x & 0xFFu], s_lut[(x >> 8) & 0xFFu],
                                                                 s_lut[(x >> 16) & 0xFFu], s_lut[x >> 24]);
            } else {
                for (; m; m &= m - 1) buf[k++] = (uint8_t)fasta_letter((x >> (2 * (__ffs(m) - 1))) & 3u);
            }
        }
        __syncwarp();
        const uint32_t nd = vcf_digits(r);
        const uint64_t G = a.framed ? fasta_record_offset(r, C) - rec0 + 6 + nd : (uint64_t)(r - a.row0) * C;   // the letters: [G, G + C)
        if (a.framed && blockIdx.x == 0) {
            for (uint32_t k = lane; k < 6 + nd; k += 32) {
                char ch = '\n';
                if (k < 5) ch = (char)((0x5F646E693Eull >> (8 * k)) & 0xFFu);   // ">ind_"
                else if (k < 5 + nd) {
                    uint32_t v = r;
                    for (uint32_t i = k + 1; i < 5 + nd; i++) v /= 10;
                    ch = (char)('0' + v % 10);
                }
                a.out[G - 6 - nd + k] = ch;
            }
            if (lane == 0) a.out[G + C] = '\n';
        }
        const uint64_t Gs = G + c0;
        const uint64_t A0 = c0 == 0 ? G & ~15ull : (Gs + 15) & ~15ull;
        for (uint64_t A = A0 + 16 * lane; A < G + ce; A += 16 * 32) {
            if (A >= G && A + 16 <= G + C) {                 // letters only
                const uint32_t o = (uint32_t)(A - Gs), w = o >> 2, sh = 8 * (o & 3u);
                const uint32_t *bw = s_buf[warp] + w;
                uint4 v;
                v.x = __funnelshift_r(bw[0], bw[1], sh);
                v.y = __funnelshift_r(bw[1], bw[2], sh);
                v.z = __funnelshift_r(bw[2], bw[3], sh);
                v.w = __funnelshift_r(bw[3], bw[4], sh);
                *reinterpret_cast<uint4 *>(a.out + A) = v;
            } else {                                         // where the letters begin or end
                const uint64_t p1 = min(A + 16, G + C);
                for (uint64_t p = max(A, G); p < p1; p++) a.out[p] = (char)buf[p - Gs];
            }
        }
        __syncwarp();
    }
}

}  // namespace pansim
