// vcf.cuh -- the core alignment as VCF text, expanded on the device (DESIGN.md section 11).
//
// Site pass: from the per-site allele counts (diversity_kernel<true, false>) and the packed ancestral row,
// vcf_site_kernel gives every site a one-byte descriptor (REF code in bits 0-1, ALT mask in bits 2-5,
// ALT = 0: the site is not written) and every 2048-site block its text length. vcf_scan_blocks_kernel
// and vcf_offsets_kernel turn the lengths into every line's byte offset (an exclusive scan of integers,
// deterministic), and vcf_chunk_kernel cuts the sites greedily into chunks of at most `cap` bytes (one
// line where a line alone is longer), so the host reads back only the chunk boundaries.
//
// Expansion: vcf_expand_kernel writes the lines of one chunk. A CTA owns a tile of 128 sites (8 packed
// words, one 32-byte sector per row) and a block of 256 rows. Each thread loads one packed word of 16
// rows and transposes the 16 x 16 block of 2-bit codes in registers, so shared memory holds the tile
// site-major: per site, the codes of the block's rows as a bit string. Every byte of a line's genotype
// span "\tg_0\tg_1..." is a function of its position q alone ('\t' at even q, the digit of row q/2 at odd
// q), so a warp writes one site's span of the row block with aligned 16-byte stores, one per lane, and
// byte stores only where the span begins or ends inside a 16-byte word. The CTA of row block 0 also
// writes the fixed prefix "core\tPOS\t.\tREF\tALT\t.\t.\t.\tGT", the last row block the newline.
#pragma once
#include "common.cuh"

namespace pansim {

constexpr uint32_t VS_THREADS = 256;
constexpr uint32_t VS_PER_THREAD = 8;                   // consecutive sites per thread in the scan
constexpr uint32_t VS_SITES = VS_THREADS * VS_PER_THREAD;   // 2048 sites per scan block
constexpr uint32_t VS_SCAN_THREADS = 1024;              // the single CTA of the block scan and of the chunking
constexpr uint32_t VX_SITES = 128;                      // sites per expansion tile: 8 packed words
constexpr uint32_t VX_ROWS = 256;                       // rows per row block
constexpr uint32_t VX_GROUPS = VX_ROWS / 16 + 1;        // row groups of 16 loaded per block: its own and one more
constexpr uint32_t VX_THREADS = 256;                    // the first 8 * VX_GROUPS: one transpose (word x row group) each
constexpr uint32_t VX_WARPS = VX_THREADS / 32;
constexpr uint32_t VX_PITCH = VX_GROUPS + 1;            // words per site column: the groups and a pad word
// fixed text of a line: "core\t" POS "\t.\t" REF "\t" ALT "\t.\t.\t.\tGT" genotypes "\n"
constexpr uint32_t VCF_FIXED_BYTES = 19;                // + digits(POS) + 2 |ALT| + 2 N

__host__ __device__ inline uint32_t vcf_digits(uint64_t x)
{
    uint32_t d = 1;
    while (x >= 10) { x /= 10; d++; }
    return d;
}

// bytes of the line of a site with descriptor `desc` (0 when the site is not written)
__device__ __forceinline__ uint64_t vcf_line_bytes(uint32_t desc, uint64_t pos, uint32_t n_rows)
{
    const uint32_t alt = desc >> 2;
    return alt ? VCF_FIXED_BYTES + vcf_digits(pos) + 2ull * __popc(alt) + 2ull * n_rows : 0ull;
}

struct VcfSiteArgs {
    const uint4 *counts;            // [n_sites] (n_A, n_C, n_G, n_T)
    const uint32_t *anc;            // packed ancestral row
    uint64_t n_sites;               // local sites
    uint64_t pos0;                  // POS of local site 0 (site_begin + 1)
    uint32_t n_rows;
    uint8_t *desc;                  // [n_blocks * VS_SITES]; 0 past n_sites
    unsigned long long *off;        // [n_sites + 1] line offsets (vcf_offsets_kernel)
    unsigned long long *block;      // [n_blocks] bytes per block, then their exclusive scan
};

// block-wide exclusive scan of one value per thread (blockDim.x = VS_THREADS); returns the block total in *total
__device__ __forceinline__ unsigned long long vcf_block_scan(unsigned long long v, unsigned long long *s_warp, unsigned long long *total)
{
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    unsigned long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = lane < nw ? s_warp[lane] : 0ull;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, w, o);
            if (lane >= (uint32_t)o) w += y;
        }
        if (lane < nw) s_warp[lane] = w;          // inclusive over warps
    }
    __syncthreads();
    const unsigned long long before = (warp ? s_warp[warp - 1] : 0ull) + x - v;
    *total = s_warp[nw - 1];
    __syncthreads();                               // s_warp is reused by the caller's next scan
    return before;
}

// descriptors and per-block text bytes; thread t of block b takes sites b*VS_SITES + 8t .. 8t+7
__global__ void __launch_bounds__(VS_THREADS) vcf_site_kernel(VcfSiteArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t s0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    uint32_t d[VS_PER_THREAD];
    unsigned long long bytes = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        const uint64_t s = s0 + i;
        d[i] = 0;
        if (s < a.n_sites) {
            const uint4 n = a.counts[s];
            const uint32_t ref = (__ldg(a.anc + (s >> 4)) >> (2 * (s & 15u))) & 3u;
            const uint32_t present = (n.x > 0) | (n.y > 0) << 1 | (n.z > 0) << 2 | (n.w > 0) << 3;
            d[i] = ref | (present & ~(1u << ref)) << 2;
            bytes += vcf_line_bytes(d[i], a.pos0 + s, a.n_rows);
        }
    }
    uint2 packed;
    packed.x = d[0] | d[1] << 8 | d[2] << 16 | d[3] << 24;
    packed.y = d[4] | d[5] << 8 | d[6] << 16 | d[7] << 24;
    reinterpret_cast<uint2 *>(a.desc)[s0 / VS_PER_THREAD] = packed;
    unsigned long long total;
    vcf_block_scan(bytes, s_warp, &total);
    if (threadIdx.x == 0) a.block[blockIdx.x] = total;
}

// one CTA: exclusive scan of the block totals in place, off[n_sites] = the whole text
__global__ void __launch_bounds__(VS_SCAN_THREADS) vcf_scan_blocks_kernel(unsigned long long *block, uint32_t n_blocks,
                                                                          unsigned long long *end)
{
    __shared__ unsigned long long s_warp[VS_SCAN_THREADS / 32];
    unsigned long long carry = 0;
    for (uint32_t b0 = 0; b0 < n_blocks; b0 += VS_SCAN_THREADS) {
        const uint32_t b = b0 + threadIdx.x;
        const unsigned long long v = b < n_blocks ? block[b] : 0ull;
        unsigned long long total;
        const unsigned long long before = vcf_block_scan(v, s_warp, &total);
        if (b < n_blocks) block[b] = carry + before;
        carry += total;
    }
    if (threadIdx.x == 0) *end = carry;
}

// every site's line offset: the block's scanned base plus the exclusive scan inside the block
__global__ void __launch_bounds__(VS_THREADS) vcf_offsets_kernel(VcfSiteArgs a)
{
    __shared__ unsigned long long s_warp[VS_THREADS / 32];
    const uint64_t s0 = (uint64_t)blockIdx.x * VS_SITES + threadIdx.x * VS_PER_THREAD;
    const uint2 packed = reinterpret_cast<const uint2 *>(a.desc)[s0 / VS_PER_THREAD];
    unsigned long long len[VS_PER_THREAD], bytes = 0;
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        const uint32_t d = ((i < 4 ? packed.x : packed.y) >> (8 * (i & 3))) & 0xFFu;
        len[i] = vcf_line_bytes(d, a.pos0 + s0 + i, a.n_rows);
        bytes += len[i];
    }
    unsigned long long total;
    unsigned long long o = a.block[blockIdx.x] + vcf_block_scan(bytes, s_warp, &total);
#pragma unroll
    for (uint32_t i = 0; i < VS_PER_THREAD; i++) {
        if (s0 + i < a.n_sites) a.off[s0 + i] = o;
        o += len[i];
    }
}

// One CTA: greedy chunks over the sites. Chunk k = sites [bounds[2k], bounds[2k+2]) starting at byte
// bounds[2k+1]; its end is the largest e with off[e] - off[start] <= cap, at least start + 1. The search
// probes VS_SCAN_THREADS offsets per round, so a chunk costs about log_1024(sites) rounds.
__global__ void __launch_bounds__(VS_SCAN_THREADS) vcf_chunk_kernel(const unsigned long long *off, uint64_t n_sites,
                                                                    unsigned long long cap, unsigned long long *bounds,
                                                                    uint32_t *n_chunks)
{
    __shared__ unsigned long long s_best;
    uint64_t s = 0;
    uint32_t k = 0;
    for (;;) {
        if (threadIdx.x == 0) { bounds[2 * (uint64_t)k] = s; bounds[2 * (uint64_t)k + 1] = off[s]; }
        if (s >= n_sites) break;
        const unsigned long long limit = off[s] + cap;
        uint64_t lo = s + 1, hi = n_sites;            // the end lies in [lo, hi]; off[lo] <= limit or lo = s + 1
        while (lo < hi) {
            const uint64_t step = (hi - lo + VS_SCAN_THREADS - 1) / VS_SCAN_THREADS;
            if (threadIdx.x == 0) s_best = lo;
            __syncthreads();
            const uint64_t p = lo + step * (threadIdx.x + 1);
            if (p <= hi && off[p] <= limit) atomicMax(&s_best, (unsigned long long)p);
            __syncthreads();
            const uint64_t best = s_best;
            __syncthreads();
            hi = min(hi, best + step - 1);          // probe best + step (if any) failed: offsets never decrease
            lo = best;
        }
        s = lo;
        k++;
    }
    if (threadIdx.x == 0) *n_chunks = k;
}

struct VcfExpandArgs {
    const uint32_t *state;          // packed rows (16 sites per word), row pitch row_words
    uint64_t row_words;
    uint32_t n_rows;
    const uint8_t *desc;
    const unsigned long long *off;
    uint64_t site0, site1;          // the chunk: local sites [site0, site1)
    unsigned long long base;        // off[site0], byte 0 of `out`
    uint64_t pos0;                  // POS of local site 0
    char *out;
};

// byte k (< 8) of the little-endian packed string x
__device__ __forceinline__ char vcf_byte(uint64_t x, uint32_t k) { return (char)((x >> (8 * k)) & 0xFFu); }

// byte k of the fixed prefix "core\tPOS\t.\tREF\tALT\t.\t.\t.\tGT" (nd digits of POS, n_alt letters in ALT);
// the fixed parts are packed into integers so that nothing is indexed in local memory
__device__ __forceinline__ char vcf_prefix_byte(uint32_t k, uint64_t pos, uint32_t nd, uint32_t ref, uint32_t alt, uint32_t n_alt)
{
    const uint64_t LETTERS = 0x54474341ull;              // "ACGT"
    const uint64_t CORE = 0x0965726F63ull;               // "core\t"
    const uint64_t DOT = 0x092E09ull;                    // "\t.\t"
    const uint64_t TAIL = 0x2E092E092E092E09ull;         // "\t.\t.\t.\t." ... the last of the 9 bytes of "\t.\t.\t.\tGT"
    if (k < 5) return vcf_byte(CORE, k);
    k -= 5;
    if (k < nd) {
        for (uint32_t i = k + 1; i < nd; i++) pos /= 10;
        return (char)('0' + pos % 10);
    }
    k -= nd;
    if (k < 3) return vcf_byte(DOT, k);
    k -= 3;
    if (k == 0) return vcf_byte(LETTERS, ref);
    if (k == 1) return '\t';
    k -= 2;
    if (k < 2 * n_alt - 1) {
        if (k & 1) return ',';
        uint32_t m = alt;
        for (uint32_t i = 0; i < k / 2; i++) m &= m - 1;   // drop the lower ALT alleles
        return vcf_byte(LETTERS, __ffs(m) - 1);
    }
    k -= 2 * n_alt - 1;                                    // "\t.\t.\t.\tGT"
    return k < 7 ? vcf_byte(TAIL, k) : k == 7 ? 'G' : 'T';
}

// one stage of the 16 x 16 transpose of 2-bit codes: swap the B x B blocks off the diagonal of every 2B x 2B
// block (m selects the codes i with i & B == 0)
template <uint32_t B>
__device__ __forceinline__ void vcf_transpose_stage(uint32_t (&x)[16], uint32_t m)
{
#pragma unroll
    for (uint32_t k = 0; k < 16; k++) {
        if (k & B) continue;
        const uint32_t t = ((x[k] >> (2 * B)) ^ x[k + B]) & m;
        x[k] ^= t << (2 * B);
        x[k + B] ^= t;
    }
}

// grid: x = tiles of the chunk, y = row blocks
__global__ void __launch_bounds__(VX_THREADS) vcf_expand_kernel(VcfExpandArgs a)
{
    __shared__ uint32_t s_col[VX_SITES * VX_PITCH];   // s_col[site][j]: 2-bit codes of rows r0 + 16j .. r0 + 16j + 15
    __shared__ unsigned long long s_off[VX_SITES];   // line offset of each written site, relative to `out`
    __shared__ uint32_t s_list[VX_SITES];          // tile positions of the written sites, then their descriptors
    __shared__ uint32_t s_n;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint64_t tile = a.site0 / VX_SITES + blockIdx.x;
    const uint32_t r0 = blockIdx.y * VX_ROWS;
    const uint32_t nr = min(VX_ROWS, a.n_rows - r0);

    // the written sites of the tile inside the chunk with their descriptors and offsets (the order does not
    // matter: every byte has its place)
    if (tid == 0) s_n = 0;
    __syncthreads();
    if (tid < VX_SITES) {
        const uint64_t s = tile * VX_SITES + tid;
        const uint32_t d = (s >= a.site0 && s < a.site1) ? a.desc[s] : 0u;
        if (d >> 2) {
            const uint32_t k = atomicAdd(&s_n, 1u);
            s_list[k] = tid | d << 8;
            s_off[k] = a.off[s] - a.base;
        }
    }
    __syncthreads();
    const uint32_t n_list = s_n;
    if (n_list == 0) return;

    // transpose: thread = (packed word w of the tile, row group j); x[k] = word of row r0 + 16j + k. Group 16
    // holds the first rows of the next block: the last vectors of a span reach up to 7 rows past the block.
    if (tid < 8 * VX_GROUPS) {
        const uint32_t w = tid & 7u, j = tid >> 3;
        const uint32_t *src = a.state + tile * (VX_SITES / 16) + w;
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
        // now x[i] = codes of the group's 16 rows at site 16w + i, row k in bits 2k
#pragma unroll
        for (uint32_t i = 0; i < 16; i++) s_col[(16 * w + i) * VX_PITCH + j] = x[i];
        if (tid < VX_SITES) s_col[tid * VX_PITCH + VX_PITCH - 1] = 0;
    }
    __syncthreads();

    // Every aligned 16-byte word of the output belongs to the row block that holds its first byte inside the
    // line (the line's first byte for the word where the line starts). Words inside the genotype span are
    // written whole; in the two words where the span begins and ends, the genotype bytes and the newline are
    // written one by one. The prefix is written by the lanes of the first block's warp, a byte each.
    const bool first_block = blockIdx.y == 0, last_block = r0 + nr == a.n_rows;
    const uint64_t span = 2 * (uint64_t)a.n_rows;
    for (uint32_t li = warp; li < n_list; li += VX_WARPS) {
        const uint32_t i = s_list[li] & 0xFFu, d = s_list[li] >> 8;
        const uint64_t s = tile * VX_SITES + i;
        const uint32_t ref = d & 3u, alt = d >> 2, n_alt = __popc(alt);
        // digit of each code: '0' for REF, else 1 + its index in ALT (A, C, G, T order)
        uint32_t lut = 0;
#pragma unroll
        for (uint32_t c = 0; c < 4; c++) {
            const uint32_t g = c == ref ? 0u : 1u + __popc(alt & ((1u << c) - 1u));
            lut |= ('0' + g) << (8 * c);
        }
        const uint64_t pos = a.pos0 + s;
        const uint32_t nd = vcf_digits(pos);
        const uint32_t P = VCF_FIXED_BYTES - 1 + nd + 2 * n_alt;      // prefix bytes
        char *ls = a.out + s_off[li];                                 // the line: [ls, le)
        char *g = ls + P;                                             // genotype span: byte q at g + q
        char *le = g + span + 1;
        char *lo = first_block ? ls : g + 2 * (uint64_t)r0;           // the block's bytes of the line: [lo, hi)
        char *hi = last_block ? le : g + 2 * (uint64_t)(r0 + nr);
        char *v0 = reinterpret_cast<char *>(first_block ? reinterpret_cast<uintptr_t>(lo) & ~uintptr_t(15)
                                                        : (reinterpret_cast<uintptr_t>(lo) + 15) & ~uintptr_t(15));
        const uint32_t n_vec = hi > v0 ? (uint32_t)((hi - v0 + 15) / 16) : 0u;
        const uint32_t *col = s_col + i * VX_PITCH;
        if (first_block)
            for (uint32_t k = lane; k < P; k += 32) ls[k] = vcf_prefix_byte(k, pos, nd, ref, alt, n_alt);
        for (uint32_t v = lane; v < n_vec; v += 32) {
            char *A = v0 + 16 * (uint64_t)v;
            if (A + 16 <= g) continue;                                // prefix only: written above
            if (A >= g && A + 16 <= g + span) {                       // genotypes only: rows rel .. rel + 7
                const int64_t q0 = A - g;
                const uint32_t rel = (uint32_t)(q0 >> 1) - r0;
                const uint32_t bits = __funnelshift_r(col[rel >> 4], col[(rel >> 4) + 1], 2 * (rel & 15u));
                uint32_t dg[8];
#pragma unroll
                for (int k = 0; k < 8; k++) dg[k] = (lut >> (8 * ((bits >> (2 * k)) & 3u))) & 0xFFu;
                uint4 o;
                if (q0 & 1) {           // digit, tab, digit, tab, ...
                    o.x = dg[0] | 0x0900u | dg[1] << 16 | 0x09000000u;
                    o.y = dg[2] | 0x0900u | dg[3] << 16 | 0x09000000u;
                    o.z = dg[4] | 0x0900u | dg[5] << 16 | 0x09000000u;
                    o.w = dg[6] | 0x0900u | dg[7] << 16 | 0x09000000u;
                } else {                // tab, digit, tab, digit, ...
                    o.x = 0x09u | dg[0] << 8 | 0x090000u | dg[1] << 24;
                    o.y = 0x09u | dg[2] << 8 | 0x090000u | dg[3] << 24;
                    o.z = 0x09u | dg[4] << 8 | 0x090000u | dg[5] << 24;
                    o.w = 0x09u | dg[6] << 8 | 0x090000u | dg[7] << 24;
                }
                *reinterpret_cast<uint4 *>(A) = o;
            } else {                    // where the span begins or ends: genotype bytes and the newline
                for (uint32_t k = 0; k < 16; k++) {
                    char *p = A + k;
                    if (p < g || p >= le) continue;
                    const uint64_t q = (uint64_t)(p - g);
                    char ch = '\n';
                    if (q < span) {
                        ch = '\t';
                        if (q & 1) {
                            const uint32_t rel = (uint32_t)(q >> 1) - r0;
                            ch = (char)((lut >> (8 * ((col[rel >> 4] >> (2 * (rel & 15u))) & 3u))) & 0xFFu);
                        }
                    }
                    *p = ch;
                }
            }
        }
    }
}

}  // namespace pansim
