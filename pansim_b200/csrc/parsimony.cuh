// parsimony.cuh -- parsimony changes of every core site or accessory gene on a rooted node table (DESIGN.md section
// 17; the definitions are in include/pansim_b200.h): Hartigan's (1973) bottom-up sets and scores, then one optimal
// assignment top-down, with the changes counted per character and per branch.
//
// One thread owns a column of 32 characters: for the core the two packed words of 16 sites (bit 2s of a plane is
// site s of the column, bit 2s + 1 site 16 + s), for the genes one accessory word. A node's set is NS one-hot bit
// planes (NS = 4 letters A < C < G < T, or 2: absent < present). Lanes of a warp take consecutive columns, so every
// row read and every scratch read of a warp is one contiguous run. Every thread walks the same nodes in the same
// order: the branches below are uniform over the CTA.
//
// Bottom-up: internal node N + v, v = 0 .. n_internal - 1 (ascending ids: children before parents), reads its
// children from the host-built CSR list; a leaf's set comes from its packed row, an internal node's from
// scratch[v][column]. Two children take Fitch's bit-sliced step (I = A & B; empty = no state in I; S = empty ? A | B :
// I; the score gains `empty`). k >= 3 children count every state in bit-sliced counters of ceil(log2(k + 1)) planes
// (shared memory, one column of counters per thread), take the bit-sliced maximum m from the top plane down (the
// states still equal to the maximum are S), and add k - m to the score. The score of each character is a 32-plane
// bit-sliced counter in registers (at most N - 1, so it never overflows). The set is written to scratch.
// Top-down in the same thread: the root takes the smallest state of its set. Internal nodes in descending id order
// read their assigned state and, for each child, compare it with the child's set (internal child: the child takes the
// parent's state when it is in its set, else the smallest state of its set, written over its scratch slot) or the
// child's letter (leaf). The branch's changes are counted by redux.sync per warp, in shared counters per CTA (one per
// position of the CSR list, 256 positions at a time), and added to global memory with one 64-bit atomic per (CTA,
// branch) when the walk leaves those positions. Finally each thread writes the u32 score of its characters and adds
// the summary terms (the per-character allele or presence counts come from the existing count kernels).
#pragma once
#include "common.cuh"

namespace pansim {

constexpr uint32_t PS_THREADS = 128;
constexpr uint32_t PS_SLOTS = 256;          // CSR positions whose branch counters a CTA holds in shared memory

struct ParsimonyArgs {
    const uint32_t *rows;                   // packed core rows (two words per column) or accessory rows (one word)
    uint64_t row_words;                     // row pitch in words
    uint32_t n_leaves, n_internal;
    const uint32_t *child_off;              // [n_internal + 1]: children of node n_leaves + v at child[child_off[v] ..]
    const uint32_t *child;                  // [n_nodes - 1]
    uint64_t col0;                          // first column of this slab
    uint32_t cols_pad;                      // scratch pitch: the slab's columns rounded up to the CTA
    uint64_t n_cols;                        // columns of the whole character range
    uint64_t n_chars;                       // sites / genes: characters at or past it are padding
    uint32_t dmax;                          // counter planes reserved per state in shared memory (bits of n_leaves)
    void *scratch;                          // [n_internal][cols_pad] sets (uint4 / uint2)
    const uint4 *site_counts;               // core: (nA, nC, nG, nT) per site
    const uint32_t *gene_counts;            // genes: presence count per gene
    uint32_t *scores;                       // [n_chars]
    unsigned long long *summary;            // [5]: variable, tree_length, min_changes, max_changes, homoplastic
    unsigned long long *branch0, *branch1;  // [n_nodes]: core changes / gene gains, gene losses
};

template <int NS> struct PsSet { uint32_t p[NS]; };

template <int NS> struct PsSlot;
template <> struct PsSlot<4> { using T = uint4; };
template <> struct PsSlot<2> { using T = uint2; };

__device__ __forceinline__ uint32_t ps_spread16(uint32_t x)   // bit i -> bit 2i
{
    x &= 0xFFFFu;
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}

__device__ __forceinline__ uint32_t ps_low_bits(uint32_t n) { return n >= 32u ? 0xFFFFFFFFu : (1u << n) - 1u; }

// the bit planes of the characters that exist in column gcol
template <int NS> __device__ __forceinline__ uint32_t ps_valid(const ParsimonyArgs &a, uint64_t gcol)
{
    if (gcol >= a.n_cols) return 0u;
    const uint64_t left = a.n_chars - gcol * 32;
    const uint32_t n = left < 32 ? (uint32_t)left : 32u;
    if (NS == 2) return ps_low_bits(n);
    return ps_spread16(ps_low_bits(min(n, 16u))) | (ps_spread16(ps_low_bits(n > 16u ? n - 16u : 0u)) << 1);
}

// the character of bit b of column gcol
template <int NS> __device__ __forceinline__ uint64_t ps_char(uint64_t gcol, uint32_t b)
{
    return gcol * 32 + (NS == 2 ? b : (b & 1u) * 16u + (b >> 1));
}

// a leaf's one-hot planes; padding characters take state 0
template <int NS> __device__ __forceinline__ PsSet<NS> ps_leaf(const ParsimonyArgs &a, uint32_t leaf, uint64_t gcol, uint32_t valid)
{
    PsSet<NS> s;
    if (NS == 4) {
        const uint2 w = __ldg(reinterpret_cast<const uint2 *>(a.rows + (uint64_t)leaf * a.row_words) + gcol);
        const uint32_t b0 = (w.x & 0x55555555u) | ((w.y & 0x55555555u) << 1);
        const uint32_t b1 = ((w.x >> 1) & 0x55555555u) | (w.y & 0xAAAAAAAAu);
        s.p[0] = (~b0 & ~b1) | ~valid;
        s.p[1] = b0 & ~b1 & valid;
        s.p[NS > 2 ? 2 : 0] = ~b0 & b1 & valid;
        s.p[NS > 3 ? 3 : 0] = b0 & b1 & valid;
    } else {
        const uint32_t w = __ldg(a.rows + (uint64_t)leaf * a.row_words + gcol) & valid;
        s.p[0] = ~w;
        s.p[1] = w;
    }
    return s;
}

template <int NS> __device__ __forceinline__ PsSet<NS> ps_load_slot(const ParsimonyArgs &a, uint32_t v, uint32_t lcol)
{
    const typename PsSlot<NS>::T x = reinterpret_cast<const typename PsSlot<NS>::T *>(a.scratch)[(uint64_t)v * a.cols_pad + lcol];
    PsSet<NS> s;
    s.p[0] = x.x;
    s.p[1] = x.y;
    if constexpr (NS == 4) { s.p[2] = x.z; s.p[3] = x.w; }
    return s;
}

template <int NS> __device__ __forceinline__ void ps_store_slot(const ParsimonyArgs &a, uint32_t v, uint32_t lcol, const PsSet<NS> &s)
{
    typename PsSlot<NS>::T x;
    x.x = s.p[0];
    x.y = s.p[1];
    if constexpr (NS == 4) { x.z = s.p[2]; x.w = s.p[3]; }
    reinterpret_cast<typename PsSlot<NS>::T *>(a.scratch)[(uint64_t)v * a.cols_pad + lcol] = x;
}

template <int NS> __device__ __forceinline__ PsSet<NS> ps_child(const ParsimonyArgs &a, uint32_t u, uint64_t gcol_ld, uint32_t lcol, uint32_t valid)
{
    return u < a.n_leaves ? ps_leaf<NS>(a, u, gcol_ld, valid) : ps_load_slot<NS>(a, u - a.n_leaves, lcol);
}

// the smallest state of every character's set
template <int NS> __device__ __forceinline__ PsSet<NS> ps_lowest(const PsSet<NS> &s)
{
    PsSet<NS> r;
    uint32_t seen = 0;
#pragma unroll
    for (int x = 0; x < NS; x++) { r.p[x] = s.p[x] & ~seen; seen |= s.p[x]; }
    return r;
}

// score += x (one bit per character)
__device__ __forceinline__ void ps_inc(uint32_t (&sc)[32], uint32_t x)
{
#pragma unroll
    for (int p = 0; p < 32; p++) {
        if (!x) break;
        const uint32_t t = sc[p] & x;
        sc[p] ^= x;
        x = t;
    }
}

template <int NS>
__global__ void __launch_bounds__(PS_THREADS) parsimony_kernel(ParsimonyArgs a)
{
    constexpr int NB = NS == 4 ? 1 : 2;          // branch counters: changes / gains, losses
    __shared__ uint32_t s_br[NB][PS_SLOTS];
    extern __shared__ uint32_t s_cnt[];          // [NS][dmax][PS_THREADS] polytomy counters
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t lcol = blockIdx.x * PS_THREADS + tid;
    const uint64_t gcol = a.col0 + lcol;
    const uint64_t gcol_ld = gcol < a.n_cols ? gcol : a.n_cols - 1;     // rows are read in range; padding columns are masked
    const uint32_t valid = ps_valid<NS>(a, gcol);
    for (uint32_t i = tid; i < NB * PS_SLOTS; i += PS_THREADS) (&s_br[0][0])[i] = 0;
    __syncthreads();
    auto cnt = [&](int x, uint32_t p) -> uint32_t & { return s_cnt[((uint32_t)x * a.dmax + p) * PS_THREADS + tid]; };

    uint32_t sc[32];
#pragma unroll
    for (int p = 0; p < 32; p++) sc[p] = 0;

    // ---- bottom-up: sets and scores
    for (uint32_t v = 0; v < a.n_internal; v++) {
        const uint32_t o0 = __ldg(a.child_off + v), o1 = __ldg(a.child_off + v + 1), k = o1 - o0;
        PsSet<NS> s;
        if (k == 2) {
            const PsSet<NS> A = ps_child<NS>(a, __ldg(a.child + o0), gcol_ld, lcol, valid);
            const PsSet<NS> B = ps_child<NS>(a, __ldg(a.child + o0 + 1), gcol_ld, lcol, valid);
            uint32_t any = 0;
#pragma unroll
            for (int x = 0; x < NS; x++) any |= A.p[x] & B.p[x];
            const uint32_t empty = ~any;
#pragma unroll
            for (int x = 0; x < NS; x++) s.p[x] = (A.p[x] & B.p[x]) | (empty & (A.p[x] | B.p[x]));
            ps_inc(sc, empty);
        } else {
            const uint32_t D = 32u - __clz(k);       // planes that hold k
            for (uint32_t p = 0; p < D; p++)
#pragma unroll
                for (int x = 0; x < NS; x++) cnt(x, p) = 0;
            for (uint32_t j = o0; j < o1; j++) {
                const PsSet<NS> C = ps_child<NS>(a, __ldg(a.child + j), gcol_ld, lcol, valid);
#pragma unroll
                for (int x = 0; x < NS; x++) {
                    uint32_t carry = C.p[x];
                    for (uint32_t p = 0; p < D && carry; p++) {
                        const uint32_t c = cnt(x, p);
                        cnt(x, p) = c ^ carry;
                        carry &= c;
                    }
                }
            }
            // bit-sliced maximum from the top plane down; the states still at the maximum form the set. The maximum's
            // plane p replaces state 0's counter plane p, which is not read again.
            uint32_t cand[NS];
#pragma unroll
            for (int x = 0; x < NS; x++) cand[x] = 0xFFFFFFFFu;
            for (int p = (int)D - 1; p >= 0; p--) {
                uint32_t bit[NS], any = 0;
#pragma unroll
                for (int x = 0; x < NS; x++) { bit[x] = cnt(x, (uint32_t)p); any |= cand[x] & bit[x]; }
#pragma unroll
                for (int x = 0; x < NS; x++) cand[x] &= bit[x] | ~any;
                cnt(0, (uint32_t)p) = any;
            }
#pragma unroll
            for (int x = 0; x < NS; x++) s.p[x] = cand[x];
            // score += k - m: the difference formed plane by plane (borrow) and added in the same pass (carry)
            uint32_t borrow = 0, carry = 0;
#pragma unroll
            for (int p = 0; p < 32; p++) {
                uint32_t d = 0;
                if ((uint32_t)p < D) {
                    const uint32_t m = cnt(0, (uint32_t)p), kb = ((k >> p) & 1u) ? 0xFFFFFFFFu : 0u;
                    d = kb ^ m ^ borrow;
                    borrow = (~kb & (m | borrow)) | (kb & m & borrow);
                } else if (!carry) {
                    break;
                }
                const uint32_t t = sc[p];
                sc[p] = t ^ d ^ carry;
                carry = (t & d) | (carry & (t ^ d));
            }
        }
        ps_store_slot<NS>(a, v, lcol, s);
    }

    // ---- top-down: one optimal assignment, changes per branch
    if (a.n_internal) {
        const uint32_t root = a.n_internal - 1;
        ps_store_slot<NS>(a, root, lcol, ps_lowest<NS>(ps_load_slot<NS>(a, root, lcol)));
        uint32_t chunk = 0xFFFFFFFFu;                // CSR positions chunk * PS_SLOTS .. held in s_br
        auto flush = [&]() {
            __syncthreads();
            for (uint32_t i = tid; i < PS_SLOTS; i += PS_THREADS) {
#pragma unroll
                for (int b = 0; b < NB; b++) {
                    const uint32_t n = s_br[b][i];
                    if (n) {
                        const uint32_t node = __ldg(a.child + (size_t)chunk * PS_SLOTS + i);
                        atomicAdd((b ? a.branch1 : a.branch0) + node, (unsigned long long)n);
                        s_br[b][i] = 0;
                    }
                }
            }
            __syncthreads();
        };
        for (int v = (int)root; v >= 0; v--) {
            const PsSet<NS> A = ps_load_slot<NS>(a, (uint32_t)v, lcol);
            const uint32_t o0 = __ldg(a.child_off + v), o1 = __ldg(a.child_off + v + 1);
            for (uint32_t j = o0; j < o1; j++) {
                if (j / PS_SLOTS != chunk) {
                    if (chunk != 0xFFFFFFFFu) flush();
                    chunk = j / PS_SLOTS;
                }
                const uint32_t u = __ldg(a.child + j);
                PsSet<NS> U;                             // the child's assigned state
                uint32_t same = 0;
                if (u < a.n_leaves) {
                    U = ps_leaf<NS>(a, u, gcol_ld, valid);
#pragma unroll
                    for (int x = 0; x < NS; x++) same |= U.p[x] & A.p[x];
                } else {
                    const PsSet<NS> S = ps_load_slot<NS>(a, u - a.n_leaves, lcol);
#pragma unroll
                    for (int x = 0; x < NS; x++) same |= S.p[x] & A.p[x];
                    const PsSet<NS> L = ps_lowest<NS>(S);
#pragma unroll
                    for (int x = 0; x < NS; x++) U.p[x] = (A.p[x] & same) | (L.p[x] & ~same);
                    ps_store_slot<NS>(a, u - a.n_leaves, lcol, U);
                }
                const uint32_t change = ~same & valid;
                const uint32_t slot = j % PS_SLOTS;
                if (NB == 1) {
                    const uint32_t n = __reduce_add_sync(0xFFFFFFFFu, __popc(change));
                    if (lane == 0 && n) atomicAdd(&s_br[0][slot], n);
                } else {
                    const uint32_t g = __popc(change & U.p[1]), l = __popc(change & U.p[0]);
                    const uint32_t n = __reduce_add_sync(0xFFFFFFFFu, g | (l << 16));   // at most 32 x 32 each
                    if (lane == 0 && n) {
                        if (n & 0xFFFFu) atomicAdd(&s_br[0][slot], n & 0xFFFFu);
                        if (n >> 16) atomicAdd(&s_br[NB - 1][slot], n >> 16);
                    }
                }
            }
        }
        flush();
    }

    // ---- per-character scores and the summary terms
    unsigned long long t[5] = {0, 0, 0, 0, 0};      // variable, tree length, min changes, max changes, homoplastic
    if (valid) {
        const uint32_t N = a.n_leaves;
        for (uint32_t b = 0; b < 32; b++) {
            if (!((valid >> b) & 1u)) continue;
            uint32_t s = 0;
#pragma unroll
            for (int p = 0; p < 32; p++) s |= ((sc[p] >> b) & 1u) << p;
            const uint64_t ch = ps_char<NS>(gcol, b);
            a.scores[ch] = s;
            uint32_t distinct, top;
            if (NS == 4) {
                const uint4 n = __ldg(a.site_counts + ch);
                distinct = (n.x > 0) + (n.y > 0) + (n.z > 0) + (n.w > 0);
                top = max(max(n.x, n.y), max(n.z, n.w));
            } else {
                const uint32_t n = __ldg(a.gene_counts + ch);
                distinct = (n > 0) + (n < N);
                top = max(n, N - n);
            }
            t[0] += distinct >= 2;
            t[1] += s;
            t[2] += distinct - 1;
            t[3] += N - top;
            t[4] += s > distinct - 1;
        }
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t[k] += __shfl_xor_sync(0xFFFFFFFFu, t[k], o);
        if (lane == 0 && t[k]) atomicAdd(a.summary + k, t[k]);
    }
}

}  // namespace pansim
