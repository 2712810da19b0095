// nj.cuh -- neighbour-joining on a dense distance matrix on the device (DESIGN.md section 18; the definitions are in
// include/pansim_b200.h): Saitou & Nei with Studier & Keppler's Q, every operation IEEE binary64 round-to-nearest in
// the order the header writes it (explicit __d*_rn, so nothing is contracted to an FMA).
//
// State on the device: the symmetric matrix D (stored dimension M, row pitch `pitch` doubles), R[M] and node[M]. The
// stored rows are the slots in list order: slot a takes the new node, slot b dies, so stored order stays slot order
// and the tie rule "smaller a, then smaller b" is "smaller stored row, then smaller stored column". A dead row has
// R = NaN: every Q that touches it is NaN, which compares false, so the scan needs no alive flags, and the join's
// closed-form R update keeps it NaN. k (the active count) is known to the host at every iteration (it falls by one),
// so it is a launch argument; nothing returns to the host until the tree is done.
//
// Per iteration: nj_scan_kernel (a warp per stored row, lanes along the row's upper triangle; per-CTA minimum of
// (Q, a, b); the last CTA to finish reduces the CTA minima) and nj_join_kernel (a thread per stored column: row and
// column u, R, and one thread for the branch lengths and the slot list). nj_compact_* repack the active rows and
// columns into a dense prefix when k falls below a fraction of M.
#pragma once
#include "common.cuh"

namespace pansim {

constexpr uint32_t NJ_THREADS = 256;
constexpr uint32_t NJ_NONE = 0xFFFFFFFFu;

struct NjBest {
    double q;
    uint32_t a, b;
};

// lexicographic (Q, a, b); a NaN Q is never less
__device__ __forceinline__ bool nj_less(double q, uint32_t a, uint32_t b, double oq, uint32_t oa, uint32_t ob)
{
    return q < oq || (q == oq && (a < oa || (a == oa && b < ob)));
}

// core: d = core_diff / core_size; acc: d = 1 - (inter + core_genes) / (uni + core_genes), 0 where the denominator is 0.
// Pair p of the block is (r1[p], r2[p]); both (i, j) and (j, i) are written.
__global__ void nj_scatter_pairs_kernel(const uint32_t *__restrict__ r1, const uint32_t *__restrict__ r2,
                                        const uint32_t *__restrict__ cd, const uint32_t *__restrict__ in,
                                        const uint32_t *__restrict__ un, uint32_t P, int acc, double core_size,
                                        double core_genes, double *__restrict__ D, uint64_t pitch)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
        double d;
        if (!acc) {
            d = __ddiv_rn((double)cd[p], core_size);
        } else {
            const double den = __dadd_rn((double)un[p], core_genes);
            d = den == 0.0 ? 0.0 : __dsub_rn(1.0, __ddiv_rn(__dadd_rn((double)in[p], core_genes), den));
        }
        const uint64_t i = r1[p], j = r2[p];
        D[i * pitch + j] = d;
        D[j * pitch + i] = d;
    }
}

// a caller's upper triangle, row-major (row i holds d(i, i+1 .. n-1)), into both halves; the diagonal is 0
__global__ void nj_scatter_upper_kernel(const double *__restrict__ upper, uint32_t n, double *__restrict__ D, uint64_t pitch)
{
    for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
        const uint64_t off = (uint64_t)i * (2ull * n - i - 1) / 2;
        if (threadIdx.x == 0) D[(uint64_t)i * pitch + i] = 0.0;
        for (uint32_t j = i + 1 + threadIdx.x; j < n; j += blockDim.x) {
            const double d = upper[off + (j - i - 1)];
            D[(uint64_t)i * pitch + j] = d;
            D[(uint64_t)j * pitch + i] = d;
        }
    }
}

// R_a = sum_b d_ab left to right over ascending b (the diagonal is 0). Thread a walks column a, which equals row a:
// the threads of a warp read consecutive doubles of row b.
__global__ void nj_rowsum_kernel(const double *__restrict__ D, uint64_t pitch, uint32_t n, double *__restrict__ R,
                                 uint32_t *__restrict__ node)
{
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n) return;
    double s = 0.0;
    for (uint32_t b = 0; b < n; b++) s = __dadd_rn(s, D[(uint64_t)b * pitch + a]);
    R[a] = s;
    node[a] = a;
}

__device__ __forceinline__ void nj_warp_min(double &q, uint32_t &a, uint32_t &b)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double q2 = __shfl_xor_sync(0xFFFFFFFFu, q, o);
        const uint32_t a2 = __shfl_xor_sync(0xFFFFFFFFu, a, o), b2 = __shfl_xor_sync(0xFFFFFFFFu, b, o);
        if (nj_less(q2, a2, b2, q, a, b)) { q = q2; a = a2; b = b2; }
    }
}

// CTA minimum into s (thread 0 holds it on return)
__device__ __forceinline__ void nj_cta_min(double &q, uint32_t &a, uint32_t &b, NjBest *s)
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    nj_warp_min(q, a, b);
    if (lane == 0) s[warp] = {q, a, b};
    __syncthreads();
    if (warp == 0) {
        if (lane < NJ_THREADS / 32) { q = s[lane].q; a = s[lane].a; b = s[lane].b; }
        else { q = __longlong_as_double(0x7FF0000000000000ll); a = b = NJ_NONE; }
        nj_warp_min(q, a, b);
    }
}

// The lexicographic minimum of (Q_ab, a, b) over active stored rows a < b, Q_ab = ((k - 2) d_ab - R_a) - R_b. Warp w
// takes rows w, w + warps, ...; each CTA writes its minimum to part[], and the last CTA to finish reduces part[] into
// *best and re-arms *done.
__global__ void __launch_bounds__(NJ_THREADS) nj_scan_kernel(const double *__restrict__ D, uint64_t pitch, uint32_t M,
                                                             double k2, const double *__restrict__ R, NjBest *part,
                                                             uint32_t *done, NjBest *best)
{
    __shared__ NjBest s[NJ_THREADS / 32];
    __shared__ bool last;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (NJ_THREADS / 32);
    double q = __longlong_as_double(0x7FF0000000000000ll);
    uint32_t ba = NJ_NONE, bb = NJ_NONE;
    for (uint32_t i = blockIdx.x * (NJ_THREADS / 32) + (threadIdx.x >> 5); i + 1 < M; i += warps) {
        const double ri = R[i];
        if (ri != ri) continue;                              // dead row (warp-uniform)
        const double *row = D + (uint64_t)i * pitch;
        for (uint32_t j0 = i + 1 + lane; j0 < M; j0 += 128) {
            double d[4], r[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t j = j0 + 32 * u;
                d[u] = j < M ? row[j] : 0.0;
                r[u] = j < M ? __ldg(R + j) : __longlong_as_double(0x7FF8000000000000ll);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const double qq = __dsub_rn(__dsub_rn(__dmul_rn(k2, d[u]), ri), r[u]);
                if (nj_less(qq, i, j0 + 32 * u, q, ba, bb)) { q = qq; ba = i; bb = j0 + 32 * u; }
            }
        }
    }
    nj_cta_min(q, ba, bb, s);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = {q, ba, bb};
        __threadfence();
        last = atomicAdd(done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    q = __longlong_as_double(0x7FF0000000000000ll);
    ba = bb = NJ_NONE;
    for (uint32_t g = threadIdx.x; g < gridDim.x; g += NJ_THREADS) {
        const double q2 = __ldcg(&part[g].q);
        const uint32_t a2 = __ldcg(&part[g].a), b2 = __ldcg(&part[g].b);
        if (nj_less(q2, a2, b2, q, ba, bb)) { q = q2; ba = a2; bb = b2; }
    }
    __syncthreads();                                         // s[] is reused
    nj_cta_min(q, ba, bb, s);
    if (threadIdx.x == 0) {
        *best = {q, ba, bb};
        *done = 0;
    }
}

// Join t = N - k of slots (a, b) = *best into node N + t at slot a. Every other stored column c: d_uc = ((d_ac + d_bc) -
// d_ab) / 2 into row and column a, R_c = ((R_c - d_ac) - d_bc) + d_uc (a dead c stays NaN). Thread 0: the branch
// lengths of the two children, R_u, the slot list (node[a] = u, R_b = NaN). No thread writes d_ab, R_a or R_b but
// thread 0.
__global__ void __launch_bounds__(NJ_THREADS) nj_join_kernel(double *__restrict__ D, uint64_t pitch, uint32_t M,
                                                             double *__restrict__ R, uint32_t *__restrict__ node,
                                                             const NjBest *__restrict__ best, uint32_t k, uint32_t N,
                                                             uint32_t *__restrict__ parent, double *__restrict__ length)
{
    const uint32_t a = best->a, b = best->b;
    const double dab = D[(uint64_t)a * pitch + b];
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0) {
        const double k2 = (double)(k - 2), ra = R[a], rb = R[b];
        const double da = __dmul_rn(__dadd_rn(dab, __ddiv_rn(__dsub_rn(ra, rb), k2)), 0.5);
        const double db = __dsub_rn(dab, da);
        const uint32_t u = N + (N - k), na = node[a], nb = node[b];
        parent[na] = u; length[na] = da;
        parent[nb] = u; length[nb] = db;
        R[a] = __dmul_rn(__dsub_rn(__dadd_rn(__dsub_rn(ra, dab), __dsub_rn(rb, dab)), __dmul_rn(k2, dab)), 0.5);
        R[b] = __longlong_as_double(0x7FF8000000000000ll);
        node[a] = u;
        node[b] = NJ_NONE;
    }
    if (c >= M || c == a || c == b) return;
    const double dac = D[(uint64_t)a * pitch + c], dbc = D[(uint64_t)b * pitch + c];
    const double duc = __dmul_rn(__dsub_rn(__dadd_rn(dac, dbc), dab), 0.5);
    D[(uint64_t)a * pitch + c] = duc;
    D[(uint64_t)c * pitch + a] = duc;
    R[c] = __dadd_rn(__dsub_rn(__dsub_rn(R[c], dac), dbc), duc);
}

// Compaction, step 1 (one CTA): old_of[i'] = the i'-th active stored row in order, with its R and node moved along.
__global__ void __launch_bounds__(1024) nj_compact_index_kernel(const double *__restrict__ R, const uint32_t *__restrict__ node,
                                                                uint32_t M, uint32_t *__restrict__ old_of,
                                                                double *__restrict__ R_new, uint32_t *__restrict__ node_new)
{
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t i0 = 0; i0 < M; i0 += blockDim.x) {
        const uint32_t i = i0 + threadIdx.x;
        const bool alive = i < M && R[i] == R[i];
        const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, alive);
        if (lane == 0) warp_sum[warp] = __popc(ballot);
        __syncthreads();
        uint32_t off = base;
        for (uint32_t w = 0; w < warp; w++) off += warp_sum[w];
        off += __popc(ballot & ((1u << lane) - 1u));
        if (alive) { old_of[off] = i; R_new[off] = R[i]; node_new[off] = node[i]; }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) base = off + (alive ? 1u : 0u);
        __syncthreads();
    }
}

// Compaction, step 2: dst[i'][j'] = src[old_of[i']][old_of[j']] over the k x k active block.
__global__ void nj_compact_copy_kernel(const double *__restrict__ src, uint64_t src_pitch, double *__restrict__ dst,
                                       uint64_t dst_pitch, const uint32_t *__restrict__ old_of, uint32_t k)
{
    for (uint32_t i = blockIdx.x; i < k; i += gridDim.x) {
        const double *s = src + (uint64_t)old_of[i] * src_pitch;
        double *d = dst + (uint64_t)i * dst_pitch;
        for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) d[j] = s[old_of[j]];
    }
}

// The last two or three active slots (one thread). Three, x < y < z: the root 2N - 3 with lengths
// ((d_xy + d_xz) - d_yz) / 2 and likewise; two (N = 2): the root 2, each branch d / 2.
__global__ void nj_finish_kernel(const double *__restrict__ D, uint64_t pitch, uint32_t M, const double *__restrict__ R,
                                 const uint32_t *__restrict__ node, uint32_t N, uint32_t *__restrict__ parent,
                                 double *__restrict__ length)
{
    uint32_t s[3], n = 0;
    for (uint32_t i = 0; i < M && n < 3; i++)
        if (R[i] == R[i]) s[n++] = i;
    auto d = [&](int x, int y) { return D[(uint64_t)s[x] * pitch + s[y]]; };
    uint32_t root;
    if (n == 2) {
        root = 2;
        const double h = __dmul_rn(d(0, 1), 0.5);
        for (int x = 0; x < 2; x++) { parent[node[s[x]]] = root; length[node[s[x]]] = h; }
    } else {
        root = 2 * N - 3;
        const double xy = d(0, 1), xz = d(0, 2), yz = d(1, 2);
        const double l[3] = {__dmul_rn(__dsub_rn(__dadd_rn(xy, xz), yz), 0.5), __dmul_rn(__dsub_rn(__dadd_rn(xy, yz), xz), 0.5),
                             __dmul_rn(__dsub_rn(__dadd_rn(xz, yz), xy), 0.5)};
        for (int x = 0; x < 3; x++) { parent[node[s[x]]] = root; length[node[s[x]]] = l[x]; }
    }
    parent[root] = NJ_NONE;
    length[root] = 0.0;
}

}  // namespace pansim
