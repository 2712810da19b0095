// genealogy.cuh -- the clonal genealogy of the present population, traced on the device from the recorded parent
// vectors (DESIGN.md section 13; the definitions are in include/pansim_b200.h).
//
// Record: a ring of `cap` parent vectors H (u32[N], child -> parent in the previous generation), one device-to-device
// copy per generation on the context's recording stream; the host knows the slot when it enqueues the copy.
//
// Trace (genealogy_trace_kernel, one CTA of 1024 threads): live lineages (node id, current ancestor) sit in two
// global buffers, in ascending order of the smallest leaf below them. Generation t = T .. 1: every lineage reads its
// parent p = H_t[ancestor] and takes atomicMin(owner[p], slot) and atomicAdd(cnt[p], 1). The lineage holding the
// minimum slot of a group represents it; it also holds the group's smallest leaf, since the slots are in that order.
// In rounds of 1024 slots, one block scan of (representative, representative of a group of >= 2) gives every new
// node its id (N, N + 1, ... in slot order) and every survivor its slot in the other buffer, so the order is kept
// without a sort. The members of a merged group read the new id from newid[p] after a barrier (the representative
// sits in the same or an earlier round). Then every lineage clears owner[p] and cnt[p]. The walk ends when one
// lineage is left (the MRCA) or after H_1; with more than one lineage left a virtual root is added.
//
// Node ids are in ascending time order (leaves 0 .. N-1 at time 0, internal nodes numbered backwards in time), so
// every parent id is larger than its child's. genealogy_tmrca_kernel walks up from both leaves of a pair, always
// moving the endpoint with the smaller id (the smaller time, ties broken by id), until they meet.
#pragma once
#include "common.cuh"

namespace pansim {

constexpr uint32_t GT_THREADS = 1024;
constexpr uint32_t GEN_NONE = 0xFFFFFFFFu;

struct GenealogyTrace {
    const uint32_t *ring;       // [cap][N]
    uint32_t cap, N, T, base;   // H_k lives in ring slot (base + k - 1) % cap
    uint32_t *owner, *cnt, *newid;              // [N] each: owner = GEN_NONE, cnt = 0 between generations
    uint32_t *lin_node[2], *lin_anc[2];         // [N] each: live lineages, double-buffered
    uint32_t *parent, *individual, *time;       // [2N] node table
    uint32_t *out;                              // [2]: n_nodes, lineages_at_start
};

// inclusive block scan of x over the 1024 threads; *total = the sum over the block. Ends with a barrier, so the
// caller may not reuse s_warp before its next barrier.
__device__ __forceinline__ uint32_t gt_block_scan(uint32_t x, uint32_t *s_warp, uint32_t *total)
{
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
    for (uint32_t o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31u) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t v = s_warp[lane];
#pragma unroll
        for (uint32_t o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += y;
        }
        s_warp[lane] = v;
    }
    __syncthreads();
    *total = s_warp[31];
    return x + (warp ? s_warp[warp - 1] : 0u);
}

__global__ void __launch_bounds__(GT_THREADS, 1) genealogy_trace_kernel(GenealogyTrace a)
{
    __shared__ uint32_t s_warp[32];
    const uint32_t tid = threadIdx.x, N = a.N;
    for (uint32_t i = tid; i < N; i += GT_THREADS) {
        a.owner[i] = GEN_NONE;
        a.cnt[i] = 0;
        a.parent[i] = GEN_NONE;
        a.individual[i] = i;
        a.time[i] = 0;
        a.lin_node[0][i] = i;
        a.lin_anc[0][i] = i;
    }
    __syncthreads();
    uint32_t m = N, next_id = N, cur = 0;
    for (uint32_t t = a.T; t >= 1 && m > 1; t--) {
        const uint32_t *H = a.ring + (size_t)(((uint64_t)a.base + t - 1) % a.cap) * N;
        // selected, not indexed: a dynamic index into the parameter struct would put it on the stack
        const uint32_t *node = cur ? a.lin_node[1] : a.lin_node[0], *anc = cur ? a.lin_anc[1] : a.lin_anc[0];
        uint32_t *onode = cur ? a.lin_node[0] : a.lin_node[1], *oanc = cur ? a.lin_anc[0] : a.lin_anc[1];
        for (uint32_t s = tid; s < m; s += GT_THREADS) {
            const uint32_t p = H[anc[s]];
            atomicMin(&a.owner[p], s);
            atomicAdd(&a.cnt[p], 1u);
        }
        __syncthreads();
        const uint32_t tnode = a.T - t + 1;     // generation t - 1
        uint32_t n_surv = 0;
        for (uint32_t s0 = 0; s0 < m; s0 += GT_THREADS) {
            const uint32_t s = s0 + tid;
            uint32_t p = 0, k = 0, flags = 0;   // bit 0: representative; bit 16: representative of a merge
            if (s < m) {
                p = H[anc[s]];
                k = a.cnt[p];
                if (a.owner[p] == s) flags = 1u | (k >= 2u ? 1u << 16 : 0u);
            }
            uint32_t tot;
            const uint32_t excl = gt_block_scan(flags, s_warp, &tot) - flags;
            if (flags) {
                uint32_t nd = node[s];
                if (flags >> 16) {
                    const uint32_t id = next_id + (excl >> 16);
                    a.individual[id] = p;
                    a.time[id] = tnode;
                    a.parent[id] = GEN_NONE;
                    a.newid[p] = id;
                    nd = id;
                }
                onode[n_surv + (excl & 0xFFFFu)] = nd;
                oanc[n_surv + (excl & 0xFFFFu)] = p;
            }
            __syncthreads();
            if (k >= 2u) a.parent[node[s]] = a.newid[p];
            n_surv += tot & 0xFFFFu;
            next_id += tot >> 16;
        }
        __syncthreads();
        for (uint32_t s = tid; s < m; s += GT_THREADS) {
            const uint32_t p = H[anc[s]];
            a.owner[p] = GEN_NONE;
            a.cnt[p] = 0;
        }
        __syncthreads();
        m = n_surv;
        cur ^= 1;
    }
    if (m > 1) {                                // not coalesced within the record: the virtual root
        const uint32_t *node = cur ? a.lin_node[1] : a.lin_node[0];
        for (uint32_t s = tid; s < m; s += GT_THREADS) a.parent[node[s]] = next_id;
        if (tid == 0) {
            a.parent[next_id] = GEN_NONE;
            a.individual[next_id] = GEN_NONE;
            a.time[next_id] = a.T;
            a.out[0] = next_id + 1;
            a.out[1] = m;
        }
    } else if (tid == 0) {
        a.out[0] = next_id;
        a.out[1] = 1;
    }
}

// TMRCA of pair k: the time of the node where the walks up from r1[k] and r2[k] meet
__global__ void genealogy_tmrca_kernel(const uint32_t *__restrict__ parent, const uint32_t *__restrict__ time,
                                       const uint32_t *__restrict__ r1, const uint32_t *__restrict__ r2, size_t P,
                                       uint32_t *__restrict__ out)
{
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < P; k += (size_t)gridDim.x * blockDim.x) {
        uint32_t u = r1[k], v = r2[k];
        while (u != v) {
            if (u < v) u = __ldg(parent + u);
            else v = __ldg(parent + v);
        }
        out[k] = __ldg(time + u);
    }
}

}  // namespace pansim
