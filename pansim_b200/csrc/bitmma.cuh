// bitmma.cuh -- the tcgen05 product of two 128-row tiles of a bit matrix, C[i][j] = popc(row_i & row_j), shared by the
// competition term (acc_inter_umma_bits_kernel, select.cuh), core LD (ld_pair_kernel, ld.cuh) and gene LD
// (gene_ld_pair_kernel, gene_ld.cuh).
//
// A CTA of UB_THREADS threads: eight warps read the BIT rows of both tiles and expand them to 0/1 bytes straight into
// the swizzled K-major operand layout the tensor core expects, make the writes visible to the async proxy
// (fence.proxy.async) and hand the stage to the MMA warp through an mbarrier; tcgen05.commit returns it. Thread = one
// row of the stage (128 rows of the i tile, 128 of the j tile), KB / 8 bytes of bits per row per stage, fetched one
// stage ahead. One thread of the MMA warp issues tcgen05.mma.kind::i8 (u8 x u8 -> s32, M = N = 128, K = 32 per
// instruction) into a 128 x 128 accumulator in tensor memory (128 lanes x 128 columns), exact: the products are 0/1 and
// the s32 accumulation cannot overflow. The 32 genes of a word go to 32 consecutive bytes, byte 4t + q = bit t + 8q: a
// fixed permutation of the k index, which a dot product does not see.
//   KB = 128: 16-byte fetch, rows of 128 bytes, 16-byte chunk c of row r stored at chunk c ^ (r % 8) (SWIZZLE_128B, what
//             a TMA load would have produced; 8-row groups 1024 bytes apart), four stages of 32 KiB.
//   KB = 64:  8-byte fetch, rows of 64 bytes, chunk c of row r at c ^ ((r / 2) % 4) (SWIZZLE_64B; 8-row groups 512 bytes
//             apart), three stages of 16 KiB: 48 KiB of shared memory, so several CTAs share an SM and one's epilogue
//             overlaps another's MMAs.
// A kernel calls bitmma_smem, then bitmma_init (one thread) and bitmma_alloc (the MMA warp), bitmma_tmem (every
// thread), bitmma_mainloop (every thread), its epilogue (bitmma_wait, bitmma_load16 in the eight expansion warps) and
// bitmma_free (every thread).
#pragma once
#include <type_traits>

#include "common.cuh"

namespace pansim {

constexpr int UM_TILE = 128;                 // rows per operand tile = UMMA M = UMMA N
constexpr uint32_t UM_TMEM_COLS = 128;
// instruction descriptor (kind::i8): D = s32 (bits 4-5 = 2), A = B = u8 (0), both K-major (0), N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t UM_IDESC = (2u << 4) | ((uint32_t)(UM_TILE >> 3) << 17) | ((uint32_t)(UM_TILE >> 4) << 24);

constexpr int UB_EXP_WARPS = 8;
constexpr int UB_THREADS = 32 * (UB_EXP_WARPS + 1);       // + the MMA warp

template <int KB> struct UbCfg {
    static_assert(KB == 128 || KB == 64, "128- or 64-byte swizzled operand rows");
    static constexpr uint32_t STAGES = KB == 128 ? 4u : 3u;
    static constexpr uint32_t TILE_BYTES = UM_TILE * KB;
    // matrix descriptor, high word: stride between 8-row groups (8 * KB bytes, in 16 B), version 1, layout 2 = SWIZZLE_128B / 4 = SWIZZLE_64B
    static constexpr uint32_t DESC_HI = ((8u * KB) >> 4) | (1u << 14) | ((KB == 128 ? 2u : 4u) << 29);
    using Row = std::conditional_t<KB == 128, uint4, uint2>;      // one row's bits of a stage
    static constexpr size_t smem_bytes() { return 1024 + 2 * (size_t)STAGES * TILE_BYTES + (2 * STAGES + 1) * sizeof(uint64_t) + 16; }
};

// mbarrier wait that traps instead of spinning forever (a wrong descriptor would otherwise hang the device)
__device__ __forceinline__ void mbar_wait_or_trap(uint32_t bar_s, uint32_t parity)
{
    for (uint32_t spin = 0; spin < (1u << 24); spin++) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar_s), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}

__device__ __forceinline__ uint32_t row_word(const uint2 &v, uint32_t q) { return q ? v.y : v.x; }
__device__ __forceinline__ uint32_t row_word(const uint4 &v, uint32_t q) { return q == 0 ? v.x : q == 1 ? v.y : q == 2 ? v.z : v.w; }

// Shared-memory addresses of the operand stages, the barriers and the tensor-memory slot in the dynamic shared memory
// (UbCfg<KB>::smem_bytes() of it).
struct BitMma {
    uint32_t a_s, b_s, full_s, empty_s, done_s, slot_s;
};

template <int KB>
__device__ __forceinline__ BitMma bitmma_smem(const uint8_t *smem)
{
    using Cfg = UbCfg<KB>;
    BitMma m;
    const uint32_t base_s = (smem_u32(smem) + 1023u) & ~1023u;      // operand tiles on 1 KiB boundaries (swizzle atom)
    m.a_s = base_s;
    m.b_s = base_s + Cfg::STAGES * Cfg::TILE_BYTES;
    m.full_s = m.b_s + Cfg::STAGES * Cfg::TILE_BYTES;
    m.empty_s = m.full_s + Cfg::STAGES * 8u;
    m.done_s = m.empty_s + Cfg::STAGES * 8u;
    m.slot_s = m.done_s + 8u;
    return m;
}

// one thread: the stage barriers and the accumulator's
template <int KB>
__device__ __forceinline__ void bitmma_init(const BitMma &m)
{
    for (uint32_t s = 0; s < UbCfg<KB>::STAGES; s++) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(m.full_s + s * 8u), "r"((uint32_t)UB_EXP_WARPS) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(m.empty_s + s * 8u), "r"(1u) : "memory");
    }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(m.done_s), "r"(1u) : "memory");
    fence_mbar_init();
}

// the MMA warp: the accumulator's tensor-memory columns
__device__ __forceinline__ void bitmma_alloc(const BitMma &m)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(m.slot_s), "r"(UM_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

// every thread, after bitmma_init and bitmma_alloc: a CTA barrier, then the accumulator's address
__device__ __forceinline__ uint32_t bitmma_tmem(const BitMma &m)
{
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    uint32_t tmem;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(m.slot_s) : "memory");
    return tmem;
}

// Main loop over k_iters stages of KB bits: threads 0..127 expand rows bi * 128 .. + 127 of `rows` (pitch_words words
// apart), threads 128..255 rows bj * 128 .. + 127; rows at or past n_valid are zero. Precondition: every row holds at
// least k_iters * KB / 32 words, so no stage reads past a row. Lane 0 of the MMA warp issues the MMAs and commits to
// done_s once the accumulator is complete.
template <int KB>
__device__ __forceinline__ void bitmma_mainloop(const BitMma &m, uint32_t tmem, const uint32_t *rows, uint32_t pitch_words,
                                                uint32_t n_valid, uint32_t k_iters, uint32_t bi, uint32_t bj, uint32_t warp,
                                                uint32_t lane)
{
    using Cfg = UbCfg<KB>;
    constexpr uint32_t STAGES = Cfg::STAGES, TILE_BYTES = Cfg::TILE_BYTES, WORDS = KB / 32;      // bit words per row per stage
    if (warp < UB_EXP_WARPS) {
        // ---- expansion ----
        const uint32_t tr = threadIdx.x & 127u;                          // row inside the tile
        const bool is_b = threadIdx.x >= 128u;
        const uint32_t grow = (is_b ? bj : bi) * UM_TILE + tr;
        const bool row_ok = grow < n_valid;
        const uint32_t row_s = (is_b ? m.b_s : m.a_s) + tr * KB;
        const uint32_t sw = (KB == 128 ? (tr & 7u) : ((tr >> 1) & 3u)) << 4;             // XOR term of the swizzle
        using Row = typename Cfg::Row;
        const Row *src = reinterpret_cast<const Row *>(rows + (uint64_t)(row_ok ? grow : 0u) * pitch_words);
        const Row zero = {};
        Row nxt = row_ok ? __ldg(src) : zero;
        for (uint32_t it = 0; it < k_iters; it++) {
            const uint32_t s = it % STAGES, n = it / STAGES;
            const Row cur = nxt;
            if (it + 1u < k_iters) nxt = row_ok ? __ldg(src + it + 1u) : zero;
            if (n) mbar_wait_or_trap(m.empty_s + s * 8u, (n - 1u) & 1u);      // the MMAs that read the stage's previous contents have completed
            const uint32_t dst = row_s + s * TILE_BYTES;
#pragma unroll
            for (uint32_t q = 0; q < WORDS; q++) {
                const uint32_t v = row_word(cur, q);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst + (((2u * q) << 4) ^ sw)), "r"(v & 0x01010101u),
                             "r"((v >> 1) & 0x01010101u), "r"((v >> 2) & 0x01010101u), "r"((v >> 3) & 0x01010101u) : "memory");
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst + (((2u * q + 1u) << 4) ^ sw)), "r"((v >> 4) & 0x01010101u),
                             "r"((v >> 5) & 0x01010101u), "r"((v >> 6) & 0x01010101u), "r"((v >> 7) & 0x01010101u) : "memory");
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes -> visible to the tensor core's reads
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(m.full_s + s * 8u) : "memory");
        }
    } else {
        if (lane == 0) {
            // ---- MMA issue ----
            for (uint32_t it = 0; it < k_iters; it++) {
                const uint32_t s = it % STAGES, n = it / STAGES;
                mbar_wait_or_trap(m.full_s + s * 8u, n & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_lo = (((m.a_s + s * TILE_BYTES) & 0x3FFFFu) >> 4) | (1u << 16);
                const uint32_t b_lo = (((m.b_s + s * TILE_BYTES) & 0x3FFFFu) >> 4) | (1u << 16);
#pragma unroll
                for (uint32_t k = 0; k < KB / 32; k++) {                     // K = 32 bytes per instruction: +32 B inside the swizzled row
                    const uint64_t da = ((uint64_t)Cfg::DESC_HI << 32) | (a_lo + 2u * k);
                    const uint64_t db = ((uint64_t)Cfg::DESC_HI << 32) | (b_lo + 2u * k);
                    const uint32_t accumulate = (it | k) ? 1u : 0u;
                    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                                 ::"r"(tmem), "l"(da), "l"(db), "r"(UM_IDESC), "r"(accumulate) : "memory");
                }
                // arrives on the barrier once the MMAs issued so far have read their operands (implies fence::before_thread_sync)
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(m.empty_s + s * 8u) : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(m.done_s) : "memory");
        }
        __syncwarp();
    }
}

// an epilogue warp: wait until the accumulator is complete
__device__ __forceinline__ void bitmma_wait(const BitMma &m)
{
    mbar_wait_or_trap(m.done_s, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// columns c0 .. c0 + 15 of accumulator lanes 32 * quad .. + 31 (the warp's lane = its row)
__device__ __forceinline__ void bitmma_load16(uint32_t tmem, uint32_t quad, uint32_t c0, uint32_t (&v)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(tmem + ((quad * 32u) << 16) + c0) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// every thread: a CTA barrier, then the MMA warp frees the accumulator
__device__ __forceinline__ void bitmma_free(uint32_t tmem, uint32_t warp)
{
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == UB_EXP_WARPS) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(UM_TMEM_COLS) : "memory");
}

}  // namespace pansim
