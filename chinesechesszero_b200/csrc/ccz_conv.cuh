// ccz_conv.cuh -- K9: 3x3 / pad 1 / 256->256 convolution over Xiangqi boards (10x9) as an implicit
// GEMM on the sm_100a tensor cores, with the ResBlock epilogue (folded-BN bias, optional skip add,
// ReLU; reference net.py:33-41) fused in.
//
//   D[m, co] = relu( sum_{tap, ci} X[pixel(m) + tap, ci] * Wt[co, tap, ci] + bias[co] (+ skip[m, co]) )
//
// m runs over the n*90 output pixels (NHWC, channel-contiguous), K = 9 taps x 256 channels = 2304.
//   * A operand (activations): TMA *im2col* loads, 128 pixels x 64 channels per stage, 128-byte swizzle;
//     the TMA unit walks w, h, n in output-pixel order and zero-fills the halo, so an M tile is any
//     128 consecutive pixels and no FLOP is spent on padding.
//   * B operand (weights, [256][9*256] K-major): plain 2-D tiled TMA, same swizzle.
//   * MMA: tcgen05.mma kind::f16 (bf16 in, fp32 accumulate in TMEM), issued by one thread.  CG = 2 pairs
//     two CTAs of a cluster on one 256x256 tile (cta_group::2): each CTA stages its own 128 pixel rows
//     and half of the weight tile, halving weight traffic through shared memory.
//   * Two TMEM accumulator buffers (2 x 256 columns): the epilogue of tile i overlaps the main loop of i+1.
//   * Epilogue: 4 warps, one accumulator row per thread (tcgen05.ld 32x32b), + bias (+ skip, prefetched by
//     TMA into the staging tile while the main loop runs) -> ReLU -> bf16 into the swizzled staging tile
//     -> TMA store.
// Warp roles (256 threads): 0 = A/B TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 3 = skip-tile
// producer, 4..7 = epilogue.
//
// mbarriers (per CTA; "leader" = the even CTA of a pair, the only one that issues MMAs):
//   full[s]   count 1 + tx bytes : both CTAs' TMA loads of stage s complete on the LEADER's barrier, which expects
//                                   the bytes of the whole pair; the MMA issuer waits on it
//   empty[s]  count PAIRS        : tcgen05.commit of the MMAs that read stage s, multicast to every CTA whose producer
//                                   may overwrite it (the pair; the whole cluster when weight stages are shared)
//   tfull[a]  count 1            : tcgen05.commit after the last k-block of a tile, multicast to the pair -> epilogue
//   tempty[a] count 4 * CG       : lane 0 of each epilogue warp of both CTAs, after its tcgen05.ld's -> MMA issuer
//   skip      count 1 + tx bytes : the skip tile has landed in the staging buffer -> epilogue
//   stfree    count 1            : the TMA store of the previous tile has finished READING the staging buffer
//                                   -> skip-tile producer (the epilogue warps themselves re-sync on bar.sync 1)
// Everything is persistent: grid = one CTA per SM, static round-robin over work items, phases tracked per role.
// Under the 1 kW cap the kernel is bound by energy per FLOP, not by issue slots or utilisation (DESIGN.md
// "K9 in detail" lists what was measured: tail slicing, load skipping, weight multicast, back-off waits).
#pragma once

#include <cuda.h> // CUtensorMap + enums only; the encode functions are fetched at run time (no -lcuda)
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#ifndef CCZ_CONV_BACKOFF_NS
#define CCZ_CONV_BACKOFF_NS 256 // poll interval of the roles that wait a whole tile ahead
#endif

namespace ccz {
namespace conv {

constexpr int C = 256;
constexpr int BOARD_H = 10, BOARD_W = 9, BOARD_HW = 90;
constexpr int BM = 128; // output pixels per CTA
constexpr int BN = 256; // all output channels
constexpr int BK = 64;  // one 128-byte swizzle row of bf16
constexpr int KBLOCKS = 9 * (C / BK);
constexpr int UMMA_K = 16;
constexpr int THREADS = 256;

template <int CG>
struct Cfg {
    static constexpr int B_ROWS = BN / CG;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = B_ROWS * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = CG == 2 ? 5 : 3;
    static constexpr int STAGING_BYTES = BM * BN * 2; // 4 boxes of 128 rows x 64 channels
    static constexpr int BIAS_BYTES = BN * 4;
    static constexpr int BAR_BYTES = 256;
    static constexpr int SMEM_BYTES = 1024 /*alignment slack*/ + STAGES * STAGE_BYTES + STAGING_BYTES + BIAS_BYTES + BAR_BYTES;
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on a barrier given by its shared::cluster address (own or peer CTA)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// Wait for the roles that are a whole tile ahead of their barrier (epilogue warps, skip-tile producer): sleep between
// polls instead of spinning.  Measured neutral (try_wait already suspends the warp in hardware); kept because it costs
// nothing and these roles have a whole main loop of slack.
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
            "selp.u32 %0, 1, 0, P1;\n"
            "}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(CCZ_CONV_BACKOFF_NS);
    }
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

constexpr uint64_t L2_HINT_DEFAULT = 0x1000000000000000ull;

// 2-D tiled load.  CG == 2: completes on the given shared::cluster barrier (the leader CTA's).
template <int CG>
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *m, uint32_t bar, int c0, int c1) {
    if constexpr (CG == 1) {
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
                     "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
                     : "memory");
    } else {
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], "
            "[%2], %5;" ::"r"(dst),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "l"(L2_HINT_DEFAULT)
            : "memory");
    }
}
// 4-D im2col load: (c, w, h, n) = first base pixel of the column, (off_w, off_h) = filter tap.
template <int CG>
__device__ __forceinline__ void tma_load_im2col(uint32_t dst, const CUtensorMap *m, uint32_t bar, int c, int w, int h, int n, uint16_t off_w,
                                                uint16_t off_h) {
    if constexpr (CG == 1) {
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::
                "r"(dst),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
            : "memory");
    } else {
        asm volatile(
            "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, "
            "%5, %6}], [%2], {%7, %8}, %9;" ::"r"(dst),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h), "l"(L2_HINT_DEFAULT)
            : "memory");
    }
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *m, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src),
                 "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t cols) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    if constexpr (CG == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
    else
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (CG == 1) {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// arrive on `bar` (same offset in every CTA of the pair) once all MMAs issued so far have completed
template <int CG>
__device__ __forceinline__ void umma_commit(uint32_t bar, uint16_t cta_mask) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    } else {
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                     "h"(cta_mask)
                     : "memory");
    }
}
// 2-D tiled load multicast to the CTAs in `cta_mask` (same smem offset in each); every destination's pair
// leader gets the complete_tx on its copy of the barrier (`bar` = the issuer's pair-leader barrier address).
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap *m, uint32_t bar, int c0, int c1, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint [%0], [%1, "
        "{%4, %5}], [%2], %3, %6;" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "h"(cta_mask), "r"(c0), "r"(c1), "l"(L2_HINT_DEFAULT)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// K-major, 128-byte-swizzled operand tile (rows of 64 bf16, 8-row groups 1024 B apart); the tile base
// is 1024-byte aligned.  Fields: start>>4 [0,14), LBO>>4 [16,30) (ignored for swizzled K-major, 1),
// SBO>>4 [32,46) = 64, version [46,48) = 1, layout [61,64) = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: fp32 accumulate [4,6)=1, A/B bf16 [7,10)=[10,13)=1, both K-major, N>>3 at 17, M>>4 at 24
__host__ __device__ constexpr uint32_t umma_idesc(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&t);
}

// ---- the kernel --------------------------------------------------------------------------------
// grid = n_clusters * CG CTAs (persistent); cluster c handles work items c, c + n_clusters, ...  The first
// n_full items are whole tiles (CG * 128 consecutive output pixels x all 256 output channels); the tiles of
// the last, partial round are split into `split` (1, 2 or 4) channel slices of 256/split so that the tail
// keeps every cluster busy for 1/split of a tile time instead of a few clusters for a whole one.
struct WorkItem {
    int tile, n_off, n_w;
};
__device__ __forceinline__ WorkItem work_item(int i, int n_full, int split_log2) {
    if (i < n_full) return {i, 0, BN};
    const int j = i - n_full, n_w = BN >> split_log2;
    return {n_full + (j >> split_log2), (j & ((1 << split_log2) - 1)) * n_w, n_w};
}

// Work plan of one launch: `n_tiles` cluster tiles over `clusters` resident clusters.  The tiles of the last, partial
// round are sliced into 2 or 4 output-channel slices while every slice still gets its own cluster.
struct Plan {
    int n_items, n_full, split_log2, clusters;
};
__host__ __device__ inline Plan plan_items(int n_tiles, int clusters, bool tail_split) {
    const int rem = n_tiles % clusters;
    int split_log2 = 0;
    if (tail_split && rem > 0) {
        while (split_log2 < 2 && (rem << (split_log2 + 1)) <= clusters) ++split_log2;
    }
    Plan p;
    p.split_log2 = split_log2;
    p.n_full = split_log2 ? n_tiles - rem : n_tiles;
    p.n_items = p.n_full + (split_log2 ? rem << split_log2 : 0);
    p.clusters = clusters > p.n_items ? p.n_items : clusters;
    return p;
}

// PAIRS > 1 (CG == 2 only): a cluster of PAIRS CTA pairs works on PAIRS consecutive tiles with the SAME weight
// stage: each CTA fetches 1/PAIRS of its half of the weight tile and multicasts it to the CTAs of equal
// parity, so weight traffic from L2 drops by PAIRS.  A stage is then free only when every pair has consumed it.
//
// DEV_COUNT: the board count is read from device memory (min(*d_count, count_cap), the tensor maps being encoded for
// count_cap boards), and every CTA derives the plan from it as the host does; the grid is every resident cluster and
// the clusters without an item only allocate / free TMEM and pass the cluster barriers.
template <int CG, int PAIRS, bool HAS_SKIP, bool DEV_COUNT>
__global__ void __launch_bounds__(THREADS, 1)
conv3x3_c256_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                    const __grid_constant__ CUtensorMap tm_skip, const __grid_constant__ CUtensorMap tm_y, const float *__restrict__ bias,
                    int n_items, int n_full, int split_log2, int dbg, const int32_t *__restrict__ d_count, int count_cap, int tail_split) {
    using K = Cfg<CG>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t a_smem = smem_base;
    const uint32_t b_smem = a_smem + K::STAGES * K::A_BYTES;
    const uint32_t staging = b_smem + K::STAGES * K::B_BYTES;
    const uint32_t bias_smem = staging + K::STAGING_BYTES;
    const uint32_t bars = bias_smem + K::BIAS_BYTES;
    const uint32_t bar_full = bars;                      // [STAGES]
    const uint32_t bar_empty = bars + 8 * K::STAGES;     // [STAGES]
    const uint32_t bar_tfull = bars + 16 * K::STAGES;    // [2]
    const uint32_t bar_tempty = bar_tfull + 16;          // [2]
    const uint32_t bar_skip = bar_tempty + 16;           // skip tile landed in staging
    const uint32_t bar_stfree = bar_skip + 8;            // staging tile may be overwritten
    const uint32_t tmem_slot = bar_stfree + 8;
    uint8_t *const smem_gen = smem_raw + (smem_base - smem_u32(smem_raw)); // generic pointer to smem_base

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    static_assert(CG == 2 || PAIRS == 1, "weight multicast needs CTA pairs");
    constexpr int CLUSTER = CG * PAIRS;
    const uint32_t rank = CLUSTER > 1 ? cluster_ctarank() : 0u;
    const uint32_t prank = rank % CG, pair_id = rank / CG, lead_rank = rank - prank; // position in the pair / pair in the cluster
    const int cluster_id = blockIdx.x / CLUSTER, n_clusters = gridDim.x / CLUSTER;
    if constexpr (DEV_COUNT) {
        const int nb = min(max(*d_count, 0), count_cap), rows_per_tile = BM * CLUSTER;
        const Plan pl = plan_items((nb * BOARD_HW + rows_per_tile - 1) / rows_per_tile, n_clusters, tail_split != 0);
        n_items = pl.n_items;
        n_full = pl.n_full;
        split_log2 = pl.split_log2;
    }

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_x);
        tma_prefetch_desc(&tm_w);
        tma_prefetch_desc(&tm_y);
        if (HAS_SKIP) tma_prefetch_desc(&tm_skip);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < K::STAGES; ++i) {
            mbar_init(bar_full + 8 * i, 1);
            mbar_init(bar_empty + 8 * i, PAIRS);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar_tfull + 8 * i, 1);
            mbar_init(bar_tempty + 8 * i, 4 * CG);
        }
        mbar_init(bar_skip, 1);
        mbar_init(bar_stfree, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) tmem_alloc<CG>(tmem_slot, 512);
    if (warp >= 4) {
        const int t = threadIdx.x - 128;
        reinterpret_cast<float *>(smem_gen + (bias_smem - smem_base))[t] = bias[t];
        reinterpret_cast<float *>(smem_gen + (bias_smem - smem_base))[t + 128] = bias[t + 128];
    }
    tc_fence_before();
    if constexpr (CLUSTER > 1) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem_gen + (tmem_slot - smem_base));

    if (warp == 0) {
        // ===== A/B producer =====
        if (lane == 0) {
            const uint32_t full0 = CG == 2 ? mapa(bar_full, lead_rank) : bar_full; // the pair leader's full barriers
            constexpr int SLICE_ROWS = K::B_ROWS / PAIRS;
            uint16_t mc_mask = 0;
            for (int j = 0; j < PAIRS; ++j) mc_mask |= (uint16_t)(1u << (j * CG + prank));
            int stage = 0;
            uint32_t phase = 0;
            for (int item = cluster_id; item < n_items; item += n_clusters) {
                const WorkItem wi = work_item(item, n_full, split_log2);
                const int m0 = ((wi.tile * PAIRS + (int)pair_id) * CG + (int)prank) * BM;
                const int b_row = wi.n_off + (int)prank * (wi.n_w / CG); // a channel slice over-reads rows it does not use
                const int img = m0 / BOARD_HW, rem = m0 - img * BOARD_HW;
                const int p = rem / BOARD_W, q = rem - p * BOARD_W;
                for (int kb = 0; kb < KBLOCKS; ++kb) {
                    const int tap = kb >> 2, c0 = (kb & 3) * BK;
                    const int r = tap / 3, s = tap - 3 * r;
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    const bool do_a = !((dbg & 2) && (kb & 1)), do_b = !((dbg & 1) && (kb & 1)); // traffic-sensitivity experiment
                    if (prank == 0) mbar_expect_tx(bar_full + 8 * stage, CG * ((do_a ? K::A_BYTES : 0) + (do_b ? K::B_BYTES : 0)));
                    if (do_a) tma_load_im2col<CG>(a_smem + stage * K::A_BYTES, &tm_x, full0 + 8 * stage, c0, q - 1, p - 1, img, (uint16_t)s, (uint16_t)r);
                    if constexpr (PAIRS == 1) {
                        if (do_b) tma_load_2d<CG>(b_smem + stage * K::B_BYTES, &tm_w, full0 + 8 * stage, kb * BK, b_row);
                    } else {
                        tma_load_2d_mc(b_smem + stage * K::B_BYTES + (int)pair_id * SLICE_ROWS * 128, &tm_w, full0 + 8 * stage, kb * BK,
                                       b_row + (int)pair_id * SLICE_ROWS, mc_mask);
                    }
                    if (++stage == K::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (leader CTA only) =====
        if (prank == 0 && lane == 0) {
            constexpr uint16_t mask_cluster = (uint16_t)((1u << CLUSTER) - 1);
            const uint16_t mask_pair = (uint16_t)(((1u << CG) - 1) << lead_rank);
            int stage = 0;
            uint32_t phase = 0, acc = 0, acc_phase = 0;
            for (int item = cluster_id; item < n_items; item += n_clusters) {
                const uint32_t idesc = umma_idesc(BM * CG, work_item(item, n_full, split_log2).n_w);
                mbar_wait_cluster(bar_tempty + 8 * acc, acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < KBLOCKS; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint64_t a_desc = umma_desc_sw128(a_smem + stage * K::A_BYTES);
                    const uint64_t b_desc = umma_desc_sw128(b_smem + stage * K::B_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) // +32 bytes along K inside the swizzle row
                        umma_bf16<CG>(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (uint32_t)((kb | k) != 0));
                    umma_commit<CG>(bar_empty + 8 * stage, mask_cluster);
                    if (++stage == K::STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit<CG>(bar_tfull + 8 * acc, mask_pair);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp == 3) {
        // ===== skip-tile producer: prefetch skip[m0 : m0+128, :] into the staging tile =====
        if (HAS_SKIP && lane == 0) {
            uint32_t it = 0;
            for (int item = cluster_id; item < n_items; item += n_clusters, ++it) {
                const WorkItem wi = work_item(item, n_full, split_log2);
                const int m0 = ((wi.tile * PAIRS + (int)pair_id) * CG + (int)prank) * BM;
                mbar_wait_relaxed(bar_stfree, (it & 1) ^ 1);
                mbar_expect_tx(bar_skip, (wi.n_w / 64) * (BM * 128));
                for (int g = 0; g < wi.n_w / 64; ++g) tma_load_2d<1>(staging + g * (BM * 128), &tm_skip, bar_skip, wi.n_off + g * 64, m0);
            }
        }
    } else if (warp >= 4) {
        // ===== epilogue: thread = one output pixel (TMEM lane), 256 channels =====
        const int quarter = warp - 4, row = quarter * 32 + lane;
        const uint32_t tempty0 = CG == 2 ? mapa(bar_tempty, lead_rank) : bar_tempty;
        const float *bias_s = reinterpret_cast<const float *>(smem_gen + (bias_smem - smem_base));
        uint8_t *stg = smem_gen + (staging - smem_base);
        uint32_t acc = 0, acc_phase = 0, it = 0;
        for (int item = cluster_id; item < n_items; item += n_clusters, ++it) {
            const WorkItem wi = work_item(item, n_full, split_log2);
            const int m0 = ((wi.tile * PAIRS + (int)pair_id) * CG + (int)prank) * BM;
            if (HAS_SKIP) mbar_wait_relaxed(bar_skip, it & 1);
            mbar_wait_relaxed(bar_tfull + 8 * acc, acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN;
#pragma unroll 1
            for (int chunk = 0; chunk < wi.n_w / 32; ++chunk) { // 32 channels per chunk
                uint32_t v[32];
                tmem_ld32(t_row + chunk * 32, v);
                tmem_ld_wait();
                uint8_t *box_row = stg + (chunk >> 1) * (BM * 128) + row * 128;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int c16 = (chunk & 1) * 4 + j; // 16-byte column of the 128-byte row
                    uint4 *cell = reinterpret_cast<uint4 *>(box_row + ((c16 ^ (row & 7)) << 4));
                    const float4 b0 = *reinterpret_cast<const float4 *>(bias_s + wi.n_off + chunk * 32 + j * 8);
                    const float4 b1 = *reinterpret_cast<const float4 *>(bias_s + wi.n_off + chunk * 32 + j * 8 + 4);
                    float f[8] = {__uint_as_float(v[j * 8 + 0]) + b0.x, __uint_as_float(v[j * 8 + 1]) + b0.y,
                                  __uint_as_float(v[j * 8 + 2]) + b0.z, __uint_as_float(v[j * 8 + 3]) + b0.w,
                                  __uint_as_float(v[j * 8 + 4]) + b1.x, __uint_as_float(v[j * 8 + 5]) + b1.y,
                                  __uint_as_float(v[j * 8 + 6]) + b1.z, __uint_as_float(v[j * 8 + 7]) + b1.w};
                    if (HAS_SKIP) {
                        const uint4 sk = *cell;
                        const uint32_t w[4] = {sk.x, sk.y, sk.z, sk.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            f[2 * e] += __uint_as_float(w[e] << 16);
                            f[2 * e + 1] += __uint_as_float(w[e] & 0xFFFF0000u);
                        }
                    }
                    uint4 o;
                    o.x = pack_bf16x2(fmaxf(f[0], 0.f), fmaxf(f[1], 0.f));
                    o.y = pack_bf16x2(fmaxf(f[2], 0.f), fmaxf(f[3], 0.f));
                    o.z = pack_bf16x2(fmaxf(f[4], 0.f), fmaxf(f[5], 0.f));
                    o.w = pack_bf16x2(fmaxf(f[6], 0.f), fmaxf(f[7], 0.f));
                    *cell = o;
                }
            }
            // accumulator buffer drained: hand it back to the MMA issuer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (CG == 2) mbar_arrive_cluster(tempty0 + 8 * acc); else mbar_arrive(bar_tempty + 8 * acc);
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            // staging tile -> global
            fence_proxy_async();
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (threadIdx.x == 128) {
                for (int g = 0; g < wi.n_w / 64; ++g) tma_store_2d(&tm_y, staging + g * (BM * 128), wi.n_off + g * 64, m0);
                tma_store_commit();
                tma_store_wait_read();
                if (HAS_SKIP) mbar_arrive(bar_stfree);
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        if (threadIdx.x == 128) tma_store_wait_all();
    }

    // teardown (re-converge the single-lane role warps before the aligned barriers)
    __syncwarp();
    tc_fence_before();
    if constexpr (CLUSTER > 1) cluster_sync_all(); else __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<CG>(tmem_base, 512);
    }
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const int *,
                                   const int *, cuuint32_t, cuuint32_t, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct Driver {
    EncodeTiledFn tiled = nullptr;
    EncodeIm2colFn im2col = nullptr;
    bool ready = false;
};

inline const char *driver_init(Driver &d) {
    if (d.ready) return nullptr;
    cudaDriverEntryPointQueryResult q;
    void *f = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !f)
        return "cuTensorMapEncodeTiled not available from the driver";
    d.tiled = reinterpret_cast<EncodeTiledFn>(f);
    f = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !f)
        return "cuTensorMapEncodeIm2col not available from the driver";
    d.im2col = reinterpret_cast<EncodeIm2colFn>(f);
    d.ready = true;
    return nullptr;
}

// [rows, 256] bf16 row-major matrix, box = 64 channels x box_rows rows, 128-byte swizzle
inline bool encode_rows(const Driver &d, CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {cols * 2};
    const cuuint32_t box[2] = {64, box_rows};
    const cuuint32_t es[2] = {1, 1};
    return d.tiled(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// NHWC activations [n,10,9,256] for a 3x3 / pad 1 fprop: base pixels span [-1, dim-1+(-1)] in w and h,
// the filter tap is added by the instruction's offsets; 64 channels x 128 pixels per load.
inline bool encode_im2col(const Driver &d, CUtensorMap *m, const void *ptr, int n) {
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)BOARD_W, (cuuint64_t)BOARD_H, (cuuint64_t)n};
    const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * BOARD_W, (cuuint64_t)C * 2 * BOARD_HW};
    const int lower[2] = {-1, -1}, upper[2] = {-1, -1};
    const cuuint32_t es[4] = {1, 1, 1, 1};
    return d.im2col(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(ptr), dims, strides, lower, upper, BK, BM, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// d_count == nullptr: `n_tiles` cluster tiles planned here.  Otherwise the kernel plans from min(*d_count, count_cap)
// boards on the device and every resident cluster is launched.
template <int CG, int PAIRS, bool HAS_SKIP, bool DEV_COUNT>
inline cudaError_t launch_variant(const CUtensorMap &tx, const CUtensorMap &tw, const CUtensorMap &ts, const CUtensorMap &ty, const float *bias,
                                  int n_tiles, int tail_split, int dbg, const int32_t *d_count, int count_cap, cudaStream_t stream) {
    auto kern = conv3x3_c256_kernel<CG, PAIRS, HAS_SKIP, DEV_COUNT>;
    constexpr int CLUSTER = CG * PAIRS;
    // per device: resident clusters of this shape (GPC boundaries can strand SMs for CLUSTER > 2); function
    // attributes are per device too
    static int max_clusters_dev[64] = {0};
    int dev = 0, n_sm = 0;
    cudaError_t e0 = cudaGetDevice(&dev);
    if (e0 != cudaSuccess) return e0;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    int &max_clusters = max_clusters_dev[dev];
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = Cfg<CG>::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CLUSTER;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (!max_clusters) {
        cudaError_t e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<CG>::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        cfg.gridDim = dim3((unsigned)(n_sm / CLUSTER * CLUSTER));
        int n = 0;
        e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
        if (e != cudaSuccess) return e;
        if (n < 1) return cudaErrorInvalidConfiguration;
        max_clusters = n < n_sm / CLUSTER ? n : n_sm / CLUSTER;
    }
    if constexpr (DEV_COUNT) {
        cfg.gridDim = dim3((unsigned)(max_clusters * CLUSTER));
        return cudaLaunchKernelEx(&cfg, kern, tx, tw, ts, ty, bias, 0, 0, 0, dbg, d_count, count_cap, tail_split);
    }
    const Plan pl = plan_items(n_tiles, max_clusters, tail_split != 0);
    cfg.gridDim = dim3((unsigned)(pl.clusters * CLUSTER));
    return cudaLaunchKernelEx(&cfg, kern, tx, tw, ts, ty, bias, pl.n_items, pl.n_full, pl.split_log2, dbg, (const int32_t *)nullptr, 0, 0);
}

} // namespace conv
} // namespace ccz
