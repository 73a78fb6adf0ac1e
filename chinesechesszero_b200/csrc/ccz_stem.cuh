// ccz_stem.cuh -- K10: the stem of Net.forward (conv_block 119->256, 3x3, pad 1, + folded BN + ReLU;
// reference net.py:84) evaluated straight from 96-byte board records for SEARCH-TIME inputs.
//
// policy_value_fn feeds the net 7 all-zero history states, the current one-hot piece planes and a
// constant turn plane (net.py:160-177): input channel 49+t-1 is 1 where a red piece of type t stands,
// 105+t-1 likewise for black, channels 112..118 all equal `turn`, every other channel is 0.  With a
// one-hot input the convolution is a sum of at most nine rows of the weight tensor per output pixel:
//
//   y[p, :] = relu( bias_turn[turn][border_class(p)][:] + sum_{tap: p+tap on the board, occupied} table[tap][code(p+tap)][:] )
//
//   table[tap][code][co]      = W[co, channel(code), tap]           (bf16, exactly the conv's folded weight)
//   bias_turn[t][class][co]   = bias[co] + t * sum_{valid taps of the class} sum_{c=112..118} W[co, c, tap]   (fp32)
//
// No planes are read (21 KB / position saved), no channel padding, no layout copy: the kernel is bound by
// the 46 KB / board NHWC bf16 output it writes.  One warp per board, lane = 8 output channels; tables
// (92 KB) staged in shared memory once per persistent CTA.  DEV_COUNT: the board count is min(*d_count, n), read
// on the device (K12's number of distinct leaves); warps past it exit.  QOUT: also an e4m3 copy of the output,
// yq = satfinite(bf16(y) * *inv_s) (the A operand of the first e4m3 tower convolution; the bf16 y stays the skip).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "ccz_conv.cuh" // pack_e4m3x4

namespace ccz {
namespace stem {

constexpr int C_OUT = 256;
constexpr int TABLE_ELEMS = 9 * 16 * C_OUT;      // bf16
constexpr int BIAS_TURN_ELEMS = 2 * 9 * C_OUT;   // fp32
constexpr int WARPS = 16; // two CTAs of 16 warps per SM (92 KB of tables each): 32 warps hide the LDS / STG latency
constexpr int SMEM_BYTES = TABLE_ELEMS * 2 + BIAS_TURN_ELEMS * 4 + WARPS * 96;

// acc[0..7] += the 8 bf16 channels of one table row (16 bytes per lane)
__device__ __forceinline__ void add_row(float (&acc)[8], const uint4 t) {
    const uint32_t v[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        acc[2 * e] += __uint_as_float(v[e] << 16);
        acc[2 * e + 1] += __uint_as_float(v[e] & 0xFFFF0000u);
    }
}

template <bool DEV_COUNT, bool QOUT = false>
__global__ void __launch_bounds__(WARPS * 32, 2)
stem_lookup_kernel(const uint8_t *__restrict__ boards, int n, const uint4 *__restrict__ table, const float4 *__restrict__ bias_turn,
                   uint4 *__restrict__ y, const int32_t *__restrict__ d_count, uint2 *__restrict__ yq = nullptr,
                   const float *__restrict__ inv_s = nullptr) {
    if constexpr (DEV_COUNT) n = min(*d_count, n);
    [[maybe_unused]] float qs = 0.f;
    if constexpr (QOUT) qs = *inv_s;
    extern __shared__ __align__(16) uint8_t smem[];
    uint4 *tab_s = reinterpret_cast<uint4 *>(smem);
    float4 *bt_s = reinterpret_cast<float4 *>(smem + TABLE_ELEMS * 2);
    uint8_t *brd_s = smem + TABLE_ELEMS * 2 + BIAS_TURN_ELEMS * 4;
    for (int i = threadIdx.x; i < TABLE_ELEMS * 2 / 16; i += blockDim.x) tab_s[i] = table[i];
    for (int i = threadIdx.x; i < BIAS_TURN_ELEMS * 4 / 16; i += blockDim.x) bt_s[i] = bias_turn[i];
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *my_board = brd_s + warp * 96;
    const uint4 *tab_lane = tab_s + lane; // row e of the table for this lane's 8 channels: tab_lane[e * 32]
    for (int b = blockIdx.x * WARPS + warp; b < n; b += gridDim.x * WARPS) {
        __syncwarp();
        reinterpret_cast<uint32_t *>(my_board)[lane < 24 ? lane : 0] =
            reinterpret_cast<const uint32_t *>(boards + (size_t)b * 96)[lane < 24 ? lane : 0];
        __syncwarp();
        const int turn = my_board[90] ? 1 : 0;
        uint4 *out = y + (size_t)b * 90 * (C_OUT / 8) + lane;
#pragma unroll 1
        for (int h = 0; h < 10; ++h) {
            const int rc = h == 0 ? 0 : (h == 9 ? 2 : 1);
            // table-row index (tap-independent part: piece code, 0 = nothing to add) of the three board rows around h;
            // all lanes hold the same values (broadcast loads), so every branch below is warp-uniform
            uint64_t code[3]; // nine 4-bit codes per row
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const int nh = h + r - 1;
                uint64_t packed = 0;
                if (nh >= 0 && nh <= 9) {
#pragma unroll
                    for (int w = 0; w < 9; ++w) {
                        const uint32_t c = my_board[nh * 9 + w];
                        packed |= (uint64_t)((c & 7) ? (c & 15) : 0) << (4 * w);
                    }
                }
                code[r] = packed;
            }
            const float4 *bt_row = bt_s + ((turn * 9 + rc * 3) * C_OUT + lane * 8) / 4;
#pragma unroll
            for (int w = 0; w < 9; ++w) { // unrolled: the w-border taps and the border class are compile-time
                const int cc = w == 0 ? 0 : (w == 8 ? 2 : 1);
                const float4 a0 = bt_row[cc * (C_OUT / 4)], a1 = bt_row[cc * (C_OUT / 4) + 1];
                float acc[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                for (int r = 0; r < 3; ++r) {
#pragma unroll
                    for (int s = 0; s < 3; ++s) {
                        const int nw = w + s - 1;
                        if (nw < 0 || nw > 8) continue;
                        const int c = (int)(code[r] >> (4 * nw)) & 15;
                        if (c) add_row(acc, tab_lane[((r * 3 + s) * 16 + c) * (C_OUT / 8)]);
                    }
                }
                uint4 o;
                __nv_bfloat162 p0 = __floats2bfloat162_rn(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f));
                __nv_bfloat162 p1 = __floats2bfloat162_rn(fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f));
                __nv_bfloat162 p2 = __floats2bfloat162_rn(fmaxf(acc[4], 0.f), fmaxf(acc[5], 0.f));
                __nv_bfloat162 p3 = __floats2bfloat162_rn(fmaxf(acc[6], 0.f), fmaxf(acc[7], 0.f));
                o.x = *reinterpret_cast<uint32_t *>(&p0);
                o.y = *reinterpret_cast<uint32_t *>(&p1);
                o.z = *reinterpret_cast<uint32_t *>(&p2);
                o.w = *reinterpret_cast<uint32_t *>(&p3);
                out[(h * 9 + w) * (C_OUT / 8)] = o; // 32 lanes x 16 B = one 512-byte NHWC pixel row
                if constexpr (QOUT) {
                    const float2 f0 = __bfloat1622float2(p0), f1 = __bfloat1622float2(p1), f2 = __bfloat1622float2(p2),
                                 f3 = __bfloat1622float2(p3);
                    yq[((size_t)b * 90 + h * 9 + w) * (C_OUT / 8) + lane] =
                        make_uint2(conv::pack_e4m3x4(f0.x * qs, f0.y * qs, f1.x * qs, f1.y * qs),
                                   conv::pack_e4m3x4(f2.x * qs, f2.y * qs, f3.x * qs, f3.y * qs));
                }
            }
        }
    }
}

} // namespace stem
} // namespace ccz
