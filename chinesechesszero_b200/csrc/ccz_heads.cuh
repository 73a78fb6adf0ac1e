// ccz_heads.cuh -- K11: operand packing between the fused 1x1 head convolutions and the two FC layers of
// Net.forward (net.py:94-107).  The head GEMM leaves h[pixel row][32] (17 policy + 7 value channels + 8 pad,
// bias added, NHWC); the FC layers want, per board, the NCHW-flattened channel-major vectors
// x.view(-1, 17*90) / x.view(-1, 7*90) (net.py:97,104) after the ReLU (net.py:96,103).  One CTA per board:
// the 90 x 32 tile goes through shared memory, ReLU is applied on the way, and both operands are written as
// contiguous 4-byte words into the K-padded rows the aligned cuBLAS kernels consume ([policy 1530 -> kp |
// value 630 -> kv]; the pad columns are never written and stay zero).  Replaces three torch element-wise
// launches (ReLU + two strided transposing copies, 2 x 48 us per 4096 boards) by one (HBM-bound: 5.8 KB in,
// 4.3 KB out per board).  `rows` (may be NULL = identity): board b's operands come from h's board rows[b], so the
// FC layers see G rows when the 1x1 GEMM ran on K12's compacted distinct leaves.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace ccz {
namespace heads {

constexpr int HW = 90, CH = 32, N_POLICY = 17, N_VALUE = 7, THREADS = 128;

__global__ void __launch_bounds__(THREADS)
heads_pack_kernel(const uint4 *__restrict__ h /*[n*90*32 bf16]*/, uint32_t *__restrict__ out /*[n][row_words]*/, int n,
                  int row_words, int value_word_off, const int32_t *__restrict__ rows) {
    __shared__ __align__(16) uint16_t s_t[HW][CH + 2]; // +2 halfwords: the column reads below hit distinct banks
    const int b = blockIdx.x;
    if (b >= n) return;
    const uint4 *src = h + (size_t)(rows ? rows[b] : b) * (HW * CH * 2 / 16);
    for (int i = threadIdx.x; i < HW * CH * 2 / 16; i += THREADS) {
        const uint4 v = src[i];
        const int row = i >> 2, col = (i & 3) * 8; // 4 vectors of 8 channels per pixel row
        uint32_t *d = reinterpret_cast<uint32_t *>(&s_t[row][col]);
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    __syncthreads();
    auto relu = [](uint16_t x) -> uint32_t { return (x & 0x8000u) ? 0u : (uint32_t)x; }; // bf16: sign bit set -> 0 (-0, NaN<0 too)
    uint32_t *row = out + (size_t)b * row_words;
    for (int w = threadIdx.x; w < N_POLICY * HW / 2; w += THREADS) { // 765 words: channel-major policy operand
        const int e0 = 2 * w, e1 = e0 + 1;
        row[w] = relu(s_t[e0 % HW][e0 / HW]) | relu(s_t[e1 % HW][e1 / HW]) << 16;
    }
    for (int w = threadIdx.x; w < N_VALUE * HW / 2; w += THREADS) { // 315 words: value operand
        const int e0 = 2 * w, e1 = e0 + 1;
        row[value_word_off + w] = relu(s_t[e0 % HW][N_POLICY + e0 / HW]) | relu(s_t[e1 % HW][N_POLICY + e1 / HW]) << 16;
    }
}

} // namespace heads
} // namespace ccz
