// ccz_dedup.cuh -- K12: the distinct positions of a lockstep leaf batch, so the forward runs once per position.
//
// At search time the net input depends only on the 90 squares and the side to move (net.py:160-177): bytes 0..90
// of a board record.  Many games of a batch send the same leaf (every game in its first move searches the same tree
// from the start position, games that opened with the same move share their second search), so the evaluator
// forwards the distinct records only and maps the results back.
//
// One CTA, everything in shared memory:
//   1. every board is inserted into an open-addressing table (2 x next_pow2(n) slots, linear probing, slot picked by
//      a 64-bit hash of its 23 key words).  A slot goes from EMPTY to the index of the first board that claims it and
//      afterwards only to smaller indices of the same position (atomicMin), so the position a slot holds never
//      changes and a probe compares the key bytes once per occupied slot;
//   2. rep[g] = the smallest game index of g's position;
//   3. a block scan over "rep[g] == g" numbers the distinct positions in order of first occurrence;
//   4. rows[g] = number of rep[g]; the first occurrence copies its record to uniq[rows[g]].
// The result does not depend on thread timing.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

namespace ccz {
namespace dedup {

constexpr int THREADS = 1024;
constexpr int MAX_BOARDS = 16384;
constexpr int KEY_WORDS = 23; // bytes 0..90: 22 whole words + the low 3 bytes of word 22
constexpr uint32_t EMPTY = 0x7fffffffu;

__host__ __device__ inline int table_slots(int n) {
    int t = 64;
    while (t < 2 * n) t <<= 1;
    return t;
}
__host__ __device__ inline int smem_bytes(int n) { return (table_slots(n) + n) * 4; }

__device__ __forceinline__ uint32_t key_word(const uint32_t *rec, int i) { return i < KEY_WORDS - 1 ? rec[i] : rec[i] & 0x00FFFFFFu; }

__global__ void __launch_bounds__(THREADS, 1)
leaf_unique_kernel(const uint8_t *__restrict__ boards, int n, int32_t *__restrict__ rows, uint8_t *__restrict__ uniq,
                   int32_t *__restrict__ n_unique, unsigned long long *__restrict__ total) {
    extern __shared__ uint32_t sm[];
    const int T = table_slots(n);
    uint32_t *table = sm;              // [T] -> reused as the number of each first occurrence in step 3
    int32_t *rep = (int32_t *)(sm + T); // [n]: slot of g, then the smallest index of g's position
    __shared__ int warp_sum[THREADS / 32];
    for (int i = threadIdx.x; i < T; i += THREADS) table[i] = EMPTY;
    __syncthreads();

    for (int g = threadIdx.x; g < n; g += THREADS) {
        const uint32_t *rec = reinterpret_cast<const uint32_t *>(boards + (size_t)g * 96);
        uint32_t key[KEY_WORDS];
        uint64_t h = 0x9E3779B97F4A7C15ull;
#pragma unroll
        for (int i = 0; i < KEY_WORDS; ++i) {
            key[i] = key_word(rec, i);
            h = (h ^ key[i]) * 0x100000001B3ull;
            h ^= h >> 29;
        }
        h *= 0xBF58476D1CE4E5B9ull;
        int slot = (int)((h ^ (h >> 32)) & (uint64_t)(T - 1));
        for (;;) {
            uint32_t v = atomicCAS(&table[slot], EMPTY, (uint32_t)g);
            if (v == EMPTY) break; // claimed a free slot
            const uint32_t *other = reinterpret_cast<const uint32_t *>(boards + (size_t)v * 96);
            bool same = true;
#pragma unroll
            for (int i = 0; i < KEY_WORDS; ++i) same &= key_word(other, i) == key[i];
            if (same) {
                atomicMin(&table[slot], (uint32_t)g);
                break;
            }
            slot = (slot + 1) & (T - 1);
        }
        rep[g] = slot;
    }
    __syncthreads();
    for (int g = threadIdx.x; g < n; g += THREADS) rep[g] = (int32_t)table[rep[g]];
    __syncthreads();

    // block-wide exclusive scan of the first-occurrence flags; thread t owns boards [t*per, (t+1)*per)
    const int per = (n + THREADS - 1) / THREADS, lo = threadIdx.x * per, hi = min(lo + per, n);
    int cnt = 0;
    for (int g = lo; g < hi; ++g) cnt += rep[g] == g;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += y;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int s = warp_sum[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        warp_sum[lane] = s; // inclusive over warps
    }
    __syncthreads();
    int next = incl - cnt + (warp ? warp_sum[warp - 1] : 0);
    for (int g = lo; g < hi; ++g)
        if (rep[g] == g) table[g] = (uint32_t)next++;
    if (threadIdx.x == 0) {
        const int u = warp_sum[THREADS / 32 - 1];
        *n_unique = u;
        if (total) atomicAdd(total, (unsigned long long)u);
    }
    __syncthreads();

    for (int g = threadIdx.x; g < n; g += THREADS) {
        const int r = (int)table[rep[g]];
        rows[g] = r;
        if (rep[g] == g) {
            const uint4 *src = reinterpret_cast<const uint4 *>(boards + (size_t)g * 96);
            uint4 *dst = reinterpret_cast<uint4 *>(uniq + (size_t)r * 96);
#pragma unroll
            for (int i = 0; i < 6; ++i) dst[i] = src[i];
        }
    }
}

} // namespace dedup
} // namespace ccz
