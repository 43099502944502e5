// Shared device helpers for the pagnerf_b200 kernels (sm_100a).
//
// Bit-exactness rule: every float expression that decides an INTEGER result (octree cell,
// lattice vertex, hash index, kept/dropped sample) is written with explicitly rounded
// intrinsics (__fmul_rn / __fadd_rn / __fmaf_rn / __fdiv_rn) so nvcc can neither contract nor
// reassociate it; the CPU oracle (oracle/f32.py) evaluates the same op sequence in numpy float32.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PAG_OK 0
#define PAG_ERR_ARG (-1)
#define PAG_ERR_UNSUPPORTED (-2)

#define PAG_LAUNCH_CHECK()                                   \
    do {                                                     \
        cudaError_t e__ = cudaGetLastError();                \
        if (e__ != cudaSuccess) return (int)e__;             \
    } while (0)

static inline int pag_grid(int64_t n, int block) { return (int)((n + block - 1) / block); }

// lowbias32 mixer; jitter u in [0,1) for flat index `idx` (oracle/f32.py::jitter_u01)
__device__ __forceinline__ uint32_t pag_lowbias32(uint32_t x) {
    x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ float pag_jitter(uint32_t seed, uint64_t idx) {
    uint32_t x = (uint32_t)(idx + (uint64_t)seed * 0x9E3779B9ull);
    return (float)(pag_lowbias32(x) >> 8) * (1.0f / 16777216.0f);
}

// open-addressing hash tables of 64-bit keys (key 0 = empty slot), linear probing, C a power of two.  pag_hash_slots(n): the
// smallest power of two >= 2n, so that n distinct keys fill at most half of a table: it never overflows, whatever the data.
static inline int64_t pag_hash_slots(int64_t n) {
    int64_t c = 2;
    while (c < 2 * n) c <<= 1;
    return c;
}

__device__ __forceinline__ uint32_t pag_hash64(unsigned long long k) {      // murmur3 fmix64
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return (uint32_t)k;
}

// slot of `key` in table[C], inserted if absent; *inserted says whether this call put it there.  A slot's key goes from 0 to its
// final value once, so a plain load that sees the key (or another key) is final; a stale 0 only sends us to the CAS, which
// returns the truth.
__device__ __forceinline__ uint32_t pag_hash_insert(unsigned long long* __restrict__ table, uint32_t C, unsigned long long key,
                                                    bool* inserted) {
    uint32_t s = pag_hash64(key) & (C - 1);
    while (true) {
        unsigned long long cur = __ldcg(table + s);
        if (cur == 0ull) cur = atomicCAS(table + s, 0ull, key);
        if (cur == 0ull || cur == key) { *inserted = cur == 0ull; return s; }
        s = (s + 1) & (C - 1);
    }
}

__device__ __forceinline__ float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// fire-and-forget vector reduction (sm_90+: red.global.add.v2.f32)
__device__ __forceinline__ void red_add_f32x2(float* addr, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void red_add_f32x4(float* addr, float a, float b, float c, float d) {   // addr 16-byte aligned
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add_f32(float* addr, float a) {
    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(a) : "memory");
}

// warp-aggregated scatter of (gx,gy) into tl[idx]: lanes with equal idx are summed, the leader issues one red
// todo0: lanes that have something to add (lanes with an exactly-zero gradient take part in the shuffles only)
__device__ __forceinline__ void scatter_aggregated(float* __restrict__ tl, uint32_t idx, float gx, float gy,
                                                   unsigned active, unsigned todo0) {
    unsigned todo = todo0;
    const int lane = threadIdx.x & 31;
    while (todo) {
        const int leader = __ffs(todo) - 1;
        const uint32_t key = __shfl_sync(active, idx, leader);
        const unsigned same = __ballot_sync(active, idx == key) & todo;
        float sx = (idx == key) ? gx : 0.f, sy = (idx == key) ? gy : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sx += __shfl_xor_sync(active, sx, o);
            sy += __shfl_xor_sync(active, sy, o);
        }
        if (lane == leader) red_add_f32x2(tl + 2 * (size_t)key, sx, sy);
        todo &= ~same;
    }
}

