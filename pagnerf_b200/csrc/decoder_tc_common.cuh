// Helpers shared by the tensor-core decoder kernels (decoder_tc.cu, decoder_tc_fused.cu).
#pragma once
#include "decoder_common.cuh"
#include "tc_common.cuh"
#include <cuda_fp16.h>

#define TCH TC_CHUNK_BYTES

// Phase timeline instrumentation (python -m pagnerf_b200.build --phase-timing -> libpagnerf_b200_dbg.so): thread 0 of
// block 0 accumulates the clock64 ticks between consecutive PAG_PHASE marks; read with pag_debug_phase_read.
#ifdef PAG_PHASE_TIMING
static __device__ unsigned long long pag_phase_clk[64];   // one copy per translation unit
#define PAG_PHASE_READER(name)                                                                        \
    extern "C" int name(unsigned long long* host64, int reset) {                                      \
        cudaError_t e = cudaMemcpyFromSymbol(host64, pag_phase_clk, sizeof(unsigned long long) * 64); \
        if (e != cudaSuccess) return (int)e;                                                          \
        if (reset) {                                                                                  \
            unsigned long long z[64] = {0};                                                           \
            e = cudaMemcpyToSymbol(pag_phase_clk, z, sizeof(z));                                      \
        }                                                                                             \
        return (int)e;                                                                                \
    }
// accumulate in shared memory (a global read-modify-write per mark would stall thread 0 for an L2 round trip and
// distort the very timeline being measured); PAG_PHASE_FLUSH adds the block-0 totals to the global counters
#define PAG_PHASE_INIT()                                                     \
    __shared__ unsigned long long _ph_s[64];                                 \
    if (threadIdx.x < 64) _ph_s[threadIdx.x] = 0ull;                         \
    __syncthreads();                                                         \
    unsigned long long _ph_t = clock64()
#define PAG_PHASE(i)                                                         \
    do {                                                                     \
        if (blockIdx.x == 0 && threadIdx.x == 0) {                           \
            const unsigned long long _t = clock64();                         \
            _ph_s[i] += _t - _ph_t;                                          \
            _ph_t = _t;                                                      \
        }                                                                    \
    } while (0)
#define PAG_PHASE_FLUSH()                                                    \
    do {                                                                     \
        __syncthreads();                                                     \
        if (blockIdx.x == 0 && threadIdx.x < 64) pag_phase_clk[threadIdx.x] += _ph_s[threadIdx.x]; \
    } while (0)
#else
#define PAG_PHASE_INIT()
#define PAG_PHASE(i)
#define PAG_PHASE_FLUSH()
#define PAG_PHASE_READER(name)
#endif

// ---------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
// features [8c, 8c+8) of row `row` into chunk c of a tile image
__device__ __forceinline__ void tile_store8(uint8_t* tile, int c, int row, const float* v) {
    uint4 u;
    u.x = pack_h2(v[0], v[1]); u.y = pack_h2(v[2], v[3]); u.z = pack_h2(v[4], v[5]); u.w = pack_h2(v[6], v[7]);
    *reinterpret_cast<uint4*>(tile + c * TCH + row * 16) = u;
}
// fp16 image of W[OUT][IN] (global fp32, torch Linear layout): [(in/8)][OUTP][8], zero padded
// colscale (nullable, [IN]): per-input-feature factor folded into the weights, W' = W diag(colscale) -- the LOD weights
// of the feature vector never touch the per-sample path (Y = (x*s) W^T = x W'^T, dX = (G W) * s = G W')
__device__ __forceinline__ void stage_w16(__half* img, const float* __restrict__ W, int OUT, int IN, int OUTP, int INP,
                                          const float* __restrict__ colscale = nullptr) {
    const int n = (INP / 8) * OUTP * 8;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int e = i & 7, r = (i >> 3) % OUTP, c = (i >> 3) / OUTP, in = c * 8 + e;
        float v = 0.f;
        if (r < OUT && in < IN) { v = __ldg(W + (size_t)r * IN + in); if (colscale) v *= __ldg(colscale + in); }
        img[i] = __float2half_rn(v);
    }
}
__device__ __forceinline__ void stage_b32(float* dst, const float* __restrict__ b, int n, int np) {
    for (int i = threadIdx.x; i < np; i += blockDim.x) dst[i] = (i < n) ? __ldg(b + i) : 0.f;
}
// generic-proxy smem writes + TMEM reads of all threads ordered before the MMAs the elected thread issues next
__device__ __forceinline__ void sync_to_mma() {
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
}
struct MmaBar {
    uint64_t* bar;
    uint32_t parity;
    __device__ __forceinline__ void commit() { umma_commit(bar); }
    __device__ __forceinline__ void wait() { mbar_wait(bar, parity); parity ^= 1; tc_fence_after(); }
};

// accumulator row (64 columns) -> +bias -> ReLU -> fp16 tile; returns the activity mask
__device__ __forceinline__ uint64_t epi_relu64(uint32_t taddr, const float* __restrict__ bias, uint8_t* tile, int row) {
    uint64_t mask = 0;
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            v[i] = fmaxf(v[i] + bias[c0 + i], 0.f);
            mask |= (v[i] > 0.f) ? (1ull << (c0 + i)) : 0ull;
        }
        tile_store8(tile, c0 / 8, row, v);
        tile_store8(tile, c0 / 8 + 1, row, v + 8);
    }
    return mask;
}

// warp reduce-scatter of N per-lane values (N = 64): afterwards v[0], v[1] hold the warp sums of
// features f0 + {0,1}, f0 = 32*b4 + 16*b3 + 8*b2 + 4*b1 + 2*b0 of the lane id bits
template <int N>
__device__ __forceinline__ void warp_reduce_scatter(float (&v)[N], int lane) {
#pragma unroll
    for (int o = 16, n = N / 2; o >= 1; o >>= 1, n >>= 1) {
        const bool hi = lane & o;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const float send = hi ? v[i] : v[i + n];
            const float keep = hi ? v[i + n] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
}
__device__ __forceinline__ int scatter_base(int lane, int n) {  // first feature owned by `lane` after the scatter of n values
    int f = 0, h = n / 2;
    for (int o = 16; o >= 1; o >>= 1, h >>= 1) f += (lane & o) ? h : 0;
    return f;
}
// masked hidden gradient: accumulator row (64 cols) * relu mask -> fp16 tile, bias-grad partial sums
__device__ __forceinline__ void epi_grad64(uint32_t taddr, uint64_t mask, uint8_t* tile, int row, int lane, float (&dbacc)[2]) {
    float g[64];
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) g[c0 + i] = ((mask >> (c0 + i)) & 1ull) ? v[i] : 0.f;
        tile_store8(tile, c0 / 8, row, g + c0);
        tile_store8(tile, c0 / 8 + 1, row, g + c0 + 8);
    }
    warp_reduce_scatter<64>(g, lane);
    dbacc[0] += g[0]; dbacc[1] += g[1];
}
// 16-feature gradient row -> tile (2 chunks) + bias partial (lane keeps 1 value when lane is even after 4 scatter steps)
__device__ __forceinline__ void grad16_store(float (&g)[16], uint8_t* tile, int row, int lane, float& dbacc) {
    tile_store8(tile, 0, row, g);
    tile_store8(tile, 1, row, g + 8);
#pragma unroll
    for (int o = 16, n = 8; o >= 2; o >>= 1, n >>= 1) {
        const bool hi = lane & o;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const float send = hi ? g[i] : g[i + n];
            const float keep = hi ? g[i + n] : g[i];
            g[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    dbacc += g[0] + __shfl_xor_sync(0xffffffffu, g[0], 1);  // feature 8*b4 + 4*b3 + 2*b2 + b1 (both lanes of a pair hold it)
}
// ---- column-split epilogues: a row's columns are divided among NCG threads (warps w, w+4, w+8, ... share the
// TMEM lane quadrant w%4), which multiplies the warps per SM without more TMEM or shared memory ----------------
// 16 accumulator columns -> +bias -> ReLU -> 2 tile chunks; returns the 16-bit activity mask
__device__ __forceinline__ uint32_t epi_relu16(uint32_t taddr, const float* __restrict__ bias, uint8_t* tile2, int row) {
    float v[16];
    tmem_ld16(taddr, v);
    uint32_t mask = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        v[i] = fmaxf(v[i] + bias[i], 0.f);
        mask |= (v[i] > 0.f) ? (1u << i) : 0u;
    }
    tile_store8(tile2, 0, row, v);
    tile_store8(tile2, 1, row, v + 8);
    return mask;
}
// 16 masked gradient columns -> 2 tile chunks + bias-gradient partial (feature 8*b4+4*b3+2*b2+b1 of the 16, on every lane pair)
__device__ __forceinline__ void epi_grad16(uint32_t taddr, uint32_t mask, uint8_t* tile2, int row, int lane, float& dbacc) {
    float v[16];
    tmem_ld16(taddr, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = ((mask >> i) & 1u) ? v[i] : 0.f;
    grad16_store(v, tile2, row, lane, dbacc);
}
// 16 masked gradient columns -> 2 tile chunks (bias gradient taken by the tensor core, see the ones tiles)
__device__ __forceinline__ void epi_grad16_nb(uint32_t taddr, uint32_t mask, uint8_t* tile2, int row) {
    float v[16];
    tmem_ld16(taddr, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = ((mask >> i) & 1u) ? v[i] : 0.f;
    tile_store8(tile2, 0, row, v);
    tile_store8(tile2, 1, row, v + 8);
}
// ---- per-CTA partial weight gradients -> gradients -------------------------------------------------------------------
// 148 CTAs accumulating the same ~100 KB of weight gradients with red.add serialise in the L2 atomic units (measured: 8 % of
// the fused backward).  With a workspace every CTA stores its partial sums privately and this kernel adds the slices of the
// CTAs that had at least one tile to the gradient tensors.
struct WsSegs { int n; int off[6]; int len[6]; float* dst[6]; };
#define WS_GROUPS 16   // blockIdx.y: each thread sums every 16th slice (all its loads independent) and adds once
static __global__ void __launch_bounds__(256) ws_reduce_kernel(const float* __restrict__ ws, int nblocks, int64_t M, const int64_t* __restrict__ m_dev,
                                                               int total, WsSegs segs) {
    if (m_dev) M = min(M, __ldg(m_dev));
    const int64_t ntiles = (M + 127) / 128;
    const int nact = (int)(ntiles < nblocks ? ntiles : nblocks);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    float* dst = nullptr;
#pragma unroll
    for (int s = 0; s < 6; ++s)
        if (s < segs.n && i >= segs.off[s] && i < segs.off[s] + segs.len[s] && segs.dst[s]) dst = segs.dst[s] + (i - segs.off[s]);
    if (!dst) return;
    float a0 = 0.f, a1 = 0.f;
    int b = blockIdx.y;
    for (; b + WS_GROUPS < nact; b += 2 * WS_GROUPS) { a0 += ws[(size_t)b * total + i]; a1 += ws[(size_t)(b + WS_GROUPS) * total + i]; }
    if (b < nact) a0 += ws[(size_t)b * total + i];
    if (blockIdx.y < nact) red_add_f32(dst, a0 + a1);
}

// flush columns [c0, c0+16) of a dW accumulator row.  plain: the destination is this CTA's private partial buffer
// (ordinary 16-byte stores, summed over CTAs by a reduce kernel) instead of the shared gradient (red.add).
__device__ __forceinline__ void flush_dw16(uint32_t taddr, float* __restrict__ gW, int row, int OUT, int IN, int c0, float inv_scale,
                                           bool plain = false) {
    float v[16];
    tmem_ld16(taddr + c0, v);
    if (row < OUT) {
        float* dst = gW + (size_t)row * IN + c0;
        if (!(IN & 3) && !(reinterpret_cast<uintptr_t>(gW) & 15)) {   // 16-byte vector accesses
#pragma unroll
            for (int i = 0; i < 16; i += 4)
                if (c0 + i < IN) {
                    if (plain) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i] * inv_scale, v[i + 1] * inv_scale, v[i + 2] * inv_scale, v[i + 3] * inv_scale);
                    else red_add_f32x4(dst + i, v[i] * inv_scale, v[i + 1] * inv_scale, v[i + 2] * inv_scale, v[i + 3] * inv_scale);
                }
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (c0 + i < IN) {
                    if (plain) dst[i] = v[i] * inv_scale;
                    else red_add_f32(dst + i, v[i] * inv_scale);
                }
        }
    }
}

// flush a dW accumulator [rows(lane) x cols] from TMEM to global with atomics
__device__ __forceinline__ void flush_dw(uint32_t taddr, float* __restrict__ gW, int row, int OUT, int IN, int ncols, float inv_scale) {
    for (int c0 = 0; c0 < ncols; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
        if (row < OUT) {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (c0 + i < IN) red_add_f32(gW + (size_t)row * IN + c0 + i, v[i] * inv_scale);
        }
    }
}

// this thread's feature row -> X tile (float4 global loads: IN is a multiple of 4 for every supported grid)
__device__ __forceinline__ void stage_x(uint8_t* tile, int row, const float* __restrict__ a, const float* __restrict__ b,
                                        const float* __restrict__ lodw, int IN, int nchunks, int64_t m) {
    const float4* a4 = reinterpret_cast<const float4*>(a + m * IN);
    const float4* b4 = b ? reinterpret_cast<const float4*>(b + m * IN) : nullptr;
    const float4* w4 = lodw ? reinterpret_cast<const float4*>(lodw) : nullptr;
    for (int c = 0; c < nchunks; ++c) {
        float v[8];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int q = 2 * c + h;   // float4 index
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (4 * q < IN) {
                x = __ldg(a4 + q);
                if (b4) { const float4 y = __ldg(b4 + q); x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w; }
                if (w4) { const float4 w = __ldg(w4 + q); x.x *= w.x; x.y *= w.y; x.z *= w.z; x.w *= w.w; }
            }
            v[4 * h] = x.x; v[4 * h + 1] = x.y; v[4 * h + 2] = x.z; v[4 * h + 3] = x.w;
        }
        tile_store8(tile, c, row, v);
    }
}
// L2 prefetch of the chunks of row m of a later tile (f32-row kernels without spare shared memory)
__device__ __forceinline__ void prefetch_x_l2(const float* __restrict__ a, const float* __restrict__ b, int IN, int nchunks, int64_t m,
                                              int cg, int ncg) {
    for (int c = cg; c < nchunks; c += ncg) {
        if (8 * c < IN) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(a + m * IN + 8 * c));
            if (b) asm volatile("prefetch.global.L2 [%0];" ::"l"(b + m * IN + 8 * c));
        }
    }
}

// ---- asynchronous X-tile prefetch (column-split kernels) ------------------------------------------------------------
// Thread (row, cg) converts the float4 quads q = cg, cg + NCG, ... of its row.  The quads of the NEXT tile are copied
// with cp.async into private 16-byte slots slots[(2k + {0:a, 1:b}) * nthreads + tid] while the current tile is being
// processed -- no registers are held and no other thread touches the slots, so the only synchronisation is the
// thread's own cp.async.wait_all.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Coalesced variant.  A lane-per-row float4 access touches 32 different 128-byte lines per warp instruction and costs 32 LSU
// cycles (measured: 3.4 k cycles per 128 x 48 tile pair); here consecutive threads copy consecutive quads of the tile's
// contiguous [128][IN] block, 4 lines per instruction, into slots[xpfc_slot(row, q)] (array b: + 128 * IN/4 slots), and
// thread (row, cg) later reads its quads q = cg + NCG k from there.  The slot order is the block's own (row-major) with the
// quads of row r rotated by r & 7: at most 2-way bank conflicts for the lane-per-quad writes of cp.async AND the lane-per-row
// reads (measured: a quad-major layout made every cp.async a 12-way conflict, 4 k cycles per tile).  The consumer reads slots
// written by other threads: call cp_async_wait_all() before the block barrier that precedes xpfc_consume.
__device__ __forceinline__ int xpfc_slot(int r, int q, int nq) {
    int t = q + (r & 7);
    while (t >= nq) t -= nq;
    return r * nq + t;
}
template <int MAXK>
__device__ __forceinline__ void xpfc_issue(float4* slots, const float* __restrict__ a, const float* __restrict__ b, int IN, int64_t row0,
                                           int64_t M) {
    const int nt = blockDim.x, tid = threadIdx.x, nq = IN >> 2, total = 128 * nq;
#pragma unroll
    for (int k = 0; k < MAXK; ++k) {
        const int g = tid + nt * k;
        if (g < total) {
            const int r = g / nq, q = g - r * nq;
            const int64_t rs = min(row0 + r, M - 1);
            const int sl = xpfc_slot(r, q, nq);
            cp_async16(slots + sl, a + rs * IN + 4 * q);
            if (b) cp_async16(slots + total + sl, b + rs * IN + 4 * q);
        }
    }
    cp_async_commit();
}
template <int NCG, int MAXK>
__device__ __forceinline__ void xpfc_consume(const float4* slots, bool has_b, int IN, int INP, uint8_t* tile, int row, int cg) {
    const int nq = IN >> 2, total = 128 * nq;
#pragma unroll
    for (int k = 0; k < MAXK; ++k) {
        const int q = cg + NCG * k;
        if (4 * q < INP) {
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (4 * q < IN) {
                const int sl = xpfc_slot(row, q, nq);
                x = slots[sl];
                if (has_b) { const float4 y = slots[total + sl]; x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w; }
            }
            uint2 u;
            u.x = pack_h2(x.x, x.y); u.y = pack_h2(x.z, x.w);
            *reinterpret_cast<uint2*>(tile + (q >> 1) * TCH + row * 16 + (q & 1) * 8) = u;
        }
    }
}
// direct (register) variant of the same coalesced mapping for kernels without spare shared memory: thread t loads quads
// t, t + nthreads, ... of the tile block and writes them into the fp16 image itself
__device__ __forceinline__ void stage_x_coalesced(uint8_t* tile, const float* __restrict__ a, const float* __restrict__ b, int IN, int INP,
                                                  int64_t row0, int64_t M) {
    const int nt = blockDim.x, nq = IN >> 2, nqp = INP >> 2;
    for (int g = threadIdx.x; g < 128 * nqp; g += nt) {
        const int r = g / nqp, q = g - r * nqp;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < nq) {
            const int64_t rs = min(row0 + r, M - 1);
            x = __ldg(reinterpret_cast<const float4*>(a + rs * IN) + q);
            if (b) { const float4 y = __ldg(reinterpret_cast<const float4*>(b + rs * IN) + q); x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w; }
        }
        uint2 u;
        u.x = pack_h2(x.x, x.y); u.y = pack_h2(x.z, x.w);
        *reinterpret_cast<uint2*>(tile + (q >> 1) * TCH + r * 16 + (q & 1) * 8) = u;
    }
}

// X (fp16 operand image tile, `bytes` long) += D, or X = A + D when A is given: the panoptic heads read feats + delta feats
// (pc_nerf/panoptic_delta_nef.py:226, a half-precision add under the reference's autocast as well)
__device__ __forceinline__ void tile_add16(uint8_t* X, const uint8_t* A, const uint8_t* D, int bytes) {
    for (int i = threadIdx.x; i < bytes / 16; i += blockDim.x) {
        uint4 a = reinterpret_cast<const uint4*>(A ? A : X)[i];
        if (D) {
            const uint4 d = reinterpret_cast<const uint4*>(D)[i];
            __half2* ah = reinterpret_cast<__half2*>(&a);
            const __half2* dh = reinterpret_cast<const __half2*>(&d);
#pragma unroll
            for (int k = 0; k < 4; ++k) ah[k] = __hadd2(ah[k], dh[k]);
        }
        reinterpret_cast<uint4*>(X)[i] = a;
    }
}

// ---- dX tile -> global through shared memory ------------------------------------------------------------------------
// A lane-per-row float4 store touches 32 lines per warp instruction: the 48 store instructions of a 128 x 48 dX tile keep
// the LSU busy for ~1.5 k cycles and everything queued behind them (the next tile's shared-memory traffic) waits.  The tile
// is staged in shared memory instead (row stride IN + 4 floats: conflict free for the lane-per-row writes) and written out
// by all threads with consecutive threads on consecutive 16-byte quads of the [128][IN] block (4 lines per instruction).
__device__ __forceinline__ int dx_ld(int IN) { return IN + 4; }
__device__ __forceinline__ void dx_stage16(uint32_t taddr, float* __restrict__ stage, int row, int IN, int c16, float inv_scale) {
    float v[16];
    tmem_ld16(taddr + c16, v);
    float* d = stage + row * dx_ld(IN) + c16;
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (c16 + 4 * q < IN)
            reinterpret_cast<float4*>(d)[q] = make_float4(v[4 * q] * inv_scale, v[4 * q + 1] * inv_scale, v[4 * q + 2] * inv_scale, v[4 * q + 3] * inv_scale);
}
__device__ __forceinline__ void dx_copy_out(const float* __restrict__ stage, float* __restrict__ dst, int IN, int64_t row0, int64_t M) {
    const unsigned nq = (unsigned)IN >> 2, total = 128u * nq;
    for (unsigned g = threadIdx.x; g < total; g += blockDim.x) {
        const unsigned r = g / nq, q = g - r * nq;
        if (row0 + r < M)
            reinterpret_cast<float4*>(dst + (row0 + r) * IN)[q] = *reinterpret_cast<const float4*>(stage + r * dx_ld(IN) + 4 * q);
    }
}

// dX row (TMEM) -> global, float4 stores
__device__ __forceinline__ void store_dx(uint32_t taddr, float* __restrict__ dst, const float* __restrict__ lodw, int IN,
                                         int INP, float inv_scale, bool valid) {
    for (int c0 = 0; c0 < INP; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
        if (valid) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (c0 + 4 * q < IN) {
                    float4 w = lodw ? __ldg(reinterpret_cast<const float4*>(lodw + c0) + q) : make_float4(1.f, 1.f, 1.f, 1.f);
                    float4 o = make_float4(v[4 * q] * inv_scale * w.x, v[4 * q + 1] * inv_scale * w.y,
                                           v[4 * q + 2] * inv_scale * w.z, v[4 * q + 3] * inv_scale * w.w);
                    reinterpret_cast<float4*>(dst + c0)[q] = o;
                }
            }
        }
    }
}
// color-decoder input row [y16 | PE(-d) | 0 pad] -> 6 chunks
__device__ __forceinline__ void stage_cin(uint8_t* tile, int row, const float (&y)[16], const float* pe) {
    float v[48];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = y[k];
#pragma unroll
    for (int k = 0; k < PE_DIM; ++k) v[16 + k] = pe[k];
#pragma unroll
    for (int k = CIN; k < 48; ++k) v[k] = 0.f;
#pragma unroll
    for (int c = 0; c < 6; ++c) tile_store8(tile, c, row, v + 8 * c);
}

struct PanTcLayout {
    int INP, nXc, CsP, CiP, nGi;
    int oGs, oX, oHs, oH1, oH2, oGi, oWs1, oWs2, oWi1, oWi2, oWi3, oBias, oStage, total;
};
__host__ __device__ inline PanTcLayout pan_tc_layout(int IN, int Cs, int Ci, bool bwd) {
    PanTcLayout l;
    l.INP = (IN + 15) & ~15; l.nXc = l.INP / 8;
    l.CsP = Cs > 0 ? ((Cs + 15) & ~15) : 16;
    l.CiP = Ci > 0 ? ((Ci + 15) & ~15) : 16;
    l.nGi = l.CiP / 8;
    int o = 0;
    l.oGs = o; o += bwd ? (l.CsP / 8) * TCH : 0;   // semantic logit gradients: CsP <= 32 features
    l.oX = o; o += 8 * TCH;
    l.oHs = o; o += 8 * TCH;
    l.oH1 = o; o += 8 * TCH;
    l.oH2 = o; o += bwd ? 8 * TCH : 0;
    l.oGi = o; o += bwd ? l.nGi * TCH : 0;
    l.oWs1 = o; o += l.nXc * 64 * 16;
    l.oWs2 = o; o += 8 * l.CsP * 16;
    l.oWi1 = o; o += l.nXc * 64 * 16;
    l.oWi2 = o; o += 8 * 64 * 16;
    l.oWi3 = o; o += 8 * l.CiP * 16;
    l.oBias = o; o += (64 + l.CsP + 64 + 64 + l.CiP) * 4;
    o = (o + 15) & ~15;
    l.oStage = o; o += bwd ? 4 * 2 * 32 * 33 * 4 : 0;   // per-warp transpose buffers for the coalesced prob / grad loads
    if (bwd) {  // MN-major A operands read 16 chunks from their base (the second dWi3 block starts 16 chunks into Gi)
        const int need = l.oGi + (l.nGi > 16 ? 32 : 16) * TCH;
        if (o < need) o = need;
    }
    l.total = o;
    return l;
}
__device__ __forceinline__ void pan_tc_stage(uint8_t* sm, const PanTcLayout& l, const PanParams& p, int IN, int Cs, int Ci) {
    float* b = reinterpret_cast<float*>(sm + l.oBias);
    if (Cs > 0) {
        stage_w16(reinterpret_cast<__half*>(sm + l.oWs1), p.Ws1, 64, IN, 64, l.INP);
        stage_w16(reinterpret_cast<__half*>(sm + l.oWs2), p.Ws2, Cs, 64, l.CsP, 64);
        stage_b32(b, p.bs1, 64, 64); stage_b32(b + 64, p.bs2, Cs, l.CsP);
    }
    if (Ci > 0) {
        stage_w16(reinterpret_cast<__half*>(sm + l.oWi1), p.Wi1, 64, IN, 64, l.INP);
        stage_w16(reinterpret_cast<__half*>(sm + l.oWi2), p.Wi2, 64, 64, 64, 64);
        stage_w16(reinterpret_cast<__half*>(sm + l.oWi3), p.Wi3, Ci, 64, l.CiP, 64);
        stage_b32(b + 64 + l.CsP, p.bi1, 64, 64); stage_b32(b + 128 + l.CsP, p.bi2, 64, 64);
        stage_b32(b + 192 + l.CsP, p.bi3, Ci, l.CiP);
    }
}

