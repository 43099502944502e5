// Panoptic point-map export on the device (the reference's utils/render_map.py, which evaluates the nef on the octree cells).
//
//   pag_map_cell_points      sub-cell centres of the occupied leaf cells: cell c, sub-point s = (ix*k + iy)*k + iz ->
//                            xyz[c*k^3 + s] = (2*(p*k + i) + 1) / (k << level) - 1 per axis.  Numerator and denominator are exact
//                            integers in fp32 and the division is IEEE (__fdiv_rn), so the CPU oracle matches bit for bit.
//   pag_map_instance_stats   per-instance count, coordinate / colour sums (float64), bounding box and semantic votes of the labelled
//                            points.  Each CTA accumulates into shared memory and flushes one global atomic per non-empty slot.
//                            bbox min / max use the order-preserving integer atomics on the float bits (pag_atomic_min_f32).
#include "common.cuh"

#define MAP_STATS_BLOCK 256

__global__ void __launch_bounds__(256) map_cell_points_kernel(const int16_t* __restrict__ cells, int64_t n, int level, int k,
                                                              float* __restrict__ xyz) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int kk = k * k;
    const int64_t c = t / (kk * k);
    const int s = (int)(t - c * (kk * k));
    const int i3[3] = {s / kk, (s / k) % k, s % k};
    const float den = (float)(k << level);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int p = cells[3 * c + a];
        xyz[3 * t + a] = __fsub_rn(__fdiv_rn((float)(2 * (p * k + i3[a]) + 1), den), 1.0f);
    }
}

// float min / max through integer atomics: for v >= 0 the float order is the signed order of the bits, for v < 0 the reversed
// unsigned order; valid for any non-NaN contents of *addr (callers start from +inf / -inf)
__device__ __forceinline__ void pag_atomic_min_f32(float* addr, float v) {
    if (v >= 0.f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void pag_atomic_max_f32(float* addr, float v) {
    if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

struct MapStatsLayout { int count, sum_xyz, sum_rgb, bmin, bmax, votes, total; };     // byte offsets in shared memory
__host__ __device__ inline MapStatsLayout map_stats_layout(int Cs, int Ci) {
    MapStatsLayout l; int o = 0;
    l.sum_xyz = o; o += Ci * 3 * 8; l.sum_rgb = o; o += Ci * 3 * 8;
    l.count = o; o += Ci * 4; l.bmin = o; o += Ci * 3 * 4; l.bmax = o; o += Ci * 3 * 4; l.votes = o; o += Ci * Cs * 4;
    l.total = o;
    return l;
}

__global__ void __launch_bounds__(MAP_STATS_BLOCK) map_instance_stats_kernel(
        const float* __restrict__ xyz, const float* __restrict__ rgb, const int64_t* __restrict__ sem, const int64_t* __restrict__ inst,
        int64_t P, int Cs, int Ci, uint32_t thing_mask, long long* __restrict__ count, double* __restrict__ sum_xyz,
        double* __restrict__ sum_rgb, int64_t* __restrict__ votes, float* __restrict__ bbox_min, float* __restrict__ bbox_max,
        long long* __restrict__ errors) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const MapStatsLayout l = map_stats_layout(Cs, Ci);
    double* s_xyz = reinterpret_cast<double*>(smem_raw + l.sum_xyz);
    double* s_rgb = reinterpret_cast<double*>(smem_raw + l.sum_rgb);
    unsigned int* s_cnt = reinterpret_cast<unsigned int*>(smem_raw + l.count);
    float* s_min = reinterpret_cast<float*>(smem_raw + l.bmin);
    float* s_max = reinterpret_cast<float*>(smem_raw + l.bmax);
    unsigned int* s_votes = reinterpret_cast<unsigned int*>(smem_raw + l.votes);
    for (int i = threadIdx.x; i < 3 * Ci; i += blockDim.x) { s_xyz[i] = 0.0; s_rgb[i] = 0.0; s_min[i] = INFINITY; s_max[i] = -INFINITY; }
    for (int i = threadIdx.x; i < Ci; i += blockDim.x) s_cnt[i] = 0u;
    for (int i = threadIdx.x; i < Ci * Cs; i += blockDim.x) s_votes[i] = 0u;
    __syncthreads();
    unsigned n_bad = 0;
    for (int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; m < P; m += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = sem[m], q = inst[m];
        if (c < 0 || c >= Cs || q < 0 || q >= Ci) { ++n_bad; continue; }
        if (!((thing_mask >> c) & 1u)) continue;
        const int i = (int)q;
        atomicAdd(s_cnt + i, 1u);
        atomicAdd(s_votes + i * Cs + (int)c, 1u);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float x = xyz[3 * m + a];
            atomicAdd(s_xyz + 3 * i + a, (double)x);
            atomicAdd(s_rgb + 3 * i + a, (double)rgb[3 * m + a]);
            pag_atomic_min_f32(s_min + 3 * i + a, x);
            pag_atomic_max_f32(s_max + 3 * i + a, x);
        }
    }
    for (int o = 16; o > 0; o >>= 1) n_bad += __shfl_xor_sync(0xffffffffu, n_bad, o);
    if ((threadIdx.x & 31) == 0 && n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(errors), (unsigned long long)n_bad);
    __syncthreads();
    for (int i = threadIdx.x; i < Ci; i += blockDim.x) {
        const unsigned int n = s_cnt[i];
        if (!n) continue;
        atomicAdd(reinterpret_cast<unsigned long long*>(count + i), (unsigned long long)n);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            atomicAdd(sum_xyz + 3 * i + a, s_xyz[3 * i + a]);
            atomicAdd(sum_rgb + 3 * i + a, s_rgb[3 * i + a]);
            pag_atomic_min_f32(bbox_min + 3 * i + a, s_min[3 * i + a]);
            pag_atomic_max_f32(bbox_max + 3 * i + a, s_max[3 * i + a]);
        }
        for (int c = 0; c < Cs; ++c) {
            const unsigned int v = s_votes[i * Cs + c];
            if (v) atomicAdd(reinterpret_cast<unsigned long long*>(votes + (int64_t)i * Cs + c), (unsigned long long)v);
        }
    }
}

static int map_num_sms() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

extern "C" {

int pag_map_cell_points(const int16_t* cells, int64_t C, int level, int k, float* xyz, void* stream) {
    if (C < 0 || level < 0 || level > 15 || k < 1 || k > 8) return PAG_ERR_ARG;
    if (C == 0) return PAG_OK;
    if (!cells || !xyz) return PAG_ERR_ARG;
    const int64_t n = C * k * k * k;
    map_cell_points_kernel<<<pag_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(cells, n, level, k, xyz);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

int pag_map_instance_stats(const float* xyz, const float* rgb, const int64_t* semantic, const int64_t* instance, int64_t P, int Cs, int Ci,
                           uint32_t thing_mask, int64_t* count, double* sum_xyz, double* sum_rgb, int64_t* votes, float* bbox_min,
                           float* bbox_max, int64_t* errors, void* stream) {
    if (P < 0 || Cs < 1 || Cs > 32 || Ci < 1) return PAG_ERR_ARG;
    const size_t bytes = (size_t)map_stats_layout(Cs, Ci).total;
    if (bytes > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    if (P == 0) return PAG_OK;
    if (!xyz || !rgb || !semantic || !instance || !count || !sum_xyz || !sum_rgb || !votes || !bbox_min || !bbox_max || !errors)
        return PAG_ERR_ARG;
    if (bytes > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(map_instance_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return (int)e;
    }
    // a few CTAs per SM: every CTA flushes its non-empty slots once, so fewer, longer-lived CTAs mean fewer global atomics
    const int64_t want = pag_grid(P, MAP_STATS_BLOCK);
    const int64_t cap = 4 * (int64_t)map_num_sms();
    const int grid = (int)(want < cap ? want : cap);
    map_instance_stats_kernel<<<grid, MAP_STATS_BLOCK, bytes, (cudaStream_t)stream>>>(
        xyz, rgb, semantic, instance, P, Cs, Ci, thing_mask, reinterpret_cast<long long*>(count), sum_xyz, sum_rgb, votes, bbox_min,
        bbox_max, reinterpret_cast<long long*>(errors));
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

}  // extern "C"
