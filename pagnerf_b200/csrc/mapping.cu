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
#define MAP_CC_MAX_POINTS (1ll << 30)

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

// Both statistics kernels read a label lab[m] per point (an instance, or an object of pag_map_components).  With unlabelled_ok a
// label of -1 means "no object" and is skipped silently; any other label outside [0, Ci), or a class outside [0, Cs), is skipped and
// counted in errors (nullable).  inst_out (nullable) receives, per label, inst_src of one of its points.
__global__ void __launch_bounds__(MAP_STATS_BLOCK) map_instance_stats_kernel(
        const float* __restrict__ xyz, const float* __restrict__ rgb, const int64_t* __restrict__ sem, const int64_t* __restrict__ lab,
        int64_t P, int Cs, int Ci, uint32_t thing_mask, int unlabelled_ok, const int64_t* __restrict__ inst_src,
        int64_t* __restrict__ inst_out, long long* __restrict__ count, double* __restrict__ sum_xyz, double* __restrict__ sum_rgb,
        int64_t* __restrict__ votes, float* __restrict__ bbox_min, float* __restrict__ bbox_max, long long* __restrict__ errors) {
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
        const int64_t c = sem[m], q = lab[m];
        if (q == -1 && unlabelled_ok) continue;
        if (c < 0 || c >= Cs || q < 0 || q >= Ci) { ++n_bad; continue; }
        if (!((thing_mask >> c) & 1u)) continue;
        const int i = (int)q;
        if (inst_out && (m == 0 || lab[m - 1] != q)) inst_out[i] = inst_src[m];
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
    if ((threadIdx.x & 31) == 0 && n_bad && errors) atomicAdd(reinterpret_cast<unsigned long long*>(errors), (unsigned long long)n_bad);
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

// The same statistics accumulated straight into global memory, for label counts whose slots do not fit in shared memory.  Each
// warp takes 32 consecutive points and reduces every run of equal labels (a segmented shuffle scan) before one set of atomics per
// run: map points arrive in Morton cell order, so neighbouring lanes mostly share a label.
__global__ void __launch_bounds__(MAP_STATS_BLOCK) map_instance_stats_global_kernel(
        const float* __restrict__ xyz, const float* __restrict__ rgb, const int64_t* __restrict__ sem, const int64_t* __restrict__ lab,
        int64_t P, int Cs, int Ci, uint32_t thing_mask, int unlabelled_ok, const int64_t* __restrict__ inst_src,
        int64_t* __restrict__ inst_out, long long* __restrict__ count, double* __restrict__ sum_xyz, double* __restrict__ sum_rgb,
        int64_t* __restrict__ votes, float* __restrict__ bbox_min, float* __restrict__ bbox_max, long long* __restrict__ errors) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lanes_le = FULL >> (31 - lane);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    unsigned n_bad = 0;
    for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31)); base < P; base += nwarps * 32) {
        const int64_t m = base + lane;
        long long q = -1;      // -1: this lane adds nothing
        int c = 0;
        if (m < P) {
            const int64_t c64 = sem[m], q64 = lab[m];
            const bool unlabelled = q64 == -1 && unlabelled_ok;
            const bool bad = !unlabelled && (c64 < 0 || c64 >= Cs || q64 < 0 || q64 >= Ci);
            n_bad += bad;
            if (!unlabelled && !bad && ((thing_mask >> c64) & 1u)) {
                q = q64;
                c = (int)c64;
            }
        }
        double sx[3] = {0.0, 0.0, 0.0}, sr[3] = {0.0, 0.0, 0.0};
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        if (q >= 0) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                lo[a] = hi[a] = xyz[3 * m + a];
                sx[a] = (double)lo[a];
                sr[a] = (double)rgb[3 * m + a];
            }
        }
        const long long qp = __shfl_up_sync(FULL, q, 1), qn = __shfl_down_sync(FULL, q, 1);
        const bool head = lane == 0 || qp != q, tail = lane == 31 || qn != q;
        const int h = 31 - __clz(__ballot_sync(FULL, head) & lanes_le);          // first lane of this lane's run
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const bool take = lane - o >= h;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double ux = __shfl_up_sync(FULL, sx[a], o), ur = __shfl_up_sync(FULL, sr[a], o);
                const float ul = __shfl_up_sync(FULL, lo[a], o), uh = __shfl_up_sync(FULL, hi[a], o);
                if (take) { sx[a] += ux; sr[a] += ur; lo[a] = fminf(lo[a], ul); hi[a] = fmaxf(hi[a], uh); }
            }
        }
        if (tail && q >= 0) {      // the run's last lane holds its totals
            atomicAdd(reinterpret_cast<unsigned long long*>(count + q), (unsigned long long)(lane - h + 1));
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                atomicAdd(sum_xyz + 3 * q + a, sx[a]);
                atomicAdd(sum_rgb + 3 * q + a, sr[a]);
                pag_atomic_min_f32(bbox_min + 3 * q + a, lo[a]);
                pag_atomic_max_f32(bbox_max + 3 * q + a, hi[a]);
            }
            if (inst_out) inst_out[q] = inst_src[m];
        }
        // votes: runs of equal (label, class) inside the label's run; their lengths are the counts
        const int cp = __shfl_up_sync(FULL, c, 1), cn = __shfl_down_sync(FULL, c, 1);
        const bool head2 = head || cp != c, tail2 = tail || cn != c;
        const int h2 = 31 - __clz(__ballot_sync(FULL, head2) & lanes_le);
        if (tail2 && q >= 0) atomicAdd(reinterpret_cast<unsigned long long*>(votes + q * Cs + c), (unsigned long long)(lane - h2 + 1));
    }
    for (int o = 16; o > 0; o >>= 1) n_bad += __shfl_xor_sync(FULL, n_bad, o);
    if (lane == 0 && n_bad && errors) atomicAdd(reinterpret_cast<unsigned long long*>(errors), (unsigned long long)n_bad);
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

// ---- connected components of the map (pag_map_components) ----
// Lattice index j per axis in [0, D), D = k << level, packed 21 bits per axis (D <= 2^18); hash key = packed + 1 (0 = empty slot).
#define MAP_CC_BLOCK 256
#define MAP_CC_SCAN_BLOCK 1024
#define MAP_CC_AXIS_BITS 21

struct CcWorkspace {      // layout in pag_map_components_workspace's comment (include/pagnerf_b200.h)
    unsigned long long* table_key;
    long long* key;       // per point: its hash key (0 = off the lattice); after the union step, the rank of each root
    int64_t* boff;        // exclusive scan of bsum, nb + 1 entries
    uint32_t* table_val;
    int* parent;          // -1 for inactive points
    int* count;
    int* bsum;
};

static int64_t cc_blocks(int64_t P) { return (P + MAP_CC_SCAN_BLOCK - 1) / MAP_CC_SCAN_BLOCK; }

static int64_t cc_workspace_bytes(int64_t P) {
    const int64_t C = pag_hash_slots(P), nb = cc_blocks(P);
    return 12 * C + 16 * P + 8 * (nb + 1) + 4 * nb;
}

static CcWorkspace cc_workspace(void* ws, int64_t P) {
    const int64_t C = pag_hash_slots(P), nb = cc_blocks(P);
    CcWorkspace w;
    w.table_key = reinterpret_cast<unsigned long long*>(ws);
    w.key = reinterpret_cast<long long*>(w.table_key + C);
    w.boff = reinterpret_cast<int64_t*>(w.key + P);
    w.table_val = reinterpret_cast<uint32_t*>(w.boff + nb + 1);
    w.parent = reinterpret_cast<int*>(w.table_val + C);
    w.count = w.parent + P;
    w.bsum = w.count + P;
    return w;
}

// lattice index of coordinate x, or -1 when x is not bit for bit fl(fl((2j+1)/D) - 1) for any j in [0, D).  For a lattice point
// |x - ((2j+1)/D - 1)| <= 2^-23 + 2^-25 (one rounding of a value below 2, one of the subtraction), so (x+1) D / 2 - 1/2 lies
// within D * 2^-24 * 1.25 <= 0.02 of j and rounding recovers it; the exact formula then decides.
__device__ __forceinline__ int cc_lattice_index(float x, int D) {
    const double t = ((double)x + 1.0) * (double)D * 0.5 - 0.5;
    if (!(t > -0.5 && t < (double)D - 0.5)) return -1;
    const int j = __double2int_rn(t);
    const float y = __fsub_rn(__fdiv_rn((float)(2 * j + 1), (float)D), 1.0f);
    return __float_as_uint(y) == __float_as_uint(x) ? j : -1;
}

__device__ __forceinline__ unsigned long long cc_key(int jx, int jy, int jz) {
    return (((unsigned long long)jx << (2 * MAP_CC_AXIS_BITS)) | ((unsigned long long)jy << MAP_CC_AXIS_BITS) | (unsigned long long)jz) + 1ull;
}

// lattice recovery of point i and its insert into the table (key -> point index), shared by the components and the map index.
// Returns the point's hash key, 0 when it is off the lattice (*off); *dup: an earlier insert already holds its lattice index.
__device__ __forceinline__ unsigned long long cc_insert_point(const float* __restrict__ xyz, int64_t i, int D,
                                                              unsigned long long* __restrict__ table_key, uint32_t* __restrict__ table_val,
                                                              uint32_t C, bool* off, bool* dup) {
    int j[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) j[a] = cc_lattice_index(xyz[3 * i + a], D);
    *off = j[0] < 0 || j[1] < 0 || j[2] < 0;
    *dup = false;
    if (*off) return 0ull;
    const unsigned long long key = cc_key(j[0], j[1], j[2]);
    bool inserted;
    const uint32_t s = pag_hash_insert(table_key, C, key, &inserted);
    if (inserted) table_val[s] = (uint32_t)i;
    *dup = !inserted;
    return key;
}

// keys and insert: lattice recovery, label checks, active test, every on-lattice point into the table (key -> point index).
// info[1] += points off the lattice, info[2] += points whose lattice index an earlier insert already holds, info[3] += points with
// a label out of range.
__global__ void __launch_bounds__(MAP_CC_BLOCK) map_cc_keys_kernel(const float* __restrict__ xyz, const int64_t* __restrict__ sem,
                                                                   const int64_t* __restrict__ inst, int64_t P, int D, int Cs, int Ci,
                                                                   uint32_t thing_mask, uint32_t C, CcWorkspace w,
                                                                   long long* __restrict__ info) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool off = false, dup = false, bad = false;
    if (i < P) {
        const unsigned long long key = cc_insert_point(xyz, i, D, w.table_key, w.table_val, C, &off, &dup);
        const int64_t c = sem[i], q = inst[i];
        bad = c < 0 || c >= Cs || q < 0 || q >= Ci;
        const bool active = !off && !bad && ((thing_mask >> c) & 1u);
        w.key[i] = (long long)key;
        w.parent[i] = active ? (int)i : -1;
    }
    const int lane = threadIdx.x & 31;
    const unsigned n_off = __popc(__ballot_sync(0xffffffffu, off)), n_dup = __popc(__ballot_sync(0xffffffffu, dup)),
                   n_bad = __popc(__ballot_sync(0xffffffffu, bad));
    if (lane == 0) {
        if (n_off) atomicAdd(reinterpret_cast<unsigned long long*>(info + 1), (unsigned long long)n_off);
        if (n_dup) atomicAdd(reinterpret_cast<unsigned long long*>(info + 2), (unsigned long long)n_dup);
        if (n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(info + 3), (unsigned long long)n_bad);
    }
}

// root of x with path halving.  parent[x] <= x always (links go from the larger root to the smaller index), so the walk ends at
// the smallest point index of the tree.  volatile: the loads must see other threads' CAS results.
__device__ __forceinline__ int cc_find(volatile int* parent, int x) {
    int cur = parent[x];
    if (cur != x) {
        int next, prev = x;
        while (cur > (next = parent[cur])) {
            parent[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

// root of x without writes: flatten stores each point's root while other threads walk through it, and a path-halving write
// there could replace a stored root by an intermediate ancestor
__device__ __forceinline__ int cc_root(volatile int* parent, int x) {
    int p;
    while ((p = parent[x]) != x) x = p;
    return x;
}

// lock-free union (ECL-CC, Jaiganesh & Burtscher 2018): hook the larger root under the smaller with atomicCAS.  A failed CAS means
// that root was hooked meanwhile: continue from the node it now points to.  a is the caller's representative of its own point,
// kept across its neighbours; on return it is a node of the merged tree.
__device__ __forceinline__ void cc_hook(int* parent, int& a, int b) {
    while (a != b) {
        if (a < b) {
            const int r = atomicCAS(parent + b, b, a);
            if (r == b) return;
            b = r;
        } else {
            const int r = atomicCAS(parent + a, a, b);
            a = r == a ? b : r;
        }
    }
}

// forward neighbour offsets (dx, dy, dz) > 0 lexicographically: each adjacent pair is visited once, from its smaller lattice index
__constant__ signed char c_cc_fwd[13][3] = {{0, 0, 1},  {0, 1, -1}, {0, 1, 0},  {0, 1, 1},  {1, -1, -1}, {1, -1, 0}, {1, -1, 1},
                                            {1, 0, -1}, {1, 0, 0},  {1, 0, 1},  {1, 1, -1}, {1, 1, 0},   {1, 1, 1}};

__global__ void __launch_bounds__(MAP_CC_BLOCK) map_cc_union_kernel(const int64_t* __restrict__ inst, int64_t P, int D, int conn6,
                                                                    uint32_t C, CcWorkspace w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    volatile int* parent = w.parent;
    if (parent[i] < 0) return;      // inactive
    const unsigned long long k = (unsigned long long)w.key[i] - 1ull;
    const unsigned mask = (1u << MAP_CC_AXIS_BITS) - 1u;
    const int jx = (int)(k >> (2 * MAP_CC_AXIS_BITS)), jy = (int)((k >> MAP_CC_AXIS_BITS) & mask), jz = (int)(k & mask);
    const int64_t q = inst[i];
    int rep = cc_find(parent, (int)i);
#pragma unroll
    for (int o = 0; o < 13; ++o) {
        const int dx = c_cc_fwd[o][0], dy = c_cc_fwd[o][1], dz = c_cc_fwd[o][2];
        if (conn6 && abs(dx) + abs(dy) + abs(dz) != 1) continue;
        const int nx = jx + dx, ny = jy + dy, nz = jz + dz;
        if (nx >= D || ny < 0 || ny >= D || nz < 0 || nz >= D) continue;      // nx >= jx >= 0
        const unsigned long long nk = cc_key(nx, ny, nz);
        uint32_t s = pag_hash64(nk) & (C - 1);
        int n = -1;
        while (true) {
            const unsigned long long cur = w.table_key[s];
            if (cur == nk) { n = (int)w.table_val[s]; break; }
            if (cur == 0ull) break;
            s = (s + 1) & (C - 1);
        }
        if (n >= 0 && parent[n] >= 0 && inst[n] == q) cc_hook(w.parent, rep, cc_find(parent, n));
    }
}

// parent[i] = root(i) and count[root] += 1 (lanes with the same root add once)
__global__ void __launch_bounds__(MAP_CC_BLOCK) map_cc_flatten_kernel(int64_t P, CcWorkspace w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int r = -1;
    if (i < P && w.parent[i] >= 0) {
        r = cc_root(w.parent, (int)i);
        w.parent[i] = r;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, r);
    if (r >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(w.count + r, __popc(peers));
}

__device__ __forceinline__ bool cc_kept_root(const CcWorkspace& w, int64_t i, int64_t min_points) {
    return w.parent[i] == i && w.count[i] >= min_points;
}

// bsum[b] = number of kept roots among points [b * 1024, (b + 1) * 1024)
__global__ void __launch_bounds__(MAP_CC_SCAN_BLOCK) map_cc_flags_kernel(int64_t P, int64_t min_points, CcWorkspace w) {
    const int64_t i = (int64_t)blockIdx.x * MAP_CC_SCAN_BLOCK + threadIdx.x;
    const int n = __syncthreads_count(i < P && cc_kept_root(w, i, min_points));
    if (threadIdx.x == 0) w.bsum[blockIdx.x] = n;
}

// rank of each kept root = number of kept roots before it (block-local scan + boff); info[0] = K
__global__ void __launch_bounds__(MAP_CC_SCAN_BLOCK) map_cc_rank_kernel(int64_t P, int64_t min_points, int64_t nb, CcWorkspace w,
                                                                        long long* __restrict__ info) {
    __shared__ int warp_tot[MAP_CC_SCAN_BLOCK / 32];
    const int64_t i = (int64_t)blockIdx.x * MAP_CC_SCAN_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool flag = i < P && cc_kept_root(w, i, min_points);
    const unsigned b = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) warp_tot[wid] = __popc(b);
    __syncthreads();
    if (wid == 0) {
        const int v = warp_tot[lane];
        int incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        warp_tot[lane] = incl - v;
    }
    __syncthreads();
    if (flag) w.key[i] = w.boff[blockIdx.x] + warp_tot[wid] + __popc(b & ((1u << lane) - 1u));
    if (i == 0) info[0] = w.boff[nb];
}

__global__ void __launch_bounds__(MAP_CC_BLOCK) map_cc_label_kernel(int64_t P, int64_t min_points, CcWorkspace w,
                                                                    int64_t* __restrict__ component) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int r = w.parent[i];
    component[i] = (r >= 0 && w.count[r] >= min_points) ? w.key[r] : -1;
}

// ---- persistent lattice index of a map and lookups into it (pag_map_index, pag_map_lookup_points / _rays) ----
// The index is the components' hash table alone: key u64[C] (packed lattice index + 1, 0 = empty) and point u32[C], C =
// pag_hash_slots(P).  A lookup resolves a query position to the nearest map point of the (2r+1)^3 lattice window around it.
#define MAP_LOOKUP_BLOCK 256
#define MAP_LOOKUP_MAX_RADIUS 4

// every point into the table; info[0] += points inserted, info[1] += points off the lattice, info[2] += repeated lattice indices
__global__ void __launch_bounds__(MAP_CC_BLOCK) map_index_kernel(const float* __restrict__ xyz, int64_t P, int D, uint32_t C,
                                                                 unsigned long long* __restrict__ table_key, uint32_t* __restrict__ table_val,
                                                                 long long* __restrict__ info) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool off = false, dup = false;
    if (i < P) cc_insert_point(xyz, i, D, table_key, table_val, C, &off, &dup);
    const bool ins = i < P && !off && !dup;
    const unsigned n_ins = __popc(__ballot_sync(0xffffffffu, ins)), n_off = __popc(__ballot_sync(0xffffffffu, off)),
                   n_dup = __popc(__ballot_sync(0xffffffffu, dup));
    if ((threadIdx.x & 31) == 0) {
        if (n_ins) atomicAdd(reinterpret_cast<unsigned long long*>(info + 0), (unsigned long long)n_ins);
        if (n_off) atomicAdd(reinterpret_cast<unsigned long long*>(info + 1), (unsigned long long)n_off);
        if (n_dup) atomicAdd(reinterpret_cast<unsigned long long*>(info + 2), (unsigned long long)n_dup);
    }
}

// lanes per query: the window offsets are spread over a group of G lanes, so a query's independent probes are in flight together
// (one lane, one probe at radius 0; a warp of 32 from radius 1, 27 offsets, on)
static int map_lookup_group(int radius) { return radius == 0 ? 1 : 32; }

// One body for both query forms.  RAYS: the query is the surface point of a rendered ray, s = depth / alpha (IEEE fp32), x = o + d s
// per axis (separately rounded mul and add, the marcher's sample-position convention); rays with alpha < min_alpha or a
// non-finite s resolve to -1.  Otherwise the query is xyz.  Per axis in float64, every operation explicitly rounded:
// t = ((x + 1) D) 0.5 - 0.5, window centre j0 = floor(t + 0.5); a non-finite x or t outside [-r - 0.5, D - 0.5 + r] resolves to -1.
// Candidates: map points with lattice index j in [0, D)^3, |j - j0| <= r per axis; the chosen one has the smallest
// ((tx-jx)^2 + (ty-jy)^2) + (tz-jz)^2, then the smallest point index: a total order, so the group's shuffle reduction is
// deterministic.
template <bool RAYS>
__global__ void __launch_bounds__(MAP_LOOKUP_BLOCK) map_lookup_kernel(
        const unsigned long long* __restrict__ table_key, const uint32_t* __restrict__ table_val, uint32_t C, int D,
        const float* __restrict__ xyz, const float* __restrict__ dirs, const float* __restrict__ depth, const float* __restrict__ alpha,
        float min_alpha, int64_t Q, int radius, int G, const int64_t* __restrict__ component, int64_t* __restrict__ point,
        int64_t* __restrict__ object) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t q = tid / G;
    const int sub = (int)(tid - q * G);
    bool ok = q < Q;
    float x[3] = {0.f, 0.f, 0.f};
    if (ok) {
        if (RAYS) {
            const float a = alpha[q];
            const float s = __fdiv_rn(depth[q], a);
            ok = a >= min_alpha && isfinite(s);
#pragma unroll
            for (int c = 0; c < 3; ++c) x[c] = __fadd_rn(xyz[3 * q + c], __fmul_rn(dirs[3 * q + c], s));
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) x[c] = xyz[3 * q + c];
        }
    }
    const double lo = -(double)radius - 0.5, hi = ((double)D - 0.5) + (double)radius;
    double t[3];
    int j0[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        t[c] = __dsub_rn(__dmul_rn(__dmul_rn(__dadd_rn((double)x[c], 1.0), (double)D), 0.5), 0.5);
        ok = ok && t[c] >= lo && t[c] <= hi;      // false for NaN; an infinite x gives an infinite t
        j0[c] = ok ? (int)floor(__dadd_rn(t[c], 0.5)) : 0;
    }
    double best_d = INFINITY;
    uint32_t best_p = 0xffffffffu;
    if (ok) {
        const int w = 2 * radius + 1, W = w * w * w;
        for (int o = sub; o < W; o += G) {
            const int jx = j0[0] + o / (w * w) - radius, jy = j0[1] + (o / w) % w - radius, jz = j0[2] + o % w - radius;
            if ((unsigned)jx >= (unsigned)D || (unsigned)jy >= (unsigned)D || (unsigned)jz >= (unsigned)D) continue;
            const unsigned long long key = cc_key(jx, jy, jz);
            uint32_t s = pag_hash64(key) & (C - 1);
            unsigned long long cur;
            while ((cur = __ldg(table_key + s)) != key && cur != 0ull) s = (s + 1) & (C - 1);
            if (cur == 0ull) continue;
            const uint32_t p = __ldg(table_val + s);
            const double dx = __dsub_rn(t[0], (double)jx), dy = __dsub_rn(t[1], (double)jy), dz = __dsub_rn(t[2], (double)jz);
            const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
            if (d2 < best_d || (d2 == best_d && p < best_p)) { best_d = d2; best_p = p; }
        }
    }
    for (int m = G >> 1; m > 0; m >>= 1) {      // G = 32: the group is the warp, every lane takes part
        const double od = __shfl_xor_sync(0xffffffffu, best_d, m);
        const uint32_t op = __shfl_xor_sync(0xffffffffu, best_p, m);
        if (od < best_d || (od == best_d && op < best_p)) { best_d = od; best_p = op; }
    }
    if (q < Q && sub == 0) {
        const int64_t p = best_p == 0xffffffffu ? -1 : (int64_t)best_p;
        point[q] = p;
        if (object) object[q] = p >= 0 ? component[p] : -1;
    }
}

static int map_lookup_launch(bool rays, const int64_t* keys, const int32_t* points, int64_t C, int level, int k, const float* xyz,
                             const float* dirs, const float* depth, const float* alpha, float min_alpha, int64_t Q, int radius,
                             const int64_t* component, int64_t* point, int64_t* object, cudaStream_t s) {
    if (C < 2 || C > (1ll << 31) || (C & (C - 1)) || Q < 0 || level < 0 || level > 15 || k < 1 || k > 8 || radius < 0 ||
        radius > MAP_LOOKUP_MAX_RADIUS)
        return PAG_ERR_ARG;
    if (rays && !(min_alpha > 0.f && min_alpha <= 1.f)) return PAG_ERR_ARG;
    if (Q == 0) return PAG_OK;
    if (!keys || !points || !xyz || !point || (rays && (!dirs || !depth || !alpha))) return PAG_ERR_ARG;
    const int G = map_lookup_group(radius);
    const int64_t blocks = (Q * G + MAP_LOOKUP_BLOCK - 1) / MAP_LOOKUP_BLOCK;
    if (blocks > 0x7fffffff) return PAG_ERR_ARG;
    const unsigned long long* tk = reinterpret_cast<const unsigned long long*>(keys);
    const uint32_t* tv = reinterpret_cast<const uint32_t*>(points);
    if (rays)
        map_lookup_kernel<true><<<(unsigned)blocks, MAP_LOOKUP_BLOCK, 0, s>>>(tk, tv, (uint32_t)C, k << level, xyz, dirs, depth, alpha,
                                                                              min_alpha, Q, radius, G, component, point, object);
    else
        map_lookup_kernel<false><<<(unsigned)blocks, MAP_LOOKUP_BLOCK, 0, s>>>(tk, tv, (uint32_t)C, k << level, xyz, nullptr, nullptr,
                                                                               nullptr, 1.f, Q, radius, G, component, point, object);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// ---- projection of a map into camera views (pag_map_project): z-buffered splatting of the lattice cells' squares ----
// The depth buffer holds one u64 key per pixel, (z bits << 32) | point, all ones where nothing is seen.  z > near > 0, so the float
// bits order like the values and the smallest key is the nearest point, then the smallest point index.
#define MAP_PROJECT_BLOCK 256
#define MAP_PROJECT_MAX_RADIUS 32
#define MAP_PROJECT_MAX_SIDE 16384
#define MAP_PROJECT_MAX_CAMERAS 65535      // gridDim.y
#define MAP_PROJECT_EMPTY 0xffffffffffffffffull

// camera b's rows 0..2 of the view matrix, then fx, fy, cx, cy, into s_cam[16]; the caller synchronises the block
__device__ __forceinline__ void map_stage_camera(const float* __restrict__ view, const float* __restrict__ intrinsics, int b, float* s_cam) {
    if (threadIdx.x < 12) s_cam[threadIdx.x] = view[16 * (int64_t)b + threadIdx.x];
    else if (threadIdx.x < 16) s_cam[threadIdx.x] = intrinsics[4 * (int64_t)b + threadIdx.x - 12];
}

struct MapFootprint {
    float z;
    int c0, c1, r0, r1;      // covered columns / rows, clipped to the image
};

// The footprint of point i in the camera of s_cam, the one definition of coverage shared by the projection and the visibility
// passes.  Every operation is separately rounded (the oracle's numpy order): p_q = ((V[q,0] x + V[q,1] y) + V[q,2] z) + V[q,3],
// depth z = -p_2, u = fx (p_0 / z) + cx, v = fy (p_1 / z) + cy, su = min((fx h) / z, R), sv likewise.  A point is projected iff
// z > near, u and v are finite and su, sv >= 0 (false for NaN, so a NaN half-size never becomes R, and a negative focal length
// covers nothing).  Pixels: columns floor(u - su) .. floor(u + su), rows floor(v - sv) .. floor(v + sv), clamped to the image in
// float before the conversion to int.  Returns false when the point is dropped or covers no pixel of the image.
__device__ __forceinline__ bool map_footprint(const float* __restrict__ xyz, int64_t i, const float* s_cam, int H, int W, float h,
                                              float near, int max_radius, MapFootprint& f) {
    const float x = xyz[3 * i], y = xyz[3 * i + 1], zw = xyz[3 * i + 2];
    float p[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const float* V = s_cam + 4 * q;
        p[q] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(V[0], x), __fmul_rn(V[1], y)), __fmul_rn(V[2], zw)), V[3]);
    }
    const float fx = s_cam[12], fy = s_cam[13], cx = s_cam[14], cy = s_cam[15];
    const float z = -p[2];
    if (!(z > near)) return false;
    const float u = __fadd_rn(__fmul_rn(fx, __fdiv_rn(p[0], z)), cx), v = __fadd_rn(__fmul_rn(fy, __fdiv_rn(p[1], z)), cy);
    const float ru = __fdiv_rn(__fmul_rn(fx, h), z), rv = __fdiv_rn(__fmul_rn(fy, h), z);
    if (!isfinite(u) || !isfinite(v) || !(ru >= 0.f) || !(rv >= 0.f)) return false;
    const float R = (float)max_radius;
    const float su = fminf(ru, R), sv = fminf(rv, R);
    const float c0f = fmaxf(floorf(__fsub_rn(u, su)), 0.f), c1f = fminf(floorf(__fadd_rn(u, su)), (float)(W - 1));
    const float r0f = fmaxf(floorf(__fsub_rn(v, sv)), 0.f), r1f = fminf(floorf(__fadd_rn(v, sv)), (float)(H - 1));
    if (c0f > c1f || r0f > r1f) return false;
    f.z = z;
    f.c0 = (int)c0f; f.c1 = (int)c1f; f.r0 = (int)r0f; f.r1 = (int)r1f;
    return true;
}

// One thread per (point, camera): grid x over points, y over cameras.  Each pixel of the footprint is tested with a plain load of
// its current key and takes an atomicMin only when the new key is smaller: the atomic decides, the load only skips the atomics
// that cannot win (points arrive in leaf-cell order, so a warp's squares overlap and the skipped atomics would serialise on one
// address).
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_project_splat_kernel(
        const float* __restrict__ xyz, int64_t P, const float* __restrict__ view, const float* __restrict__ intrinsics, int H, int W,
        float h, float near, int max_radius, unsigned long long* __restrict__ zbuf) {
    __shared__ float s_cam[16];
    const int b = blockIdx.y;
    map_stage_camera(view, intrinsics, b, s_cam);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    MapFootprint f;
    if (!map_footprint(xyz, i, s_cam, H, W, h, near, max_radius, f)) return;
    const unsigned long long key = ((unsigned long long)__float_as_uint(f.z) << 32) | (unsigned long long)i;
    unsigned long long* img = zbuf + (int64_t)b * H * W;
    for (int r = f.r0; r <= f.r1; ++r) {
        unsigned long long* row = img + (int64_t)r * W;
        for (int c = f.c0; c <= f.c1; ++c)
            if (key < __ldcg(row + c)) atomicMin(row + c, key);
    }
}

// one thread per pixel: the key's point and depth, and component[point] (component nullable)
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_project_resolve_kernel(
        const unsigned long long* __restrict__ zbuf, int64_t N, const int64_t* __restrict__ component, int64_t* __restrict__ point,
        float* __restrict__ depth, int64_t* __restrict__ object) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N) return;
    const unsigned long long key = zbuf[t];
    const bool hit = key != MAP_PROJECT_EMPTY;
    const int64_t p = hit ? (int64_t)(key & 0xffffffffull) : -1;
    point[t] = p;
    depth[t] = hit ? __uint_as_float((uint32_t)(key >> 32)) : INFINITY;
    if (object) object[t] = hit ? component[p] : -1;
}

// ---- per-object visibility in camera views (pag_map_visibility, pag_map_visibility_silhouette) ----
// Pair n = b K + o: object o in view b.  Boxes i32[N][4] = (col_min, row_min, col_max, row_max), empty as (BIG, BIG, -1, -1).  A
// pair's silhouette bitmap covers its footprint-union box, one bit per pixel, each row padded to whole 32-bit words of the image
// (word w holds columns 32 w .. 32 w + 31), so a pair takes rows * ((col_max >> 5) - (col_min >> 5) + 1) words.
#define MAP_VIS_BIG 0x7fffffff

__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_vis_init_kernel(int64_t N, int* __restrict__ box, int* __restrict__ bbox,
                                                                         long long* __restrict__ visible, long long* __restrict__ silhouette) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int4 e = make_int4(MAP_VIS_BIG, MAP_VIS_BIG, -1, -1);
    reinterpret_cast<int4*>(box)[n] = e;
    reinterpret_cast<int4*>(bbox)[n] = e;
    visible[n] = 0;
    silhouette[n] = 0;
}

// Lanes with equal pair (all 32 lanes call; pair < 0: nothing to add) merge their rectangles with warp reductions, and the group's
// first lane widens box[pair] with one atomic per side that the rectangle extends (a plain load skips the others: boxes stop
// growing early, and the skipped atomics would serialise on one address) and adds the group's size to count[pair] (nullable).
__device__ __forceinline__ void map_vis_widen(long long pair, int c0, int r0, int c1, int r1, int* __restrict__ box,
                                              unsigned long long* __restrict__ count) {
    const unsigned peers = __match_any_sync(0xffffffffu, pair);
    c0 = __reduce_min_sync(peers, c0);
    r0 = __reduce_min_sync(peers, r0);
    c1 = __reduce_max_sync(peers, c1);
    r1 = __reduce_max_sync(peers, r1);
    if (pair < 0 || (int)(threadIdx.x & 31) != __ffs(peers) - 1) return;
    if (count) atomicAdd(count + pair, (unsigned long long)__popc(peers));
    int* bx = box + 4 * pair;
    if (c0 < __ldcg(bx + 0)) atomicMin(bx + 0, c0);
    if (r0 < __ldcg(bx + 1)) atomicMin(bx + 1, r0);
    if (c1 > __ldcg(bx + 2)) atomicMax(bx + 2, c1);
    if (r1 > __ldcg(bx + 3)) atomicMax(bx + 3, r1);
}

// one thread per pixel of the depth buffer: the front point's object o in [0, K) counts the pixel toward visible[b, o] and widens
// bbox[b, o]; components outside [0, K) are skipped (out-of-range ones are counted by map_vis_box_kernel)
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_vis_visible_kernel(
        const unsigned long long* __restrict__ zbuf, int64_t N, int H, int W, const int64_t* __restrict__ component, int K,
        long long* __restrict__ visible, int* __restrict__ bbox) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // every lane stays for the warp collectives
    long long pair = -1;
    int r = 0, c = 0;
    if (t < N) {
        const unsigned long long key = zbuf[t];
        if (key != MAP_PROJECT_EMPTY) {
            const int64_t o = component[key & 0xffffffffull];
            if (o >= 0 && o < K) {
                const int64_t hw = (int64_t)H * W, b = t / hw, pix = t - b * hw;
                r = (int)(pix / W);
                c = (int)(pix - (int64_t)r * W);
                pair = b * K + o;
            }
        }
    }
    map_vis_widen(pair, c, r, c, r, bbox, reinterpret_cast<unsigned long long*>(visible));
}

// one thread per (point, camera), grid y = max(B, 1): the footprint of a point of object o in [0, K) widens box[b, o].  The cameras'
// first row counts the points whose component lies outside [-1, K) into errors[0], once per point, also when B = 0.
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_vis_box_kernel(
        const float* __restrict__ xyz, int64_t P, const float* __restrict__ view, const float* __restrict__ intrinsics, int B, int H,
        int W, float h, float near, int max_radius, const int64_t* __restrict__ component, int K, int* __restrict__ box,
        long long* __restrict__ errors) {
    __shared__ float s_cam[16];
    const int b = blockIdx.y;
    if (b < B) map_stage_camera(view, intrinsics, b, s_cam);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t o = i < P ? component[i] : -1;
    if (b == 0) {
        const unsigned n_bad = __popc(__ballot_sync(0xffffffffu, o < -1 || o >= K));
        if ((threadIdx.x & 31) == 0 && n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(errors), (unsigned long long)n_bad);
    }
    MapFootprint f = {0.f, 0, 0, 0, 0};
    const bool on = b < B && o >= 0 && o < K && map_footprint(xyz, i, s_cam, H, W, h, near, max_radius, f);
    map_vis_widen(on ? (long long)b * K + o : -1, f.c0, f.r0, f.c1, f.r1, box, nullptr);
}

// one thread per pair: bbox = -1 where nothing is visible, words[n] = the size of the pair's bitmap (0 for an empty box)
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_vis_pairs_kernel(int64_t N, const long long* __restrict__ visible,
                                                                          const int* __restrict__ box, int* __restrict__ bbox,
                                                                          int* __restrict__ words) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    if (visible[n] == 0) reinterpret_cast<int4*>(bbox)[n] = make_int4(-1, -1, -1, -1);
    const int4 e = reinterpret_cast<const int4*>(box)[n];
    words[n] = e.z >= e.x ? (e.w - e.y + 1) * ((e.z >> 5) - (e.x >> 5) + 1) : 0;
}

// One round of silhouettes: thread per (point, camera); a point of object o whose pair's bitmap starts at offset[pair] in
// [lo, hi) (in words) ORs its footprint into that bitmap at bits + offset - lo.  A footprint row spans at most 66 columns, so at
// most 4 words; a plain load skips the atomicOr when the word already holds the bits.
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_vis_or_kernel(
        const float* __restrict__ xyz, int64_t P, const float* __restrict__ view, const float* __restrict__ intrinsics, int H, int W,
        float h, float near, int max_radius, const int64_t* __restrict__ component, int K, const int* __restrict__ box,
        const int64_t* __restrict__ offset, int64_t lo, int64_t hi, unsigned* __restrict__ bits) {
    __shared__ float s_cam[16];
    const int b = blockIdx.y;
    map_stage_camera(view, intrinsics, b, s_cam);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int64_t o = component[i];
    if (o < 0 || o >= K) return;
    const int64_t pair = (int64_t)b * K + o;
    const int64_t off = offset[pair];
    if (off < lo || off >= hi) return;
    MapFootprint f;
    if (!map_footprint(xyz, i, s_cam, H, W, h, near, max_radius, f)) return;
    const int4 e = reinterpret_cast<const int4*>(box)[pair];
    const int w0 = e.x >> 5, wpr = (e.z >> 5) - w0 + 1;
    unsigned* img = bits + (off - lo) - w0;          // + row * wpr + word: word (c >> 5) of the pair's row
    for (int r = f.r0; r <= f.r1; ++r) {
        unsigned* row = img + (int64_t)(r - e.y) * wpr;
        for (int w = f.c0 >> 5; w <= (f.c1 >> 5); ++w) {
            const int a = max(f.c0 - 32 * w, 0), z = min(f.c1 - 32 * w, 31);
            const unsigned m = (0xffffffffu >> (31 - z)) & (0xffffffffu << a);
            if ((__ldcg(row + w) & m) != m) atomicOr(row + w, m);
        }
    }
}

// one warp per pair of the round: silhouette[n] = the popcount of its bitmap
__global__ void __launch_bounds__(MAP_PROJECT_BLOCK) map_vis_popc_kernel(int64_t N, const int* __restrict__ words,
                                                                         const int64_t* __restrict__ offset, int64_t lo, int64_t hi,
                                                                         const unsigned* __restrict__ bits,
                                                                         long long* __restrict__ silhouette) {
    const int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;                                                      // warp-uniform
    const int64_t off = offset[n];
    const int nw = words[n];
    if (nw == 0 || off < lo || off >= hi) return;
    const unsigned* w = bits + (off - lo);
    long long s = 0;
    for (int j = lane; j < nw; j += 32) s += __popc(__ldcg(w + j));
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) silhouette[n] = s;
}

static int map_stats_launch(const float* xyz, const float* rgb, const int64_t* semantic, const int64_t* lab, int64_t P, int Cs, int Ci,
                            uint32_t thing_mask, int unlabelled_ok, const int64_t* inst_src, int64_t* inst_out, int64_t* count,
                            double* sum_xyz, double* sum_rgb, int64_t* votes, float* bbox_min, float* bbox_max, int64_t* errors,
                            cudaStream_t stream) {
    // a few CTAs per SM: every CTA of the shared-memory kernel flushes its non-empty slots once, so fewer, longer-lived CTAs mean
    // fewer global atomics
    const int64_t want = pag_grid(P, MAP_STATS_BLOCK);
    const int64_t cap = 4 * (int64_t)map_num_sms();
    const int grid = (int)(want < cap ? want : cap);
    const int64_t slot_bytes = 76 + 4 * (int64_t)Cs;      // map_stats_layout per label
    if ((int64_t)Ci * slot_bytes <= 227 * 1024) {
        const size_t bytes = (size_t)map_stats_layout(Cs, Ci).total;
        if (bytes > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(map_instance_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            if (e != cudaSuccess) return (int)e;
        }
        map_instance_stats_kernel<<<grid, MAP_STATS_BLOCK, bytes, stream>>>(
            xyz, rgb, semantic, lab, P, Cs, Ci, thing_mask, unlabelled_ok, inst_src, inst_out, reinterpret_cast<long long*>(count),
            sum_xyz, sum_rgb, votes, bbox_min, bbox_max, reinterpret_cast<long long*>(errors));
    } else {
        map_instance_stats_global_kernel<<<(int)want, MAP_STATS_BLOCK, 0, stream>>>(
            xyz, rgb, semantic, lab, P, Cs, Ci, thing_mask, unlabelled_ok, inst_src, inst_out, reinterpret_cast<long long*>(count),
            sum_xyz, sum_rgb, votes, bbox_min, bbox_max, reinterpret_cast<long long*>(errors));
    }
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

extern "C" int pag_exclusive_scan_i32(const int32_t* in, int64_t N, int64_t* out, void* stream);      // csrc/octree.cu

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
    if (P == 0) return PAG_OK;
    if (!xyz || !rgb || !semantic || !instance || !count || !sum_xyz || !sum_rgb || !votes || !bbox_min || !bbox_max || !errors)
        return PAG_ERR_ARG;
    return map_stats_launch(xyz, rgb, semantic, instance, P, Cs, Ci, thing_mask, 0, nullptr, nullptr, count, sum_xyz, sum_rgb, votes,
                            bbox_min, bbox_max, errors, (cudaStream_t)stream);
}

int pag_map_components_workspace(int64_t P, int64_t* bytes) {
    if (P < 0 || P > MAP_CC_MAX_POINTS || bytes == nullptr) return PAG_ERR_ARG;
    *bytes = cc_workspace_bytes(P);
    return PAG_OK;
}

int pag_map_components(const float* xyz, const int64_t* semantic, const int64_t* instance, int64_t P, int level, int k, int Cs, int Ci,
                       uint32_t thing_mask, int connectivity, int64_t min_points, void* workspace, int64_t workspace_bytes,
                       int64_t* component, int64_t* info, void* stream) {
    if (P < 0 || P > MAP_CC_MAX_POINTS || level < 0 || level > 15 || k < 1 || k > 8 || Cs < 1 || Cs > 32 || Ci < 1) return PAG_ERR_ARG;
    if ((connectivity != 6 && connectivity != 26) || min_points < 1 || !info) return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(info, 0, 4 * sizeof(int64_t), s);
    if (e != cudaSuccess) return (int)e;
    if (P == 0) return PAG_OK;
    if (!xyz || !semantic || !instance || !component || !workspace || workspace_bytes < cc_workspace_bytes(P)) return PAG_ERR_ARG;
    if (reinterpret_cast<uintptr_t>(workspace) & 7) return PAG_ERR_ARG;
    const int64_t C = pag_hash_slots(P), nb = cc_blocks(P);
    const CcWorkspace w = cc_workspace(workspace, P);
    const int D = k << level;
    long long* inf = reinterpret_cast<long long*>(info);
    if ((e = cudaMemsetAsync(w.table_key, 0, C * sizeof(unsigned long long), s)) != cudaSuccess) return (int)e;
    if ((e = cudaMemsetAsync(w.count, 0, P * sizeof(int), s)) != cudaSuccess) return (int)e;
    const int g = pag_grid(P, MAP_CC_BLOCK);
    map_cc_keys_kernel<<<g, MAP_CC_BLOCK, 0, s>>>(xyz, semantic, instance, P, D, Cs, Ci, thing_mask, (uint32_t)C, w, inf);
    PAG_LAUNCH_CHECK();
    map_cc_union_kernel<<<g, MAP_CC_BLOCK, 0, s>>>(instance, P, D, connectivity == 6, (uint32_t)C, w);
    PAG_LAUNCH_CHECK();
    map_cc_flatten_kernel<<<g, MAP_CC_BLOCK, 0, s>>>(P, w);
    PAG_LAUNCH_CHECK();
    map_cc_flags_kernel<<<(int)nb, MAP_CC_SCAN_BLOCK, 0, s>>>(P, min_points, w);
    PAG_LAUNCH_CHECK();
    const int rc = pag_exclusive_scan_i32(w.bsum, nb, w.boff, stream);
    if (rc != PAG_OK) return rc;
    map_cc_rank_kernel<<<(int)nb, MAP_CC_SCAN_BLOCK, 0, s>>>(P, min_points, nb, w, inf);
    PAG_LAUNCH_CHECK();
    map_cc_label_kernel<<<g, MAP_CC_BLOCK, 0, s>>>(P, min_points, w, component);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

int pag_map_component_stats(const float* xyz, const float* rgb, const int64_t* semantic, const int64_t* instance, const int64_t* component,
                            int64_t P, int Cs, int K, int64_t* count, double* sum_xyz, double* sum_rgb, int64_t* votes, float* bbox_min,
                            float* bbox_max, int64_t* object_instance, void* stream) {
    if (P < 0 || Cs < 1 || Cs > 32 || K < 0) return PAG_ERR_ARG;
    if (P == 0 || K == 0) return PAG_OK;
    if (!xyz || !rgb || !semantic || !instance || !component || !count || !sum_xyz || !sum_rgb || !votes || !bbox_min || !bbox_max ||
        !object_instance)
        return PAG_ERR_ARG;
    return map_stats_launch(xyz, rgb, semantic, component, P, Cs, K, 0xffffffffu, 1, instance, object_instance, count, sum_xyz, sum_rgb,
                            votes, bbox_min, bbox_max, nullptr, (cudaStream_t)stream);
}

int pag_map_index_bytes(int64_t P, int64_t* bytes) {
    if (P < 0 || P > MAP_CC_MAX_POINTS || bytes == nullptr) return PAG_ERR_ARG;
    *bytes = 12 * pag_hash_slots(P);
    return PAG_OK;
}

int pag_map_index(const float* xyz, int64_t P, int level, int k, int64_t* keys, int32_t* points, int64_t C, int64_t* info,
                  void* stream) {
    if (P < 0 || P > MAP_CC_MAX_POINTS || level < 0 || level > 15 || k < 1 || k > 8 || !info || !keys || !points) return PAG_ERR_ARG;
    if (C != pag_hash_slots(P) || (P > 0 && !xyz)) return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(info, 0, 4 * sizeof(int64_t), s);
    if (e != cudaSuccess) return (int)e;
    if ((e = cudaMemsetAsync(keys, 0, C * sizeof(int64_t), s)) != cudaSuccess) return (int)e;
    if (P == 0) return PAG_OK;
    map_index_kernel<<<pag_grid(P, MAP_CC_BLOCK), MAP_CC_BLOCK, 0, s>>>(xyz, P, k << level, (uint32_t)C,
                                                                       reinterpret_cast<unsigned long long*>(keys),
                                                                       reinterpret_cast<uint32_t*>(points), reinterpret_cast<long long*>(info));
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

int pag_map_lookup_points(const int64_t* keys, const int32_t* points, int64_t C, int level, int k, const float* xyz, int64_t Q,
                          int radius, const int64_t* component, int64_t* point, int64_t* object, void* stream) {
    return map_lookup_launch(false, keys, points, C, level, k, xyz, nullptr, nullptr, nullptr, 1.f, Q, radius, component, point, object,
                             (cudaStream_t)stream);
}

int pag_map_lookup_rays(const int64_t* keys, const int32_t* points, int64_t C, int level, int k, const float* origins,
                        const float* dirs, const float* depth, const float* alpha, float min_alpha, int64_t Q, int radius,
                        const int64_t* component, int64_t* point, int64_t* object, void* stream) {
    return map_lookup_launch(true, keys, points, C, level, k, origins, dirs, depth, alpha, min_alpha, Q, radius, component, point, object,
                             (cudaStream_t)stream);
}

int pag_map_project(const float* xyz, int64_t P, const float* view, const float* intrinsics, int B, int H, int W, float h, float near,
                    int max_radius, int64_t* zbuf, const int64_t* component, int64_t* point, float* depth, int64_t* object,
                    void* stream) {
    if (P < 0 || P > MAP_CC_MAX_POINTS || B < 0 || B > MAP_PROJECT_MAX_CAMERAS || H < 1 || H > MAP_PROJECT_MAX_SIDE || W < 1 ||
        W > MAP_PROJECT_MAX_SIDE || max_radius < 0 || max_radius > MAP_PROJECT_MAX_RADIUS || !(near > 0.f) || !isfinite(near) ||
        !(h > 0.f) || !isfinite(h))
        return PAG_ERR_ARG;
    if (B == 0) return PAG_OK;
    // an empty map's xyz and component may be null (torch gives an empty tensor no storage): no pixel is covered, nothing is read
    if (!view || !intrinsics || !zbuf || !point || !depth || (P > 0 && (!xyz || (object && !component)))) return PAG_ERR_ARG;
    const int64_t N = (int64_t)B * H * W;
    if ((N + MAP_PROJECT_BLOCK - 1) / MAP_PROJECT_BLOCK > 0x7fffffff) return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(zbuf, 0xff, N * sizeof(int64_t), s);
    if (e != cudaSuccess) return (int)e;
    unsigned long long* zb = reinterpret_cast<unsigned long long*>(zbuf);
    if (P > 0) {
        map_project_splat_kernel<<<dim3((unsigned)pag_grid(P, MAP_PROJECT_BLOCK), (unsigned)B), MAP_PROJECT_BLOCK, 0, s>>>(
            xyz, P, view, intrinsics, H, W, h, near, max_radius, zb);
        PAG_LAUNCH_CHECK();
    }
    map_project_resolve_kernel<<<(unsigned)pag_grid(N, MAP_PROJECT_BLOCK), MAP_PROJECT_BLOCK, 0, s>>>(zb, N, component, point, depth,
                                                                                                      object);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

static bool map_vis_args_ok(int64_t P, int B, int H, int W, float h, float near, int max_radius, int K) {
    return P >= 0 && P <= MAP_CC_MAX_POINTS && B >= 0 && B <= MAP_PROJECT_MAX_CAMERAS && H >= 1 && H <= MAP_PROJECT_MAX_SIDE && W >= 1 &&
           W <= MAP_PROJECT_MAX_SIDE && max_radius >= 0 && max_radius <= MAP_PROJECT_MAX_RADIUS && near > 0.f && isfinite(near) &&
           h > 0.f && isfinite(h) && K >= 0 && K <= MAP_CC_MAX_POINTS;
}

int pag_map_visibility(const float* xyz, int64_t P, const float* view, const float* intrinsics, int B, int H, int W, float h, float near,
                       int max_radius, const int64_t* component, int K, int64_t* zbuf, int32_t* box, int32_t* words, int64_t* offset,
                       int64_t* visible, int64_t* silhouette, int32_t* bbox, void* stream) {
    if (!map_vis_args_ok(P, B, H, W, h, near, max_radius, K) || !offset) return PAG_ERR_ARG;
    const int64_t N = (int64_t)B * K, NP = (int64_t)B * H * W;
    if ((NP + MAP_PROJECT_BLOCK - 1) / MAP_PROJECT_BLOCK > 0x7fffffff || (32 * N + MAP_PROJECT_BLOCK - 1) / MAP_PROJECT_BLOCK > 0x7fffffff)
        return PAG_ERR_ARG;      // a thread per pixel, a warp per pair
    if ((P > 0 && (!xyz || !component)) || (B > 0 && (!view || !intrinsics)) ||
        (N > 0 && (!box || !words || !visible || !silhouette || !bbox)) || (N > 0 && P > 0 && !zbuf))
        return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(offset + N + 1, 0, sizeof(int64_t), s);      // the error count
    if (e != cudaSuccess) return (int)e;
    long long* errors = reinterpret_cast<long long*>(offset + N + 1);
    if (N > 0) {
        map_vis_init_kernel<<<pag_grid(N, MAP_PROJECT_BLOCK), MAP_PROJECT_BLOCK, 0, s>>>(N, box, bbox, reinterpret_cast<long long*>(visible),
                                                                                          reinterpret_cast<long long*>(silhouette));
        PAG_LAUNCH_CHECK();
    }
    unsigned long long* zb = reinterpret_cast<unsigned long long*>(zbuf);
    if (N > 0 && P > 0) {      // the front points (pag_map_project's fill and splat) and the visible counts; none in an empty map
        if ((e = cudaMemsetAsync(zbuf, 0xff, NP * sizeof(int64_t), s)) != cudaSuccess) return (int)e;
        map_project_splat_kernel<<<dim3((unsigned)pag_grid(P, MAP_PROJECT_BLOCK), (unsigned)B), MAP_PROJECT_BLOCK, 0, s>>>(
            xyz, P, view, intrinsics, H, W, h, near, max_radius, zb);
        PAG_LAUNCH_CHECK();
        map_vis_visible_kernel<<<(unsigned)pag_grid(NP, MAP_PROJECT_BLOCK), MAP_PROJECT_BLOCK, 0, s>>>(
            zb, NP, H, W, component, K, reinterpret_cast<long long*>(visible), bbox);
        PAG_LAUNCH_CHECK();
    }
    if (P > 0) {      // footprint boxes; the out-of-range count also when there is no pair
        map_vis_box_kernel<<<dim3((unsigned)pag_grid(P, MAP_PROJECT_BLOCK), (unsigned)(B > 0 ? B : 1)), MAP_PROJECT_BLOCK, 0, s>>>(
            xyz, P, view, intrinsics, B, H, W, h, near, max_radius, component, K, box, errors);
        PAG_LAUNCH_CHECK();
    }
    if (N > 0) {
        map_vis_pairs_kernel<<<pag_grid(N, MAP_PROJECT_BLOCK), MAP_PROJECT_BLOCK, 0, s>>>(N, reinterpret_cast<const long long*>(visible),
                                                                                           box, bbox, words);
        PAG_LAUNCH_CHECK();
        return pag_exclusive_scan_i32(words, N, offset, stream);
    }
    e = cudaMemsetAsync(offset, 0, sizeof(int64_t), s);      // no pair: total 0
    return e == cudaSuccess ? PAG_OK : (int)e;
}

int pag_map_visibility_silhouette(const float* xyz, int64_t P, const float* view, const float* intrinsics, int B, int H, int W, float h,
                                  float near, int max_radius, const int64_t* component, int K, const int32_t* box, const int32_t* words,
                                  const int64_t* offset, int64_t total_words, int32_t* bits, int64_t bits_words, int64_t* silhouette,
                                  void* stream) {
    if (!map_vis_args_ok(P, B, H, W, h, near, max_radius, K) || total_words < 0 || bits_words < 0) return PAG_ERR_ARG;
    const int64_t N = (int64_t)B * K;
    if (N == 0 || P == 0 || total_words == 0) return PAG_OK;
    if (!xyz || !view || !intrinsics || !component || !box || !words || !offset || !bits || !silhouette) return PAG_ERR_ARG;
    // rounds are windows [lo, lo + step) of the bitmaps' offsets: a pair starting in the window ends before lo + step + (its size
    // <= max_pair), so every round fits in bits_words = step + max_pair words
    const int64_t max_pair = (int64_t)H * (((W - 1) >> 5) + 1);
    const int64_t step = total_words <= bits_words ? total_words : bits_words - max_pair;
    if (step <= 0) return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned* bw = reinterpret_cast<unsigned*>(bits);
    for (int64_t lo = 0; lo < total_words; lo += step) {
        const int64_t hi = lo + step, used = (total_words < hi + max_pair ? total_words : hi + max_pair) - lo;
        cudaError_t e = cudaMemsetAsync(bits, 0, (used < bits_words ? used : bits_words) * sizeof(int32_t), s);
        if (e != cudaSuccess) return (int)e;
        map_vis_or_kernel<<<dim3((unsigned)pag_grid(P, MAP_PROJECT_BLOCK), (unsigned)B), MAP_PROJECT_BLOCK, 0, s>>>(
            xyz, P, view, intrinsics, H, W, h, near, max_radius, component, K, box, offset, lo, hi, bw);
        PAG_LAUNCH_CHECK();
        map_vis_popc_kernel<<<pag_grid(32 * N, MAP_PROJECT_BLOCK), MAP_PROJECT_BLOCK, 0, s>>>(N, words, offset, lo, hi, bw,
                                                                                            reinterpret_cast<long long*>(silhouette));
        PAG_LAUNCH_CHECK();
    }
    return PAG_OK;
}

}  // extern "C"
