// Panoptic quality (PQ) update on the device (validation metric of pc_nerf/trainer.py:651-941).
//
// Replaces the update step of the vendored torchmetrics PanopticQuality (utils/metrics/panoptic_quality.py), which runs
// torch.unique per image, turns every segment colour into a Python tuple (a device-to-host copy each) and walks segments and
// segment pairs in Python dictionaries.  Here one update of B images is three launches with no host synchronisation, and the
// launch geometry depends on (B, P) only:
//   hist       thread per pixel: category -> continuous id through a sorted table in shared memory, preprocessing (stuff ->
//              instance 0, unknown -> void), then per image open-addressing hash tables with 64-bit keys count the area of every
//              prediction segment, of every target segment, the void overlap of each (|p ∩ void_target|, |t ∩ void_pred|) and
//              the intersection of every same-category (prediction, target) pair.  Lanes of a warp with the same key are merged
//              with __match_any_sync: one atomic per distinct key per warp.
//   match      thread per pair slot: IoU = |p∩t| / (|p| - |p ∩ void_t| + |t| - |p∩t|); the decision IoU > 0.5 is taken on the exact
//              integers (2|p∩t| > union), the IoU added to iou_sum in float64; matched segments get bit 31 of their area.
//              Clears the pair slot.
//   unmatched  thread per segment slot (prediction and target tables): an unmatched segment whose void overlap is at most half
//              of its area counts as FP (prediction) or FN (target).  Clears the segment slot.
// The workspace therefore starts and ends zeroed: the caller zero-fills it once and every update leaves it clean.
//
// Workspace of B images of P pixels, C = pag_hash_slots(P) = smallest power of two >= 2P slots per table (so that P distinct
// segments -- every pixel its own segment -- fill at most half of a table: nothing overflows, whatever the data):
//   u64 pred_key[B][C] | u64 tgt_key[B][C] | u64 pair_key[B][C] | u32 pred_area[B][C] | u32 pred_void[B][C] | u32 tgt_area[B][C]
//   | u32 tgt_void[B][C] | u32 pair_cnt[B][C]                                           = 44 * B * C bytes (key 0 = empty slot)
// Segment key = (continuous id + 1) << 32 | instance; pair key = (prediction slot + 1) << 32 | target slot.  Void pixels are never
// inserted: torchmetrics discards the void colour from both FP and FN and never matches it, only its overlaps are used.
#include "common.cuh"

#define PQ_MAX_CATEGORIES 256
#define PQ_HIST_BLOCK 256
#define PQ_HIST_PIXELS_PER_THREAD 4

struct PqTables {
    unsigned long long *pred_key, *tgt_key, *pair_key;
    unsigned int *pred_area, *pred_void, *tgt_area, *tgt_void, *pair_cnt;
};

static PqTables pq_tables(void* ws, int64_t n) {      // n = B * C slots per table
    PqTables t;
    unsigned long long* k = reinterpret_cast<unsigned long long*>(ws);
    t.pred_key = k;
    t.tgt_key = k + n;
    t.pair_key = k + 2 * n;
    unsigned int* u = reinterpret_cast<unsigned int*>(k + 3 * n);
    t.pred_area = u;
    t.pred_void = u + n;
    t.tgt_area = u + 2 * n;
    t.tgt_void = u + 3 * n;
    t.pair_cnt = u + 4 * n;
    return t;
}

// -> continuous id | 0x100 if thing, or -1 if the category is unknown (sorted ids in shared memory, binary search)
__device__ __forceinline__ int pq_lookup(const int* __restrict__ ids, const int* __restrict__ code, int K, long long cat) {
    if (cat < 0 || cat > 0x7fffffffll) return -1;
    int lo = 0, hi = K;
    const int c = (int)cat;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (ids[mid] < c) lo = mid + 1; else hi = mid;
    }
    return (lo < K && ids[lo] == c) ? code[lo] : -1;
}

// one map's pixel -> segment key (0 = void).  bad: a thing's instance id outside [0, 2^31); unknown: category in neither set.
__device__ __forceinline__ unsigned long long pq_key(const int* ids, const int* code, int K, long long cat, long long inst,
                                                     bool& unknown, bool& bad) {
    const int cc = pq_lookup(ids, code, K, cat);
    unknown = cc < 0;
    bad = false;
    if (cc < 0) return 0ull;
    unsigned long long k = (unsigned long long)((cc & 0xff) + 1) << 32;
    if (cc & 0x100) {      // thing: keep the instance id
        if (inst < 0 || inst > 0x7fffffffll) { bad = true; return 0ull; }
        k |= (unsigned long long)inst;
    }
    return k;
}

#define PQ_NO_SLOT 0xffffffffu

// insert of the per-image tables: 2+ slots per pixel, never full
struct PqInsert {
    static constexpr bool bounded = false;
    unsigned long long* keys;
    uint32_t C;
    __device__ __forceinline__ uint32_t operator()(unsigned long long key, unsigned) const {
        bool inserted;
        return pag_hash_insert(keys, C, key, &inserted);
    }
};

// warp-aggregated insert + count: lanes with equal nonzero key merge; the group's lowest lane inserts and adds.  Returns the slot
// (valid in lanes with key != 0; PQ_NO_SLOT when a bounded insert refused the key).  All 32 lanes call it.
// A: the area type (u32 per image, u64 per scene); Insert: (key, pixels) -> slot, or PQ_NO_SLOT when Insert::bounded.
template <typename A, typename Insert>
__device__ __forceinline__ uint32_t pq_count_t(const Insert& insert, A* __restrict__ area, A* __restrict__ voida, unsigned long long key,
                                               unsigned void_mask) {
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(peers) - 1;
    uint32_t slot = 0;
    if (key != 0ull && lane == leader) {
        slot = insert(key, (unsigned)__popc(peers));
        if (!Insert::bounded || slot != PQ_NO_SLOT) {
            atomicAdd(area + slot, (A)__popc(peers));
            if (voida != nullptr) {
                const unsigned nv = (unsigned)__popc(peers & void_mask);
                if (nv) atomicAdd(voida + slot, (A)nv);
            }
        }
    }
    return __shfl_sync(0xffffffffu, slot, leader);
}

__device__ __forceinline__ uint32_t pq_count(unsigned long long* __restrict__ keys, unsigned int* __restrict__ area,
                                             unsigned int* __restrict__ voida, uint32_t C, unsigned long long key, unsigned void_mask) {
    return pq_count_t(PqInsert{keys, C}, area, voida, key, void_mask);
}

__global__ void __launch_bounds__(PQ_HIST_BLOCK) pq_hist_kernel(const long long* __restrict__ preds, const long long* __restrict__ target,
                                                                int64_t P, uint32_t C, const int* __restrict__ cat_ids,
                                                                const int* __restrict__ cat_code, int K, int allow_unknown_preds,
                                                                PqTables t, long long* __restrict__ errors) {
    __shared__ int s_ids[PQ_MAX_CATEGORIES], s_code[PQ_MAX_CATEGORIES];
    for (int i = threadIdx.x; i < K; i += blockDim.x) { s_ids[i] = cat_ids[i]; s_code[i] = cat_code[i]; }
    __syncthreads();
    const int64_t b = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int64_t tb = b * (int64_t)C;
    const long long* pr = preds + b * P * 2;
    const long long* tg = target + b * P * 2;
    unsigned n_unknown = 0, n_bad = 0;
    // warp-uniform loop: every lane takes part in the match / shuffle, lanes past P carry void keys
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) * PQ_HIST_PIXELS_PER_THREAD;
    for (int it = 0; it < PQ_HIST_PIXELS_PER_THREAD; ++it) {
        const int64_t base = warp0 + it * 32;
        if (base >= P) break;
        const int64_t px = base + lane;
        unsigned long long kp = 0ull, kt = 0ull;
        bool p_void = false, t_void = false;
        if (px < P) {
            const longlong2 p = __ldcs(reinterpret_cast<const longlong2*>(pr) + px);
            const longlong2 q = __ldcs(reinterpret_cast<const longlong2*>(tg) + px);
            bool unk, bad;
            kp = pq_key(s_ids, s_code, K, p.x, p.y, unk, bad);
            p_void = kp == 0ull;
            n_unknown += (unk && !allow_unknown_preds);
            n_bad += bad;
            kt = pq_key(s_ids, s_code, K, q.x, q.y, unk, bad);
            t_void = kt == 0ull;
            n_bad += bad;
        }
        const unsigned pvoid_mask = __ballot_sync(0xffffffffu, px < P && p_void);
        const unsigned tvoid_mask = __ballot_sync(0xffffffffu, px < P && t_void);
        const uint32_t sp = pq_count(t.pred_key + tb, t.pred_area + tb, t.pred_void + tb, C, kp, tvoid_mask);
        const uint32_t st = pq_count(t.tgt_key + tb, t.tgt_area + tb, t.tgt_void + tb, C, kt, pvoid_mask);
        // pairs that can match: both non-void, same category
        const bool pair = kp != 0ull && kt != 0ull && (kp >> 32) == (kt >> 32);
        const unsigned long long kpair = pair ? ((unsigned long long)(sp + 1) << 32) | st : 0ull;
        pq_count(t.pair_key + tb, t.pair_cnt + tb, nullptr, C, kpair, 0u);
    }
    // error counters: one atomic per warp that saw any
    for (int o = 16; o > 0; o >>= 1) {
        n_unknown += __shfl_xor_sync(0xffffffffu, n_unknown, o);
        n_bad += __shfl_xor_sync(0xffffffffu, n_bad, o);
    }
    if (lane == 0) {
        if (n_unknown) atomicAdd(reinterpret_cast<unsigned long long*>(errors), (unsigned long long)n_unknown);
        if (n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(errors + 1), (unsigned long long)n_bad);
    }
}

#define PQ_MATCHED 0x80000000u

__global__ void __launch_bounds__(256) pq_match_kernel(PqTables t, int64_t n, uint32_t C, double* __restrict__ iou_sum,
                                                       long long* __restrict__ tp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long key = t.pair_key[i];
    if (key == 0ull) return;
    const int64_t tb = i - (i & (C - 1));      // first slot of this image's tables
    const int64_t sp = tb + (int64_t)(key >> 32) - 1, st = tb + (int64_t)(key & 0xffffffffull);
    const long long inter = t.pair_cnt[i];
    const long long ap = t.pred_area[sp] & ~PQ_MATCHED, at = t.tgt_area[st] & ~PQ_MATCHED;
    const long long uni = ap - (long long)t.pred_void[sp] + at - inter;
    if (2 * inter > uni) {
        const int c = (int)(t.pred_key[sp] >> 32) - 1;
        atomicAdd(iou_sum + c, (double)inter / (double)uni);
        atomicAdd(reinterpret_cast<unsigned long long*>(tp + c), 1ull);
        atomicOr(t.pred_area + sp, PQ_MATCHED);
        atomicOr(t.tgt_area + st, PQ_MATCHED);
    }
    t.pair_key[i] = 0ull;
    t.pair_cnt[i] = 0u;
}

// i < n: prediction slots (-> fp), n <= i < 2n: target slots (-> fn); the two tables are adjacent in the workspace
__global__ void __launch_bounds__(256) pq_unmatched_kernel(PqTables t, int64_t n, long long* __restrict__ fp, long long* __restrict__ fn) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * n) return;
    const unsigned long long key = t.pred_key[i];      // tgt_key == pred_key + n
    if (key == 0ull) return;
    unsigned int* area = t.pred_area + (i < n ? i : n + i);     // pred_area | pred_void | tgt_area | tgt_void
    unsigned int* voida = area + n;
    const unsigned a = *area;
    if (!(a & PQ_MATCHED) && 2ull * *voida <= (unsigned long long)a) {
        const int c = (int)(key >> 32) - 1;
        atomicAdd(reinterpret_cast<unsigned long long*>((i < n ? fp : fn) + c), 1ull);
    }
    t.pred_key[i] = 0ull;
    *area = 0u;
    *voida = 0u;
}

extern "C" int pag_pq_workspace(int64_t B, int64_t P, int64_t* bytes) {
    if (B < 1 || P < 1 || P > 0x40000000ll || bytes == nullptr) return PAG_ERR_ARG;
    *bytes = 44 * B * pag_hash_slots(P);
    return PAG_OK;
}

extern "C" int pag_pq_update(const int64_t* preds, const int64_t* target, int64_t B, int64_t P, const int32_t* cat_ids,
                             const int32_t* cat_code, int K, int allow_unknown_preds, void* workspace, int64_t workspace_bytes,
                             double* iou_sum, int64_t* counts, int64_t* errors, void* stream) {
    if (B < 1 || B > 65535 || P < 1 || P > 0x40000000ll || K < 1 || K > PQ_MAX_CATEGORIES) return PAG_ERR_ARG;
    if (!preds || !target || !cat_ids || !cat_code || !workspace || !iou_sum || !counts || !errors) return PAG_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(preds) | reinterpret_cast<uintptr_t>(target)) & 15) return PAG_ERR_ARG;
    const int64_t C = pag_hash_slots(P);
    if (workspace_bytes < 44 * B * C || (reinterpret_cast<uintptr_t>(workspace) & 15)) return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = B * C;
    const PqTables t = pq_tables(workspace, n);
    long long* cnt = reinterpret_cast<long long*>(counts);      // tp | fp | fn, K each
    const int64_t per_block = (int64_t)PQ_HIST_BLOCK * PQ_HIST_PIXELS_PER_THREAD;
    const dim3 grid((unsigned)((P + per_block - 1) / per_block), (unsigned)B);
    pq_hist_kernel<<<grid, PQ_HIST_BLOCK, 0, s>>>(reinterpret_cast<const long long*>(preds), reinterpret_cast<const long long*>(target), P,
                                                  (uint32_t)C, cat_ids, cat_code, K, allow_unknown_preds, t,
                                                  reinterpret_cast<long long*>(errors));
    PAG_LAUNCH_CHECK();
    pq_match_kernel<<<pag_grid(n, 256), 256, 0, s>>>(t, n, (uint32_t)C, iou_sum, cnt);
    PAG_LAUNCH_CHECK();
    pq_unmatched_kernel<<<pag_grid(2 * n, 256), 256, 0, s>>>(t, n, cnt + K, cnt + 2 * K);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// ---------------------------------------------------------------------------------------------------------------------------
// Scene-level panoptic quality: one segment per (category, instance) across every frame of a sequence.
//
// The result after updates with frames F1..Fn is the per-image result for ONE image made of all their pixels, so the three tables
// persist across updates instead of being scanned and cleared per image.  They are sized by a capacity (distinct keys per table),
// not by the data, so the insert is bounded: a table admits at most `capacity` keys and refuses the pixels of any further key
// (counted per table, raised by the caller).  C = pag_hash_slots(capacity) >= 2 * capacity, so no table is ever more than half full
// and every probe loop ends.  Workspace (zero-filled by the caller once; it persists across updates):
//   u64 pred_key[C] | u64 tgt_key[C] | u64 pair_key[C] | u64 pred_area[C] | u64 pred_void[C] | u64 tgt_area[C] | u64 tgt_void[C]
//   | u64 pair_cnt[C] | u64 counters[16]                                                        = 64 * C + 128 bytes
// counters: reserved[3] (keys admitted plus inserts in flight) | used[3] (keys in the table) | refused[3] (pixels refused), in table
// order pred | tgt | pair.  Keys as per image; a pair is inserted only when both of its segments are present.
//   update  one histogram launch over all B*P pixels (pq_key, pq_count_t with u64 areas and the bounded insert)
//   stats   match over the pair slots (sets bit 63 of matched segment areas), then unmatched over the segment slots (counts FP /
//           FN and clears that bit): the tables are left as found, so stats can run at any point of a sequence
//   merge   another rank's tables into the local ones; pair keys are translated through that rank's segment keys
#define SCENE_COUNTERS 16
#define SCENE_MATCHED 0x8000000000000000ull

struct ScenePqTables {
    unsigned long long *pred_key, *tgt_key, *pair_key;
    unsigned long long *pred_area, *pred_void, *tgt_area, *tgt_void, *pair_cnt;
    unsigned long long *reserved, *used, *refused;
};

static ScenePqTables scene_tables(void* ws, int64_t C) {
    unsigned long long* k = reinterpret_cast<unsigned long long*>(ws);
    ScenePqTables t;
    t.pred_key = k;
    t.tgt_key = k + C;
    t.pair_key = k + 2 * C;
    t.pred_area = k + 3 * C;
    t.pred_void = k + 4 * C;
    t.tgt_area = k + 5 * C;
    t.tgt_void = k + 6 * C;
    t.pair_cnt = k + 7 * C;
    t.reserved = k + 8 * C;
    t.used = t.reserved + 3;
    t.refused = t.reserved + 6;
    return t;
}

__device__ __forceinline__ unsigned long long ld_volatile(const unsigned long long* p) {
    return *reinterpret_cast<const volatile unsigned long long*>(p);
}

// slot of `key` in table[C], inserted if absent and fewer than `limit` keys are in the table; PQ_NO_SLOT when the table is full
// and the key absent.  A creating insert reserves a count before its CAS (a CAS loop that never takes `reserved` past `limit`, so
// threads that find no room only read it) and releases it on a lost CAS; `used` counts keys only after their CAS.  No room while
// used < limit means reservations of CASes in flight: they resolve without waiting on anyone, so the slot is read again.  With
// used >= limit no key can be added any more: a slot still empty after the fence means the key is absent for good.
__device__ __forceinline__ uint32_t scene_insert(unsigned long long* __restrict__ table, uint32_t C, unsigned long long key,
                                                 unsigned long long* reserved, unsigned long long* used, unsigned long long limit) {
    uint32_t s = pag_hash64(key) & (C - 1);
    while (true) {
        unsigned long long cur = ld_volatile(table + s);
        if (cur == 0ull) {
            unsigned long long r = ld_volatile(reserved);
            bool admitted = false;
            while (r < limit) {
                const unsigned long long old = atomicCAS(reserved, r, r + 1);
                if (old == r) { admitted = true; break; }
                r = old;
            }
            if (admitted) {
                cur = atomicCAS(table + s, 0ull, key);
                if (cur == 0ull) {
                    __threadfence();
                    atomicAdd(used, 1ull);
                    return s;
                }
                atomicAdd(reserved, ~0ull);      // lost the CAS: release
            } else {
                if (ld_volatile(used) < limit) {
                    __nanosleep(64);
                    continue;
                }
                __threadfence();
                cur = ld_volatile(table + s);
                if (cur == 0ull) return PQ_NO_SLOT;
            }
        }
        if (cur == key) return s;
        s = (s + 1) & (C - 1);
    }
}

// slot of `key`, or PQ_NO_SLOT if absent (tables not written concurrently)
__device__ __forceinline__ uint32_t scene_find(const unsigned long long* __restrict__ table, uint32_t C, unsigned long long key) {
    uint32_t s = pag_hash64(key) & (C - 1);
    while (true) {
        const unsigned long long cur = table[s];
        if (cur == key) return s;
        if (cur == 0ull) return PQ_NO_SLOT;
        s = (s + 1) & (C - 1);
    }
}

struct SceneInsert {
    static constexpr bool bounded = true;
    unsigned long long* keys;
    uint32_t C;
    unsigned long long *reserved, *used, *refused;
    unsigned long long limit;
    __device__ __forceinline__ uint32_t operator()(unsigned long long key, unsigned n) const {
        const uint32_t s = scene_insert(keys, C, key, reserved, used, limit);
        if (s == PQ_NO_SLOT) atomicAdd(refused, (unsigned long long)n);
        return s;
    }
};

__device__ __forceinline__ SceneInsert scene_inserter(const ScenePqTables& t, int table, uint32_t C, unsigned long long limit) {
    unsigned long long* keys = table == 0 ? t.pred_key : table == 1 ? t.tgt_key : t.pair_key;
    return SceneInsert{keys, C, t.reserved + table, t.used + table, t.refused + table, limit};
}

__global__ void __launch_bounds__(PQ_HIST_BLOCK) scene_pq_hist_kernel(const long long* __restrict__ preds, const long long* __restrict__ target,
                                                                      int64_t N, uint32_t C, unsigned long long limit,
                                                                      const int* __restrict__ cat_ids, const int* __restrict__ cat_code, int K,
                                                                      int allow_unknown_preds, ScenePqTables t, long long* __restrict__ errors) {
    __shared__ int s_ids[PQ_MAX_CATEGORIES], s_code[PQ_MAX_CATEGORIES];
    for (int i = threadIdx.x; i < K; i += blockDim.x) { s_ids[i] = cat_ids[i]; s_code[i] = cat_code[i]; }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const SceneInsert ins_p = scene_inserter(t, 0, C, limit), ins_t = scene_inserter(t, 1, C, limit), ins_pair = scene_inserter(t, 2, C, limit);
    unsigned n_unknown = 0, n_bad = 0;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) * PQ_HIST_PIXELS_PER_THREAD;
    for (int it = 0; it < PQ_HIST_PIXELS_PER_THREAD; ++it) {
        const int64_t base = warp0 + it * 32;
        if (base >= N) break;
        const int64_t px = base + lane;
        unsigned long long kp = 0ull, kt = 0ull;
        bool p_void = false, t_void = false;
        if (px < N) {
            const longlong2 p = __ldcs(reinterpret_cast<const longlong2*>(preds) + px);
            const longlong2 q = __ldcs(reinterpret_cast<const longlong2*>(target) + px);
            bool unk, bad;
            kp = pq_key(s_ids, s_code, K, p.x, p.y, unk, bad);
            p_void = kp == 0ull;
            n_unknown += (unk && !allow_unknown_preds);
            n_bad += bad;
            kt = pq_key(s_ids, s_code, K, q.x, q.y, unk, bad);
            t_void = kt == 0ull;
            n_bad += bad;
        }
        const unsigned pvoid_mask = __ballot_sync(0xffffffffu, px < N && p_void);
        const unsigned tvoid_mask = __ballot_sync(0xffffffffu, px < N && t_void);
        const uint32_t sp = pq_count_t(ins_p, t.pred_area, t.pred_void, kp, tvoid_mask);
        const uint32_t st = pq_count_t(ins_t, t.tgt_area, t.tgt_void, kt, pvoid_mask);
        const bool pair = kp != 0ull && kt != 0ull && (kp >> 32) == (kt >> 32) && sp != PQ_NO_SLOT && st != PQ_NO_SLOT;
        const unsigned long long kpair = pair ? ((unsigned long long)(sp + 1) << 32) | st : 0ull;
        pq_count_t(ins_pair, t.pair_cnt, (unsigned long long*)nullptr, kpair, 0u);
    }
    for (int o = 16; o > 0; o >>= 1) {
        n_unknown += __shfl_xor_sync(0xffffffffu, n_unknown, o);
        n_bad += __shfl_xor_sync(0xffffffffu, n_bad, o);
    }
    if (lane == 0) {
        if (n_unknown) atomicAdd(reinterpret_cast<unsigned long long*>(errors), (unsigned long long)n_unknown);
        if (n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(errors + 1), (unsigned long long)n_bad);
    }
}

__global__ void __launch_bounds__(256) scene_pq_match_kernel(ScenePqTables t, uint32_t C, double* __restrict__ iou_sum,
                                                             long long* __restrict__ tp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C) return;
    const unsigned long long key = t.pair_key[i];
    if (key == 0ull) return;
    const int64_t sp = (int64_t)(key >> 32) - 1, st = (int64_t)(key & 0xffffffffull);
    const unsigned long long inter = t.pair_cnt[i];
    const unsigned long long ap = t.pred_area[sp] & ~SCENE_MATCHED, at = t.tgt_area[st] & ~SCENE_MATCHED;
    const unsigned long long uni = ap - t.pred_void[sp] + at - inter;
    if (2 * inter > uni) {
        const int c = (int)(t.pred_key[sp] >> 32) - 1;
        atomicAdd(iou_sum + c, (double)inter / (double)uni);
        atomicAdd(reinterpret_cast<unsigned long long*>(tp + c), 1ull);
        atomicOr(t.pred_area + sp, SCENE_MATCHED);
        atomicOr(t.tgt_area + st, SCENE_MATCHED);
    }
}

// i < C: prediction slots (-> fp), C <= i < 2C: target slots (-> fn).  Clears the matched bit the match kernel set.
__global__ void __launch_bounds__(256) scene_pq_unmatched_kernel(ScenePqTables t, uint32_t C, long long* __restrict__ fp,
                                                                 long long* __restrict__ fn) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * (int64_t)C) return;
    const unsigned long long key = t.pred_key[i];      // tgt_key == pred_key + C
    if (key == 0ull) return;
    unsigned long long* area = t.pred_area + (i < C ? i : C + i);      // pred_area | pred_void | tgt_area | tgt_void
    const unsigned long long a = *area;
    if (a & SCENE_MATCHED) {
        *area = a & ~SCENE_MATCHED;
    } else if (2 * area[C] <= a) {
        const int c = (int)(key >> 32) - 1;
        atomicAdd(reinterpret_cast<unsigned long long*>((i < C ? fp : fn) + c), 1ull);
    }
}

// segments of another rank's tables (r) into the local ones (t); i < C prediction, C <= i < 2C target slots.  Thread 0 adds r's
// refused counts.
__global__ void __launch_bounds__(256) scene_pq_merge_segments_kernel(ScenePqTables t, ScenePqTables r, uint32_t C, unsigned long long limit) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0)
        for (int k = 0; k < 3; ++k)
            if (r.refused[k]) atomicAdd(t.refused + k, r.refused[k]);
    if (i >= 2 * (int64_t)C) return;
    const unsigned long long key = r.pred_key[i];
    if (key == 0ull) return;
    const int table = i < C ? 0 : 1;
    const int64_t j = i < C ? i : C + i;      // area index, as in the unmatched kernel
    const unsigned long long area = r.pred_area[j] & ~SCENE_MATCHED, voida = r.pred_area[j + C];
    const SceneInsert ins = scene_inserter(t, table, C, limit);
    const uint32_t s = ins(key, 0u);
    if (s == PQ_NO_SLOT) {
        atomicAdd(t.refused + table, area);
        return;
    }
    const int64_t ls = table == 0 ? s : 2 * (int64_t)C + s;
    atomicAdd(t.pred_area + ls, area);
    if (voida) atomicAdd(t.pred_area + ls + C, voida);
}

// pairs of r: slot numbers differ between ranks, so each pair is translated through r's segment keys to the local slots.  A pair
// with a refused segment was counted in that segment's table.
__global__ void __launch_bounds__(256) scene_pq_merge_pairs_kernel(ScenePqTables t, ScenePqTables r, uint32_t C, unsigned long long limit) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C) return;
    const unsigned long long key = r.pair_key[i];
    if (key == 0ull) return;
    const uint32_t sp = scene_find(t.pred_key, C, r.pred_key[(key >> 32) - 1]);
    const uint32_t st = scene_find(t.tgt_key, C, r.tgt_key[key & 0xffffffffull]);
    if (sp == PQ_NO_SLOT || st == PQ_NO_SLOT) return;
    const unsigned long long cnt = r.pair_cnt[i];
    const uint32_t s = scene_inserter(t, 2, C, limit)(((unsigned long long)(sp + 1) << 32) | st, 0u);
    if (s == PQ_NO_SLOT) atomicAdd(t.refused + 2, cnt);
    else atomicAdd(t.pair_cnt + s, cnt);
}

#define SCENE_MAX_CAPACITY (1ll << 26)

static int64_t scene_bytes(int64_t C) { return 64 * C + 8 * SCENE_COUNTERS; }

extern "C" int pag_scene_pq_workspace(int64_t capacity, int64_t* bytes) {
    if (capacity < 1 || capacity > SCENE_MAX_CAPACITY || bytes == nullptr) return PAG_ERR_ARG;
    *bytes = scene_bytes(pag_hash_slots(capacity));
    return PAG_OK;
}

static bool scene_ws_ok(const void* ws, int64_t capacity, int64_t bytes) {
    return ws != nullptr && capacity >= 1 && capacity <= SCENE_MAX_CAPACITY && !(reinterpret_cast<uintptr_t>(ws) & 15) &&
           bytes >= scene_bytes(pag_hash_slots(capacity));
}

extern "C" int pag_scene_pq_update(const int64_t* preds, const int64_t* target, int64_t N, const int32_t* cat_ids, const int32_t* cat_code,
                                   int K, int allow_unknown_preds, void* workspace, int64_t capacity, int64_t workspace_bytes,
                                   int64_t* errors, void* stream) {
    if (N < 1 || K < 1 || K > PQ_MAX_CATEGORIES || !preds || !target || !cat_ids || !cat_code || !errors) return PAG_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(preds) | reinterpret_cast<uintptr_t>(target)) & 15) return PAG_ERR_ARG;
    if (!scene_ws_ok(workspace, capacity, workspace_bytes)) return PAG_ERR_ARG;
    const int64_t per_block = (int64_t)PQ_HIST_BLOCK * PQ_HIST_PIXELS_PER_THREAD;
    const int64_t blocks = (N + per_block - 1) / per_block;
    if (blocks > 0x7fffffffll) return PAG_ERR_ARG;
    const int64_t C = pag_hash_slots(capacity);
    scene_pq_hist_kernel<<<(unsigned)blocks, PQ_HIST_BLOCK, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(preds), reinterpret_cast<const long long*>(target), N, (uint32_t)C, (unsigned long long)capacity,
        cat_ids, cat_code, K, allow_unknown_preds, scene_tables(workspace, C), reinterpret_cast<long long*>(errors));
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

extern "C" int pag_scene_pq_stats(void* workspace, int64_t capacity, int64_t workspace_bytes, int K, double* iou_sum, int64_t* counts,
                                  void* stream) {
    if (!scene_ws_ok(workspace, capacity, workspace_bytes) || K < 1 || K > PQ_MAX_CATEGORIES || !iou_sum || !counts) return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t C = pag_hash_slots(capacity);
    const ScenePqTables t = scene_tables(workspace, C);
    long long* cnt = reinterpret_cast<long long*>(counts);      // tp | fp | fn, K each
    scene_pq_match_kernel<<<pag_grid(C, 256), 256, 0, s>>>(t, (uint32_t)C, iou_sum, cnt);
    PAG_LAUNCH_CHECK();
    scene_pq_unmatched_kernel<<<pag_grid(2 * C, 256), 256, 0, s>>>(t, (uint32_t)C, cnt + K, cnt + 2 * K);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

extern "C" int pag_scene_pq_merge(void* workspace, const void* other, int64_t capacity, int64_t workspace_bytes, void* stream) {
    if (!scene_ws_ok(workspace, capacity, workspace_bytes) || !scene_ws_ok(other, capacity, workspace_bytes) || workspace == other)
        return PAG_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t C = pag_hash_slots(capacity);
    const ScenePqTables t = scene_tables(workspace, C), r = scene_tables(const_cast<void*>(other), C);
    scene_pq_merge_segments_kernel<<<pag_grid(2 * C, 256), 256, 0, s>>>(t, r, (uint32_t)C, (unsigned long long)capacity);
    PAG_LAUNCH_CHECK();
    scene_pq_merge_pairs_kernel<<<pag_grid(C, 256), 256, 0, s>>>(t, r, (uint32_t)C, (unsigned long long)capacity);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}
