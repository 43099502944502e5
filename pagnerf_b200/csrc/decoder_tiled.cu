// Exact-FP32 decoders for INFERENCE, register-tiled (forward only).
//
// decoder.cu keeps one sample per thread: every FFMA needs its own shared-memory weight operand and the instance head's
// 200 logits per sample go through global memory twice (logits -> softmax -> composite kernel).  ncu on the 1 MP frame
// (profiles/r02_ncu_tiled.md): pan_fwd 120 ms, dc_fwd 36 ms of a 186 ms frame, FFMA pipe 16-23 % busy.  Here a group of threads
// owns a 64- or 128-sample tile held k-major in shared memory ([k][ROWS+4] floats) and every thread accumulates an 8-sample x
// 4-output (8 x 13 for the instance logits) register block -- 16 (52) packed FFMA2 per 3 (9) LDS -- and the instance / semantic
// probabilities are composited straight from registers into the per-ray maps (red.add), never written per sample.
// Arithmetic order per output is the same as decoder.cu (bias, then k ascending, fmaf), so hidden activations (and the density) are
// bit-identical to that path; the composited sums differ in association only, the colour through the view embedding's
// double-angle recurrence (<= 1e-6).
//
// Reference semantics: pc_nerf/panoptic_nef.py:253-363 (decoders), tracers/panoptic_packed_rf_tracer.py:148-178
// (semantics / instance maps = alpha * sum_s w_s p_s with detached weights).
#include "decoder_common.cuh"

// ROWS = samples per tile; a tile is worked by a GROUP of 2 * ROWS threads with its own named barrier; a CTA holds NG groups that
// walk their own tiles and share the staged weights (one group's staging / epilogue / barrier wait is filled by the others' FMA
// phases).  Measured on the 1 MP frame: density + colour 21.0 ms with 1 x 128 rows, 18.7 ms with 3 x 64; the panoptic heads (whose
// weights leave room for two 64-row groups only) 35.9 ms with 1 x 128, 38.0 ms with 2 x 64 (36.6 vs 36.7 ms after the class-pair
// loads: decoupling the phases is not what the heads kernel lacks).
#define TL_LDA(ROWS) ((ROWS) + 4)
#define TL_BUF(ROWS) (H * TL_LDA(ROWS))   // one activation buffer [64][ROWS+4]; also holds a raw [ROWS][IN <= 64] row block
#define PAN_ROWS 128
#define PAN_MAXG 1
#define DC_ROWS 64
#define DC_MAXG 3
#define TL_CIP 208          // instance classes padded: 16 lanes x 13

// packed FP32 FMA (sm_100: FFMA2) -- c.x = a.x * w + c.x, c.y = a.y * w + c.y, each rounded like fmaf.  One issue slot per two
// FMAs: with scalar FFMA every LDS / address instruction takes an issue slot away from the FMA pipe (ncu: 54 % issue-active, FMA 41 %).
__device__ __forceinline__ void ffma2(float2& c, const float2 a, const float w) {
    unsigned long long cc = *reinterpret_cast<unsigned long long*>(&c);
    const float2 w2 = make_float2(w, w);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(cc) : "l"(*reinterpret_cast<const unsigned long long*>(&a)),
        "l"(*reinterpret_cast<const unsigned long long*>(&w2)));
    c = *reinterpret_cast<float2*>(&cc);
}
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int ROWS>
__device__ __forceinline__ void group_sync(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(2 * ROWS) : "memory"); }

// D[o][s] = relu(b[o] + sum_k WT[k][o] A[k][s]) for o < 64, s < ROWS; A, D k-major with stride TL_LDA(ROWS); WT [K][64].
// thread = 8 samples x 4 outputs: 16 FFMA2 per 3 LDS.128
template <int ROWS>
__device__ __forceinline__ void tl_layer64(const float* __restrict__ A, int K, const float* __restrict__ WT,
                                           const float* __restrict__ b, float* __restrict__ D, int tid) {
    const int og = tid & 15, sg = tid >> 4;
    float2 acc[4][4];
    {
        const float4 bb = *reinterpret_cast<const float4*>(b + og * 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            acc[j][0] = make_float2(bb.x, bb.x); acc[j][1] = make_float2(bb.y, bb.y);
            acc[j][2] = make_float2(bb.z, bb.z); acc[j][3] = make_float2(bb.w, bb.w);
        }
    }
    const float* a = A + sg * 8;
    const float* w = WT + og * 4;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const float4 a0 = *reinterpret_cast<const float4*>(a + k * TL_LDA(ROWS));
        const float4 a1 = *reinterpret_cast<const float4*>(a + k * TL_LDA(ROWS) + 4);
        const float4 ww = *reinterpret_cast<const float4*>(w + k * 64);
        const float2 av[4] = {make_float2(a0.x, a0.y), make_float2(a0.z, a0.w), make_float2(a1.x, a1.y), make_float2(a1.z, a1.w)};
        const float wv[4] = {ww.x, ww.y, ww.z, ww.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) ffma2(acc[j][i], av[j], wv[i]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float* d = D + (og * 4 + i) * TL_LDA(ROWS) + sg * 8;
        *reinterpret_cast<float4*>(d) = make_float4(fmaxf(acc[0][i].x, 0.f), fmaxf(acc[0][i].y, 0.f), fmaxf(acc[1][i].x, 0.f), fmaxf(acc[1][i].y, 0.f));
        *reinterpret_cast<float4*>(d + 4) = make_float4(fmaxf(acc[2][i].x, 0.f), fmaxf(acc[2][i].y, 0.f), fmaxf(acc[3][i].x, 0.f), fmaxf(acc[3][i].y, 0.f));
    }
}

// Output head fused with its compositing.  thread = 8 consecutive samples (sg) x NC classes: NC/2 adjacent pairs
// {32 ip + 2 cg, + 1} (weights by LDS.64: a 16-lane group reads one 128-byte line; composited with red.v2) and, for odd NC, the
// single class 32 (NC/2) + cg.  logits z = b + WT^T h (WT [64][16*NC]);  p = softmax ? softmax(z * scale) : z * scale;
// out[ray][c] += coef_s * p_s[c], summed over the thread's samples with one red per (ray run, class pair).
template <int NC>
__device__ __forceinline__ int tl_class(int i, int cg) {
    constexpr int NP = NC / 2;
    return i < 2 * NP ? (i >> 1) * 32 + 2 * cg + (i & 1) : NP * 32 + cg;
}
template <int NC>
__device__ __forceinline__ void tl_flush(float* __restrict__ row, int C, int cg, const float (&run)[NC]) {
    constexpr int NP = NC / 2;
    if ((C & 1) == 0) {                    // even class count: rows stay 8-byte aligned
#pragma unroll
        for (int ip = 0; ip < NP; ++ip)
            if (ip * 32 + 2 * cg < C) red_add_f32x2(row + ip * 32 + 2 * cg, run[2 * ip], run[2 * ip + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < 2 * NP; ++i)
            if (tl_class<NC>(i, cg) < C) red_add_f32(row + tl_class<NC>(i, cg), run[i]);
    }
    if (NC & 1)
        if (NP * 32 + cg < C) red_add_f32(row + NP * 32 + cg, run[NC - 1]);
}
template <int NC, int ROWS>
__device__ __forceinline__ void tl_head(const float* __restrict__ A, const float* __restrict__ WT, const float* __restrict__ b, int C,
                                        bool softmax, float scale, const float* __restrict__ coef, const int* __restrict__ rr,
                                        float* __restrict__ out, int tid) {
    constexpr int NP = NC / 2;
    const int cg = tid & 15, sg = tid >> 4;
    float2 acc[4][NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        const float bv = b[tl_class<NC>(i, cg)];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j][i] = make_float2(bv, bv);
    }
    {
        const float* a = A + sg * 8;
        const float* wt = WT + 2 * cg;
        const float* wl = WT + NP * 32 + cg;
#pragma unroll 2
        for (int k = 0; k < H; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(a + k * TL_LDA(ROWS));
            const float4 a1 = *reinterpret_cast<const float4*>(a + k * TL_LDA(ROWS) + 4);
            const float2 av[4] = {make_float2(a0.x, a0.y), make_float2(a0.z, a0.w), make_float2(a1.x, a1.y), make_float2(a1.z, a1.w)};
#pragma unroll
            for (int ip = 0; ip < NP; ++ip) {
                const float2 wv = *reinterpret_cast<const float2*>(wt + k * (16 * NC) + ip * 32);
#pragma unroll
                for (int j = 0; j < 4; ++j) { ffma2(acc[j][2 * ip], av[j], wv.x); ffma2(acc[j][2 * ip + 1], av[j], wv.y); }
            }
            if (NC & 1) {
                const float wv = wl[k * (16 * NC)];
#pragma unroll
                for (int j = 0; j < 4; ++j) ffma2(acc[j][NC - 1], av[j], wv);
            }
        }
    }
    const float4 c0 = *reinterpret_cast<const float4*>(coef + sg * 8), c1 = *reinterpret_cast<const float4*>(coef + sg * 8 + 4);
    float cf[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
    if (softmax) {
        const float sc2 = scale * 1.4426950408889634f;      // exp((z - mx) * scale) = 2^((z - mx) * scale * log2 e)
        float mx[8], sum[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) mx[j] = -INFINITY;
#pragma unroll
        for (int i = 0; i < NC; ++i)
            if (tl_class<NC>(i, cg) < C) {
#pragma unroll
                for (int j = 0; j < 4; ++j) { mx[2 * j] = fmaxf(mx[2 * j], acc[j][i].x); mx[2 * j + 1] = fmaxf(mx[2 * j + 1], acc[j][i].y); }
            }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) mx[j] = fmaxf(mx[j], __shfl_xor_sync(0xffffffffu, mx[j], o));
            sum[j] = 0.f;
        }
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const bool on = tl_class<NC>(i, cg) < C;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[j][i].x = on ? ex2_approx((acc[j][i].x - mx[2 * j]) * sc2) : 0.f;
                acc[j][i].y = on ? ex2_approx((acc[j][i].y - mx[2 * j + 1]) * sc2) : 0.f;
                sum[2 * j] += acc[j][i].x; sum[2 * j + 1] += acc[j][i].y;
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) sum[j] += __shfl_xor_sync(0xffffffffu, sum[j], o);
            cf[j] *= 1.f / sum[j];
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) cf[j] *= scale;
    }
    // segmented sum over the thread's 8 consecutive samples
    const int4 r0 = *reinterpret_cast<const int4*>(rr + sg * 8), r1 = *reinterpret_cast<const int4*>(rr + sg * 8 + 4);
    const int rv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
    float run[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) run[i] = acc[0][i].x * cf[0];
    int rprev = rv[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) {
        if (rv[j] != rprev) {              // uniform over the 16 lanes of this sample group
            tl_flush<NC>(out + (size_t)rprev * C, C, cg, run);
#pragma unroll
            for (int i = 0; i < NC; ++i) run[i] = 0.f;
            rprev = rv[j];
        }
#pragma unroll
        for (int i = 0; i < NC; ++i) run[i] = fmaf((j & 1) ? acc[j >> 1][i].y : acc[j >> 1][i].x, cf[j], run[i]);
    }
    tl_flush<NC>(out + (size_t)rprev * C, C, cg, run);
}

// WT[k][o] = k < IN ? W[o][k] : 0 for o < OUT, zero for OUT <= o < OUTP  (W: torch Linear [OUT][IN])
__device__ __forceinline__ void tl_stage_wt(float* __restrict__ WT, const float* __restrict__ W, int OUT, int OUTP, int IN, int KP) {
    for (int i = threadIdx.x; i < KP * OUTP; i += blockDim.x) {
        const int k = i / OUTP, o = i - k * OUTP;
        WT[i] = (o < OUT && k < IN) ? __ldg(W + (size_t)o * IN + k) : 0.f;
    }
}
__device__ __forceinline__ void tl_stage_b(float* __restrict__ dst, const float* __restrict__ b, int n, int np) {
    for (int i = threadIdx.x; i < np; i += blockDim.x) dst[i] = i < n ? __ldg(b + i) : 0.f;
}

// asynchronous copy of rows [row0, row0 + ROWS) x IN (one contiguous span) into a raw shared-memory block [ROWS][IN]
template <int ROWS>
__device__ __forceinline__ void tl_fetch_rows(float* __restrict__ raw, const float* __restrict__ src, int IN, int64_t row0, int64_t M, int gt) {
    const int64_t left = M - row0;
    const int nch = (int)(left >= ROWS ? ROWS : (left > 0 ? left : 0)) * (IN >> 2);
    const float* g = src + row0 * IN;
    for (int c = gt; c < nch; c += (2 * ROWS)) cp_async16(raw + 4 * c, g + 4 * c);
}
// XT[k][r] = (rawA[r][k] + rawB[r][k]) * lodw[k], rows past M zero
template <int ROWS>
__device__ __forceinline__ void tl_transpose_x(float* __restrict__ XT, const float* __restrict__ rawA, const float* __restrict__ rawB,
                                               const float* __restrict__ lodw, int IN, int64_t row0, int64_t M, int gt) {
    const int nq = IN >> 2;
    for (int g = gt; g < ROWS * nq; g += (2 * ROWS)) {
        const int r = g / nq, q = g - r * nq;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + r < M) {
            v = *reinterpret_cast<const float4*>(rawA + 4 * g);
            if (rawB) { const float4 u = *reinterpret_cast<const float4*>(rawB + 4 * g); v.x += u.x; v.y += u.y; v.z += u.z; v.w += u.w; }
            if (lodw) { const float4 l = ldg4(lodw + 4 * q); v.x *= l.x; v.y *= l.y; v.z *= l.z; v.w *= l.w; }
        }
        float* d = XT + (4 * q) * TL_LDA(ROWS) + r;
        d[0] = v.x; d[TL_LDA(ROWS)] = v.y; d[2 * TL_LDA(ROWS)] = v.z; d[3 * TL_LDA(ROWS)] = v.w;
    }
}

struct TlPanLayout { int Ws1T, bs1, Ws2T, bs2, Wi1T, bi1, Wi2T, bi2, Wi3T, bi3, groups, gstride, total; };
// per group: P, Q, R activation buffers + coef[PAN_ROWS] + ray[PAN_ROWS]
__host__ __device__ inline TlPanLayout tl_pan_layout(int IN, int NG) {
    TlPanLayout l; int o = 0;
    l.Ws1T = o; o += IN * H; l.bs1 = o; o += H; l.Ws2T = o; o += H * 16; l.bs2 = o; o += 16;
    l.Wi1T = o; o += IN * H; l.bi1 = o; o += H; l.Wi2T = o; o += H * H; l.bi2 = o; o += H;
    l.Wi3T = o; o += H * TL_CIP; l.bi3 = o; o += TL_CIP;
    l.groups = o; l.gstride = 3 * TL_BUF(PAN_ROWS) + 2 * PAN_ROWS;
    l.total = o + NG * l.gstride;
    return l;
}

// Per tile and group (4 group barriers):  raw rows (cp.async, issued one tile ahead) in P, Q -> X k-major in R | first layers R -> P
// (semantic hidden), R -> Q (instance hidden 1) | semantic head from P, instance layer 2 Q -> R | next tile's raw rows -> P, Q in
// flight while the instance head (55 % of the arithmetic) runs from R.
__global__ void __launch_bounds__(PAN_MAXG * (2 * PAN_ROWS), 1)
pan_comp_fwd_tiled_kernel(const float* __restrict__ feats, const float* __restrict__ dfeats, const float* __restrict__ lodw,
                          int64_t M, int IN, PanParams p, int Cs, int Ci, int sem_softmax, int inst_softmax, float inv_temp,
                          const float* __restrict__ w, const float* __restrict__ alpha, const int64_t* __restrict__ ridx,
                          float* __restrict__ out_sem, float* __restrict__ out_inst) {
    extern __shared__ __align__(16) float smem[];
    const int NG = blockDim.x / (2 * PAN_ROWS), grp = threadIdx.x / (2 * PAN_ROWS), gt = threadIdx.x - grp * (2 * PAN_ROWS);
    const TlPanLayout l = tl_pan_layout(IN, NG);
    float* P = smem + l.groups + grp * l.gstride;
    float *Q = P + TL_BUF(PAN_ROWS), *R = Q + TL_BUF(PAN_ROWS), *coef = R + TL_BUF(PAN_ROWS);
    int* rr = reinterpret_cast<int*>(coef + PAN_ROWS);
    const int64_t ntiles = (M + PAN_ROWS - 1) / PAN_ROWS;
    const int64_t tile0 = (int64_t)blockIdx.x * NG + grp, tstride = (int64_t)gridDim.x * NG;
    int ray_n = 0;
    float coef_n = 0.f;
    auto fetch = [&](int64_t tile) {      // raw rows + this thread's compositing coefficient of `tile`
        tl_fetch_rows<PAN_ROWS>(P, feats, IN, tile * PAN_ROWS, M, gt);
        if (dfeats) tl_fetch_rows<PAN_ROWS>(Q, dfeats, IN, tile * PAN_ROWS, M, gt);
        cp_async_commit();
        if (gt < PAN_ROWS) {
            const int64_t m = tile * PAN_ROWS + gt;
            const bool valid = m < M;
            const int64_t ray = ridx[valid ? m : M - 1];
            ray_n = (int)ray;
            coef_n = valid ? __ldg(alpha + ray) * __ldg(w + m) : 0.f;
        }
    };
    if (tile0 < ntiles) fetch(tile0);
    if (Cs > 0) {
        tl_stage_wt(smem + l.Ws1T, p.Ws1, H, H, IN, IN); tl_stage_b(smem + l.bs1, p.bs1, H, H);
        tl_stage_wt(smem + l.Ws2T, p.Ws2, Cs, 16, H, H); tl_stage_b(smem + l.bs2, p.bs2, Cs, 16);
    }
    if (Ci > 0) {
        tl_stage_wt(smem + l.Wi1T, p.Wi1, H, H, IN, IN); tl_stage_b(smem + l.bi1, p.bi1, H, H);
        tl_stage_wt(smem + l.Wi2T, p.Wi2, H, H, H, H); tl_stage_b(smem + l.bi2, p.bi2, H, H);
        tl_stage_wt(smem + l.Wi3T, p.Wi3, Ci, TL_CIP, H, H); tl_stage_b(smem + l.bi3, p.bi3, Ci, TL_CIP);
    }
    __syncthreads();                       // weights staged (the only block-wide barrier)
    for (int64_t tile = tile0; tile < ntiles; tile += tstride) {
        const int64_t row0 = tile * PAN_ROWS;
        cp_async_wait_all();
        group_sync<PAN_ROWS>(grp);                   // raw rows landed; the previous tile's instance head is done with R / coef / rr
        if (gt < PAN_ROWS) { rr[gt] = ray_n; coef[gt] = coef_n; }
        tl_transpose_x<PAN_ROWS>(R, P, dfeats ? Q : nullptr, lodw, IN, row0, M, gt);
        group_sync<PAN_ROWS>(grp);
        if (Cs > 0) tl_layer64<PAN_ROWS>(R, IN, smem + l.Ws1T, smem + l.bs1, P, gt);
        if (Ci > 0) tl_layer64<PAN_ROWS>(R, IN, smem + l.Wi1T, smem + l.bi1, Q, gt);
        group_sync<PAN_ROWS>(grp);
        if (Cs > 0) tl_head<1, PAN_ROWS>(P, smem + l.Ws2T, smem + l.bs2, Cs, sem_softmax != 0, 1.f, coef, rr, out_sem, gt);
        if (Ci > 0) tl_layer64<PAN_ROWS>(Q, H, smem + l.Wi2T, smem + l.bi2, R, gt);
        group_sync<PAN_ROWS>(grp);
        if (tile + tstride < ntiles) fetch(tile + tstride);
        if (Ci > 0) tl_head<13, PAN_ROWS>(R, smem + l.Wi3T, smem + l.bi3, Ci, inst_softmax != 0, inv_temp, coef, rr, out_inst, gt);
    }
}

// Output head reduced to its label: the logits of tl_head (same registers, same arithmetic order), then per sample the winning
// class and its value of the channel the nef returns -- the [M,C] probabilities are never formed.  (z_max, argmax) and the softmax
// denominator are reduced over the 16 lanes of the sample group with shuffles; ties go to the lowest class index (torch.argmax).
// score = softmax ? 1 / sum_c exp((z_c - z_max) * scale) : z_max * scale.  Lane j < 8 of the group writes sample j of its 8.
template <int NC, int ROWS>
__device__ __forceinline__ void tl_head_label(const float* __restrict__ A, const float* __restrict__ WT, const float* __restrict__ b, int C,
                                              bool softmax, float scale, int64_t row0, int64_t M, int64_t* __restrict__ label,
                                              float* __restrict__ score, int tid) {
    constexpr int NP = NC / 2;
    const int cg = tid & 15, sg = tid >> 4;
    float2 acc[4][NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        const float bv = b[tl_class<NC>(i, cg)];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j][i] = make_float2(bv, bv);
    }
    {
        const float* a = A + sg * 8;
        const float* wt = WT + 2 * cg;
        const float* wl = WT + NP * 32 + cg;
#pragma unroll 2
        for (int k = 0; k < H; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(a + k * TL_LDA(ROWS));
            const float4 a1 = *reinterpret_cast<const float4*>(a + k * TL_LDA(ROWS) + 4);
            const float2 av[4] = {make_float2(a0.x, a0.y), make_float2(a0.z, a0.w), make_float2(a1.x, a1.y), make_float2(a1.z, a1.w)};
#pragma unroll
            for (int ip = 0; ip < NP; ++ip) {
                const float2 wv = *reinterpret_cast<const float2*>(wt + k * (16 * NC) + ip * 32);
#pragma unroll
                for (int j = 0; j < 4; ++j) { ffma2(acc[j][2 * ip], av[j], wv.x); ffma2(acc[j][2 * ip + 1], av[j], wv.y); }
            }
            if (NC & 1) {
                const float wv = wl[k * (16 * NC)];
#pragma unroll
                for (int j = 0; j < 4; ++j) ffma2(acc[j][NC - 1], av[j], wv);
            }
        }
    }
    // per lane: classes tl_class<NC>(i, cg) ascend with i, so a strict > keeps the lowest index among equal logits
    float mx[8];
    int am[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { mx[j] = -INFINITY; am[j] = 0x7fffffff; }
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        const int c = tl_class<NC>(i, cg);
        if (c < C) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (acc[j][i].x > mx[2 * j] || am[2 * j] == 0x7fffffff) { mx[2 * j] = acc[j][i].x; am[2 * j] = c; }
                if (acc[j][i].y > mx[2 * j + 1] || am[2 * j + 1] == 0x7fffffff) { mx[2 * j + 1] = acc[j][i].y; am[2 * j + 1] = c; }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
            const float v = __shfl_xor_sync(0xffffffffu, mx[j], o);
            const int c = __shfl_xor_sync(0xffffffffu, am[j], o);
            if (v > mx[j] || (v == mx[j] && c < am[j]) || am[j] == 0x7fffffff) { mx[j] = v; am[j] = c; }
        }
    }
    float sc[8];
    if (softmax) {
        const float sc2 = scale * 1.4426950408889634f;      // exp((z - mx) * scale) = 2^((z - mx) * scale * log2 e)
#pragma unroll
        for (int j = 0; j < 8; ++j) sc[j] = 0.f;
#pragma unroll
        for (int i = 0; i < NC; ++i)
            if (tl_class<NC>(i, cg) < C) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    sc[2 * j] += ex2_approx((acc[j][i].x - mx[2 * j]) * sc2);
                    sc[2 * j + 1] += ex2_approx((acc[j][i].y - mx[2 * j + 1]) * sc2);
                }
            }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) sc[j] += __shfl_xor_sync(0xffffffffu, sc[j], o);
            sc[j] = 1.f / sc[j];
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) sc[j] = mx[j] * scale;
    }
    // lane cg < 8 writes sample sg * 8 + cg (a select chain keeps the arrays in registers)
    int lab = am[0];
    float s = sc[0];
#pragma unroll
    for (int j = 1; j < 8; ++j)
        if (cg == j) { lab = am[j]; s = sc[j]; }
    const int64_t m = row0 + sg * 8 + cg;
    if (cg < 8 && m < M) { label[m] = lab; score[m] = s; }
}

// Labels of the semantic / instance heads (csrc map export): the staging, tiling and layers of pan_comp_fwd_tiled_kernel with the
// label epilogue instead of the compositing one.
__global__ void __launch_bounds__(PAN_MAXG * (2 * PAN_ROWS), 1)
pan_labels_fwd_tiled_kernel(const float* __restrict__ feats, const float* __restrict__ dfeats, const float* __restrict__ lodw,
                            int64_t M, int IN, PanParams p, int Cs, int Ci, int sem_softmax, int inst_softmax, float inv_temp,
                            int64_t* __restrict__ sem_label, float* __restrict__ sem_score, int64_t* __restrict__ inst_label,
                            float* __restrict__ inst_score) {
    extern __shared__ __align__(16) float smem[];
    const int NG = blockDim.x / (2 * PAN_ROWS), grp = threadIdx.x / (2 * PAN_ROWS), gt = threadIdx.x - grp * (2 * PAN_ROWS);
    const TlPanLayout l = tl_pan_layout(IN, NG);
    float* P = smem + l.groups + grp * l.gstride;
    float *Q = P + TL_BUF(PAN_ROWS), *R = Q + TL_BUF(PAN_ROWS);
    const int64_t ntiles = (M + PAN_ROWS - 1) / PAN_ROWS;
    const int64_t tile0 = (int64_t)blockIdx.x * NG + grp, tstride = (int64_t)gridDim.x * NG;
    auto fetch = [&](int64_t tile) {
        tl_fetch_rows<PAN_ROWS>(P, feats, IN, tile * PAN_ROWS, M, gt);
        if (dfeats) tl_fetch_rows<PAN_ROWS>(Q, dfeats, IN, tile * PAN_ROWS, M, gt);
        cp_async_commit();
    };
    if (tile0 < ntiles) fetch(tile0);
    if (Cs > 0) {
        tl_stage_wt(smem + l.Ws1T, p.Ws1, H, H, IN, IN); tl_stage_b(smem + l.bs1, p.bs1, H, H);
        tl_stage_wt(smem + l.Ws2T, p.Ws2, Cs, 16, H, H); tl_stage_b(smem + l.bs2, p.bs2, Cs, 16);
    }
    if (Ci > 0) {
        tl_stage_wt(smem + l.Wi1T, p.Wi1, H, H, IN, IN); tl_stage_b(smem + l.bi1, p.bi1, H, H);
        tl_stage_wt(smem + l.Wi2T, p.Wi2, H, H, H, H); tl_stage_b(smem + l.bi2, p.bi2, H, H);
        tl_stage_wt(smem + l.Wi3T, p.Wi3, Ci, TL_CIP, H, H); tl_stage_b(smem + l.bi3, p.bi3, Ci, TL_CIP);
    }
    __syncthreads();                       // weights staged (the only block-wide barrier)
    for (int64_t tile = tile0; tile < ntiles; tile += tstride) {
        const int64_t row0 = tile * PAN_ROWS;
        cp_async_wait_all();
        group_sync<PAN_ROWS>(grp);                   // raw rows landed; the previous tile's instance head is done with R
        tl_transpose_x<PAN_ROWS>(R, P, dfeats ? Q : nullptr, lodw, IN, row0, M, gt);
        group_sync<PAN_ROWS>(grp);
        if (Cs > 0) tl_layer64<PAN_ROWS>(R, IN, smem + l.Ws1T, smem + l.bs1, P, gt);
        if (Ci > 0) tl_layer64<PAN_ROWS>(R, IN, smem + l.Wi1T, smem + l.bi1, Q, gt);
        group_sync<PAN_ROWS>(grp);
        if (Cs > 0) tl_head_label<1, PAN_ROWS>(P, smem + l.Ws2T, smem + l.bs2, Cs, sem_softmax != 0, 1.f, row0, M, sem_label, sem_score, gt);
        if (Ci > 0) tl_layer64<PAN_ROWS>(Q, H, smem + l.Wi2T, smem + l.bi2, R, gt);
        group_sync<PAN_ROWS>(grp);
        if (tile + tstride < ntiles) fetch(tile + tstride);
        if (Ci > 0) tl_head_label<13, PAN_ROWS>(R, smem + l.Wi3T, smem + l.bi3, Ci, inst_softmax != 0, inv_temp, row0, M, inst_label, inst_score, gt);
    }
}

// ---------------------------------------------------------------------------------------------
// density + colour
// ---------------------------------------------------------------------------------------------
// view_embed (decoder_common.cuh) with one sincosf per component and the double-angle recurrence for the octaves 2, 4, 8 (|v| <= 1:
// the recurrence doubles the absolute error per octave, <= 1e-6 at the last one) instead of 24 sinf / cosf calls per sample
__device__ __forceinline__ void view_embed_doubling(float dx, float dy, float dz, float* pe /*27*/) {
    const float v[3] = {-dx, -dy, -dz};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        pe[c] = v[c];
        float sn, cs;
        sincosf(v[c], &sn, &cs);
#pragma unroll
        for (int f = 0; f < PE_F; ++f) {
            pe[3 + 3 * f + c] = sn;
            pe[3 + 3 * PE_F + 3 * f + c] = cs;
            const float s2 = 2.f * sn * cs, c2 = fmaf(-2.f * sn, sn, 1.f);
            sn = s2; cs = c2;
        }
    }
}

struct TlDcLayout { int Wd1T, bd1, Wd2T, bd2, Wc1T, bc1, Wc2T, bc2, Wc3, bc3, groups, oX, oA, oB, gstride, total; };
// per group: RAW [DC_ROWS][IN] (next tile's rows, cp.async) | X [max(IN, CINP)][LDA] (features k-major, then the colour decoder's input) | A | B
__host__ __device__ inline TlDcLayout tl_dc_layout(int IN, int NG) {
    TlDcLayout l; int o = 0;
    l.Wd1T = o; o += IN * H; l.bd1 = o; o += H; l.Wd2T = o; o += H * DOUT; l.bd2 = o; o += DOUT;
    l.Wc1T = o; o += CINP * H; l.bc1 = o; o += H; l.Wc2T = o; o += H * H; l.bc2 = o; o += H;
    l.Wc3 = o; o += 4 * H; l.bc3 = o; o += 4;
    l.groups = o;
    l.oX = DC_ROWS * IN; l.oA = l.oX + (IN > CINP ? IN : CINP) * TL_LDA(DC_ROWS); l.oB = l.oA + TL_BUF(DC_ROWS); l.gstride = l.oB + TL_BUF(DC_ROWS);
    l.total = o + NG * l.gstride;
    return l;
}

__global__ void __launch_bounds__(DC_MAXG * (2 * DC_ROWS), 1)
dc_fwd_tiled_kernel(const float* __restrict__ feats, const float* __restrict__ lodw, const float* __restrict__ ray_d, int S,
                    int64_t M, int IN, DcParams p, int want_rgb, float* __restrict__ sigma, float* __restrict__ rgb) {
    extern __shared__ __align__(16) float smem[];
    const int NG = blockDim.x / (2 * DC_ROWS), grp = threadIdx.x / (2 * DC_ROWS), gt = threadIdx.x - grp * (2 * DC_ROWS);
    const TlDcLayout l = tl_dc_layout(IN, NG);
    float* RAW = smem + l.groups + grp * l.gstride;
    float *XT = RAW + l.oX, *A = RAW + l.oA, *B = RAW + l.oB;
    const int64_t ntiles = (M + DC_ROWS - 1) / DC_ROWS;
    const int64_t tile0 = (int64_t)blockIdx.x * NG + grp, tstride = (int64_t)gridDim.x * NG;
    if (tile0 < ntiles) { tl_fetch_rows<DC_ROWS>(RAW, feats, IN, tile0 * DC_ROWS, M, gt); cp_async_commit(); }
    tl_stage_wt(smem + l.Wd1T, p.Wd1, H, H, IN, IN); tl_stage_b(smem + l.bd1, p.bd1, H, H);
    tl_stage_wt(smem + l.Wd2T, p.Wd2, DOUT, DOUT, H, H); tl_stage_b(smem + l.bd2, p.bd2, DOUT, DOUT);
    if (want_rgb) {
        tl_stage_wt(smem + l.Wc1T, p.Wc1, H, H, CIN, CINP); tl_stage_b(smem + l.bc1, p.bc1, H, H);
        tl_stage_wt(smem + l.Wc2T, p.Wc2, H, H, H, H); tl_stage_b(smem + l.bc2, p.bc2, H, H);
        for (int i = threadIdx.x; i < 3 * H; i += blockDim.x) smem[l.Wc3 + i] = __ldg(p.Wc3 + i);
        tl_stage_b(smem + l.bc3, p.bc3, 3, 4);
    }
    __syncthreads();                       // weights staged (the only block-wide barrier)
    for (int64_t tile = tile0; tile < ntiles; tile += tstride) {
        const int64_t row0 = tile * DC_ROWS;
        cp_async_wait_all();
        group_sync<DC_ROWS>(grp);                   // raw rows landed; the previous tile's readers of X / A are done
        tl_transpose_x<DC_ROWS>(XT, RAW, nullptr, lodw, IN, row0, M, gt);
        group_sync<DC_ROWS>(grp);
        if (tile + tstride < ntiles) { tl_fetch_rows<DC_ROWS>(RAW, feats, IN, (tile + tstride) * DC_ROWS, M, gt); cp_async_commit(); }
        tl_layer64<DC_ROWS>(XT, IN, smem + l.Wd1T, smem + l.bd1, A, gt);
        group_sync<DC_ROWS>(grp);
        {   // density head 64 -> 16 (no activation) into rows 0..15 of the colour input: thread = 4 samples x 2 outputs
            const int og = gt & 7, sg = gt >> 3;
            float2 acc[2][2];
            const float b0 = smem[l.bd2 + 2 * og], b1 = smem[l.bd2 + 2 * og + 1];
#pragma unroll
            for (int j = 0; j < 2; ++j) { acc[j][0] = make_float2(b0, b0); acc[j][1] = make_float2(b1, b1); }
            const float* a = A + sg * 4;
            const float* wt = smem + l.Wd2T + 2 * og;
#pragma unroll 8
            for (int k = 0; k < H; ++k) {
                const float4 av = *reinterpret_cast<const float4*>(a + k * TL_LDA(DC_ROWS));
                const float2 wv = *reinterpret_cast<const float2*>(wt + k * DOUT);
                ffma2(acc[0][0], make_float2(av.x, av.y), wv.x); ffma2(acc[1][0], make_float2(av.z, av.w), wv.x);
                ffma2(acc[0][1], make_float2(av.x, av.y), wv.y); ffma2(acc[1][1], make_float2(av.z, av.w), wv.y);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
                *reinterpret_cast<float4*>(XT + (2 * og + i) * TL_LDA(DC_ROWS) + sg * 4) = make_float4(acc[0][i].x, acc[0][i].y, acc[1][i].x, acc[1][i].y);
            if (og == 0) {
                const float sg4[4] = {acc[0][0].x, acc[0][0].y, acc[1][0].x, acc[1][0].y};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int64_t m = row0 + sg * 4 + j;
                    if (m < M) sigma[m] = fmaxf(sg4[j], 0.f);
                }
            }
        }
        if (!want_rgb) continue;
        if (gt >= (2 * DC_ROWS) - DC_ROWS) {   // view-direction embedding into rows 16..42, row 43 zero (the group's upper warps)
            const int s = gt - ((2 * DC_ROWS) - DC_ROWS);
            const int64_t m = row0 + s;
            const int64_t r = (m < M ? m : M - 1) / S;
            float pe[PE_DIM];
            view_embed_doubling(__ldg(ray_d + 3 * r), __ldg(ray_d + 3 * r + 1), __ldg(ray_d + 3 * r + 2), pe);
#pragma unroll
            for (int k = 0; k < PE_DIM; ++k) XT[(DOUT + k) * TL_LDA(DC_ROWS) + s] = pe[k];
            XT[CIN * TL_LDA(DC_ROWS) + s] = 0.f;
        }
        group_sync<DC_ROWS>(grp);
        tl_layer64<DC_ROWS>(XT, CINP, smem + l.Wc1T, smem + l.bc1, B, gt);
        group_sync<DC_ROWS>(grp);
        tl_layer64<DC_ROWS>(B, H, smem + l.Wc2T, smem + l.bc2, A, gt);
        group_sync<DC_ROWS>(grp);
        if (gt < DC_ROWS) {
            const int64_t m = row0 + gt;
            const float* hcol = A + gt;
            const float* w3 = smem + l.Wc3;
            float a0 = smem[l.bc3], a1 = smem[l.bc3 + 1], a2 = smem[l.bc3 + 2];
#pragma unroll 8
            for (int k = 0; k < H; ++k) {
                const float h = hcol[k * TL_LDA(DC_ROWS)];
                a0 = fmaf(w3[k], h, a0); a1 = fmaf(w3[H + k], h, a1); a2 = fmaf(w3[2 * H + k], h, a2);
            }
            if (m < M) {
                rgb[3 * m] = 1.f / (1.f + expf(-a0));
                rgb[3 * m + 1] = 1.f / (1.f + expf(-a1));
                rgb[3 * m + 2] = 1.f / (1.f + expf(-a2));
            }
        }
    }
}

static int tl_num_sms() {
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

// Semantic + instance heads of (feats + dfeats) * lodw fused with their compositing, exact FP32, forward only.
// out_sem[N,Cs] / out_inst[N,Ci] must be zero-initialised by the caller; results are accumulated with red.add.
int pag_pan_composite_fwd_f32(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                              const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                              float inst_temperature, const float* w, const float* alpha, const int64_t* ridx,
                              float* out_sem, float* out_inst, void* stream) {
    if (hidden != H || IN < 4 || IN > 64 || (IN & 3) || Cs < 0 || Cs > 16 || Ci < 0 || Ci > TL_CIP) return PAG_ERR_UNSUPPORTED;
    if (M == 0 || (Cs == 0 && Ci == 0)) return PAG_OK;
    if (!feats || !w || !alpha || !ridx || (Cs && !out_sem) || (Ci && !out_inst)) return PAG_ERR_ARG;
    PanParams p{};
    p.Ws1 = weights[0]; p.bs1 = weights[1]; p.Ws2 = weights[2]; p.bs2 = weights[3]; p.Wi1 = weights[4]; p.bi1 = weights[5];
    p.Wi2 = weights[6]; p.bi2 = weights[7]; p.Wi3 = weights[8]; p.bi3 = weights[9];
    int NG = PAN_MAXG;                      // as many tile groups as the shared memory holds next to the weights
    while (NG > 1 && (size_t)tl_pan_layout(IN, NG).total * sizeof(float) > 227 * 1024) --NG;
    const size_t bytes = (size_t)tl_pan_layout(IN, NG).total * sizeof(float);
    if (bytes > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(pan_comp_fwd_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
    const int64_t tiles = ((M + PAN_ROWS - 1) / PAN_ROWS + NG - 1) / NG;
    const int grid = (int)(tiles < tl_num_sms() ? tiles : tl_num_sms());
    const float it = inst_temperature > 0.f ? 1.f / inst_temperature : 1.f;
    pan_comp_fwd_tiled_kernel<<<grid, NG * (2 * PAN_ROWS), bytes, (cudaStream_t)stream>>>(feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax,
                                                                            inst_softmax, it, w, alpha, ridx, out_sem, out_inst);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// Semantic + instance labels of (feats + dfeats) * lodw, exact FP32, forward only: argmax class (lowest on ties) and its value of
// the head's output channel per sample, no per-class output.
int pag_pan_labels_fwd_f32(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN, const float* const* weights,
                           int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax, float inst_temperature, int64_t* sem_label,
                           float* sem_score, int64_t* inst_label, float* inst_score, void* stream) {
    if (hidden != H || IN < 4 || IN > 64 || (IN & 3) || Cs < 0 || Cs > 16 || Ci < 0 || Ci > TL_CIP) return PAG_ERR_UNSUPPORTED;
    if (M == 0 || (Cs == 0 && Ci == 0)) return PAG_OK;
    if (!feats || (Cs && (!sem_label || !sem_score)) || (Ci && (!inst_label || !inst_score))) return PAG_ERR_ARG;
    PanParams p{};
    p.Ws1 = weights[0]; p.bs1 = weights[1]; p.Ws2 = weights[2]; p.bs2 = weights[3]; p.Wi1 = weights[4]; p.bi1 = weights[5];
    p.Wi2 = weights[6]; p.bi2 = weights[7]; p.Wi3 = weights[8]; p.bi3 = weights[9];
    int NG = PAN_MAXG;
    while (NG > 1 && (size_t)tl_pan_layout(IN, NG).total * sizeof(float) > 227 * 1024) --NG;
    const size_t bytes = (size_t)tl_pan_layout(IN, NG).total * sizeof(float);
    if (bytes > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(pan_labels_fwd_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
    const int64_t tiles = ((M + PAN_ROWS - 1) / PAN_ROWS + NG - 1) / NG;
    const int grid = (int)(tiles < tl_num_sms() ? tiles : tl_num_sms());
    const float it = inst_temperature > 0.f ? 1.f / inst_temperature : 1.f;
    pan_labels_fwd_tiled_kernel<<<grid, NG * (2 * PAN_ROWS), bytes, (cudaStream_t)stream>>>(feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax,
                                                                              inst_softmax, it, sem_label, sem_score, inst_label, inst_score);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// Density + colour decoders, exact FP32, forward only: same contract as pag_decode_dc_fwd.
int pag_decode_dc_fwd_tiled(const float* feats, const float* lodw, const float* ray_d, int samples_per_ray, int64_t M, int IN,
                            const float* const* weights, int hidden, int view_dim, int want_rgb, float* sigma, float* rgb,
                            void* stream) {
    if (hidden != H || view_dim != PE_DIM || IN < 4 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M == 0) return PAG_OK;
    if (!feats || !sigma || (want_rgb && (!rgb || !ray_d)) || samples_per_ray < 1) return PAG_ERR_ARG;
    DcParams p{};
    p.Wd1 = weights[0]; p.bd1 = weights[1]; p.Wd2 = weights[2]; p.bd2 = weights[3]; p.Wc1 = weights[4]; p.bc1 = weights[5];
    p.Wc2 = weights[6]; p.bc2 = weights[7]; p.Wc3 = weights[8]; p.bc3 = weights[9];
    int NG = DC_MAXG;
    while (NG > 1 && (size_t)tl_dc_layout(IN, NG).total * sizeof(float) > 227 * 1024) --NG;
    const size_t bytes = (size_t)tl_dc_layout(IN, NG).total * sizeof(float);
    if (bytes > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(dc_fwd_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
    const int64_t tiles = ((M + DC_ROWS - 1) / DC_ROWS + NG - 1) / NG;
    const int grid = (int)(tiles < tl_num_sms() ? tiles : tl_num_sms());
    dc_fwd_tiled_kernel<<<grid, NG * (2 * DC_ROWS), bytes, (cudaStream_t)stream>>>(feats, lodw, ray_d, samples_per_ray, M, IN, p, want_rgb, sigma, rgb);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

}  // extern "C"
