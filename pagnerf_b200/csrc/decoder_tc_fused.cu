// Panoptic heads FUSED with their compositing (tensor-core path, training mode).
//
// In the reference the semantic / instance decoders materialise softmax probabilities [M,6] / [M,200]
// (pc_nerf/panoptic_delta_nef.py:238-257) which the tracer multiplies by the detached weights and segment-sums
// per ray (tracers/panoptic_packed_rf_tracer.py:178-205).  At 380 k samples the [M,200] fp32 tensor alone is
// 304 MB written + read in forward and twice that in backward -- more traffic than everything else in the step.
// Here the probabilities never leave the SM:
//   forward : logits (tcgen05, TMEM) -> block-wise online softmax, ONE ex2 per logit, exponentials parked back in TMEM
//             (tcgen05.st) -> per-warp fp16 transpose -> lanes = classes walk the warp's 32 samples, accumulate
//             c_s * p[s][j] (c_s = alpha_ray * w_s) and flush one coalesced red.add per ray segment into out[N, C];
//             the log2-domain log-sum-exp of every sample is kept for the backward; two CTAs per SM;
//   backward: logits recomputed (tcgen05), p = 2^(z - lse) (one ex2 per logit), per-ray gradients g_out[N, C] read through a
//             per-tile fp16 shared-memory cache of the tile's first 16 rays, d logits = c_s * p * (g - <p, g>) / T, then the
//             dX / dW chain with joint first-layer MMAs (semantic | instance) and tensor-core bias gradients (ones tile).
// 512 threads = 4 column groups x 128 rows as in decoder_tc.cu; inputs as f32 rows or as the encoders' fp16 operand images
// (bulk copies), see decoder_tc.cu's header.
// Output convention: out[ray] = alpha_p * sum_s w_p[s] * f[s].  For PanopticPackedRFTracer alpha_p, w_p are the detached
// colour weights: only the decoders and the delta grid receive gradient, exactly as in the reference.  For the DD tracer they
// come from the panoptic density and carry gradient: the backward additionally emits <p_s, g_ray> per sample (gw_sem, gw_inst).
#include "decoder_tc_common.cuh"

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
struct PanCompFwdLayout {
    int INP, nXc, CsP, CiP;
    int oX, oT1, oT2, oStage, oCR, oWs1, oWs2, oWi1, oWi2, oWi3, oBias, total;
};
__host__ __device__ inline PanCompFwdLayout pan_comp_fwd_layout(int IN, int Cs, int Ci) {
    PanCompFwdLayout l;
    l.INP = (IN + 15) & ~15; l.nXc = l.INP / 8;
    l.CsP = 16; l.CiP = Ci > 0 ? ((Ci + 15) & ~15) : 16;
    int o = 0;
    l.oX = o; o += l.nXc * TCH;
    l.oT1 = o; o += 8 * TCH;
    l.oT2 = o; o += 8 * TCH;
    l.oStage = 0;   // 16 fp16 transpose buffers [32][34] (34 KB) alias X|T1|T2 (>= 36 KB), all dead once the last MMA has completed
    l.oCR = o; o += 4 * 32 * 8;           // per lane quadrant: c[32] floats + ray[32] ints
    o = (o + 15) & ~15;
    l.oWs1 = o; o += l.nXc * 64 * 16;
    l.oWs2 = o; o += 8 * l.CsP * 16;
    l.oWi1 = o; o += l.nXc * 64 * 16;
    l.oWi2 = o; o += 8 * 64 * 16;
    l.oWi3 = o; o += 8 * l.CiP * 16;
    l.oBias = o; o += (64 + l.CsP + 64 + 64 + l.CiP) * 4;
    l.total = o;
    return l;
}

#define PCF_THREADS 512
#define PCF_NCG 4
#define LOG2E_F 1.4426950408889634f

// instance output bias in the units the softmax works in: b * (log2e / T), -inf on the padded columns (p = 0 there);
// without softmax: b / T and 0
__device__ __forceinline__ void stage_bi3_scaled(float* dst, const float* __restrict__ b, int n, int np, float s2, int softmax) {
    for (int i = threadIdx.x; i < np; i += blockDim.x) dst[i] = (i < n) ? __ldg(b + i) * s2 : (softmax ? -INFINITY : 0.f);
}

#define STG_LD 34   // halfs per staged row: 17 words -> conflict-free transposed access
// weighted segment-sum of one transposed 32-column block (stage[row][col], fp16) over the warp's rows into out[N, C].
// bmask bit r = row r starts a new ray (bit 0 never set); rows are walked four at a time, the common group without an
// interior ray boundary costs one LDS.128 of coefficients + 4 x (LDS, cvt, FFMA).
__device__ __forceinline__ void comp_block(const __half* stage, const float* __restrict__ wc, const int* __restrict__ wr, uint32_t bmask,
                                           int nrows, float* __restrict__ out, int C, int c0, int lane) {
    if (c0 + lane < C && nrows > 0) {
        float acc = 0.f;
        float* o = out + c0 + lane;
        const __half* st = stage + lane;
        int r = 0;
        for (; r + 4 <= nrows; r += 4) {
            const float4 c4 = *reinterpret_cast<const float4*>(wc + r);
            const float s0 = __half2float(st[r * STG_LD]), s1 = __half2float(st[(r + 1) * STG_LD]),
                        s2 = __half2float(st[(r + 2) * STG_LD]), s3 = __half2float(st[(r + 3) * STG_LD]);
            const uint32_t b = (bmask >> r) & 0xFu;
            if (b) {
                if (b & 1u) { red_add_f32(o + (int64_t)wr[r - 1] * C, acc); acc = 0.f; }
                acc = fmaf(c4.x, s0, acc);
                if (b & 2u) { red_add_f32(o + (int64_t)wr[r] * C, acc); acc = 0.f; }
                acc = fmaf(c4.y, s1, acc);
                if (b & 4u) { red_add_f32(o + (int64_t)wr[r + 1] * C, acc); acc = 0.f; }
                acc = fmaf(c4.z, s2, acc);
                if (b & 8u) { red_add_f32(o + (int64_t)wr[r + 2] * C, acc); acc = 0.f; }
                acc = fmaf(c4.w, s3, acc);
            } else {
                acc = fmaf(c4.x, s0, acc); acc = fmaf(c4.y, s1, acc); acc = fmaf(c4.z, s2, acc); acc = fmaf(c4.w, s3, acc);
            }
        }
        for (; r < nrows; ++r) {
            if ((bmask >> r) & 1u) { red_add_f32(o + (int64_t)wr[r - 1] * C, acc); acc = 0.f; }
            acc = fmaf(wc[r], __half2float(st[r * STG_LD]), acc);
        }
        red_add_f32(o + (int64_t)wr[nrows - 1] * C, acc);
    }
}

// IMG: feats / dfeats are the encoders' fp16 operand images (one 12 KB bulk copy per tile each), see pag_permuto_fwd_img16_dyn
template <bool IMG>
__global__ void __launch_bounds__(PCF_THREADS) pan_comp_fwd_kernel(
    const float* __restrict__ feats, const float* __restrict__ dfeats, const float* __restrict__ lodw, int64_t M, int IN,
    PanParams p, int Cs, int Ci, int sem_softmax, int inst_softmax, float inst_inv_temp,
    const float* __restrict__ w, const float* __restrict__ alpha, const int64_t* __restrict__ ridx,
    float* __restrict__ out_sem, float* __restrict__ out_inst, float* __restrict__ inst_lse, const int64_t* __restrict__ m_dev) {
    if (m_dev) M = min(M, __ldg(m_dev));
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ uint64_t bar_s;
    __shared__ uint64_t xbar_s;
    __shared__ uint32_t tmem_s;
    __shared__ float part_s[PCF_NCG][128][2];   // (max, sum) partials of the row softmax per column group
    const PanCompFwdLayout l = pan_comp_fwd_layout(IN, Cs, Ci);
    const int tid = threadIdx.x, warp = warp_id_uniform(), lane = tid & 31;
    const int q = warp & 3, cg = warp >> 2;
    const int row = 32 * q + lane;
    const float s2 = inst_softmax ? inst_inv_temp * LOG2E_F : inst_inv_temp;   // logits -> log2-domain scaled logits
    {   // weights (same images as decoder_tc.cu)
        float* b = reinterpret_cast<float*>(sm + l.oBias);
        if (Cs > 0) {
            stage_w16(reinterpret_cast<__half*>(sm + l.oWs1), p.Ws1, 64, IN, 64, l.INP, lodw);
            stage_w16(reinterpret_cast<__half*>(sm + l.oWs2), p.Ws2, Cs, 64, l.CsP, 64);
            stage_b32(b, p.bs1, 64, 64); stage_b32(b + 64, p.bs2, Cs, l.CsP);
        }
        if (Ci > 0) {
            stage_w16(reinterpret_cast<__half*>(sm + l.oWi1), p.Wi1, 64, IN, 64, l.INP, lodw);
            stage_w16(reinterpret_cast<__half*>(sm + l.oWi2), p.Wi2, 64, 64, 64, 64);
            stage_w16(reinterpret_cast<__half*>(sm + l.oWi3), p.Wi3, Ci, 64, l.CiP, 64);
            stage_b32(b + 64 + l.CsP, p.bi1, 64, 64); stage_b32(b + 128 + l.CsP, p.bi2, 64, 64);
            stage_bi3_scaled(b + 192 + l.CsP, p.bi3, Ci, l.CiP, s2, inst_softmax);
        }
    }
    if (tid == 0) { mbar_init(&bar_s, 1); mbar_init(&xbar_s, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_s, 256);
    sync_to_mma();
    tc_fence_after();
    const uint32_t tm = tmem_s, tl = tm + ((uint32_t)(q * 32) << 16);
    MmaBar mb{&bar_s, 0};
    const float* bias = reinterpret_cast<const float*>(sm + l.oBias);
    const float *bs1 = bias, *bs2 = bias + 64, *bi1 = bias + 64 + l.CsP, *bi2 = bi1 + 64, *bi3 = bi2 + 64;
    uint8_t *X = sm + l.oX, *T1 = sm + l.oT1, *T2 = sm + l.oT2;
    const uint32_t aX = smem_u32(X), aT1 = smem_u32(T1), aT2 = smem_u32(T2);
    const uint32_t ws1 = smem_u32(sm + l.oWs1), ws2 = smem_u32(sm + l.oWs2), wi1 = smem_u32(sm + l.oWi1),
                   wi2 = smem_u32(sm + l.oWi2), wi3 = smem_u32(sm + l.oWi3);
    const uint32_t semcol = (Ci > 0) ? (uint32_t)(l.CiP > 64 ? l.CiP : 64) : 128u;
    __half* stage = reinterpret_cast<__half*>(sm + l.oStage) + warp * (32 * STG_LD);  // one transpose buffer per warp
    float* wc = reinterpret_cast<float*>(sm + l.oCR) + q * 64;                      // shared by the 4 column groups of a quadrant
    int* wr = reinterpret_cast<int*>(wc + 32);
    const int c16 = 16 * cg;
    const int64_t ntiles = (M + 127) / 128;
    uint32_t xpar = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t m = tile * 128 + row;
        const bool valid = m < M;
        const int64_t mm = valid ? m : M - 1;
        if (IMG) {
            // feats tile -> X, delta tile -> T1 (idle until the first epilogue), then X += delta in place
            const uint32_t xbytes = (uint32_t)l.nXc * TCH;
            if (warp == 0 && elect_one()) {
                mbar_expect_tx(&xbar_s, dfeats ? 2 * xbytes : xbytes);
                bulk_g2s(X, reinterpret_cast<const uint8_t*>(feats) + (size_t)tile * xbytes, xbytes, &xbar_s);
                if (dfeats) bulk_g2s(T1, reinterpret_cast<const uint8_t*>(dfeats) + (size_t)tile * xbytes, xbytes, &xbar_s);
            }
            mbar_wait(&xbar_s, xpar);
            xpar ^= 1u;
            if (dfeats) tile_add16(X, nullptr, T1, (int)xbytes);
        } else {
            stage_x_coalesced(X, feats, dfeats, IN, l.INP, tile * 128, M);   // LOD weights are folded into the first-layer weights
            if (tile + gridDim.x < ntiles)
                prefetch_x_l2(feats, dfeats, IN, l.nXc, min((tile + gridDim.x) * 128 + row, M - 1), cg, PCF_NCG);
        }
        if (cg == 0) {   // compositing coefficients of this quadrant's rows
            const int64_t ray = ridx[mm];
            wr[lane] = (int)ray;
            wc[lane] = valid ? __ldg(alpha + ray) * __ldg(w + mm) : 0.f;
        }
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (Cs > 0) mma16_fwd(tm, aX, ws1, 64, 64, l.INP, false);
            if (Ci > 0) mma16_fwd(tm + 64, aX, wi1, 64, 64, l.INP, false);
            mb.commit();
        }
        mb.wait();
        if (Cs > 0) epi_relu16(tl + c16, bs1 + c16, T1 + 2 * cg * TCH, row);
        if (Ci > 0) epi_relu16(tl + 64 + c16, bi1 + c16, T2 + 2 * cg * TCH, row);
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (Cs > 0) mma16_fwd(tm + semcol, aT1, ws2, l.CsP, l.CsP, 64, false);
            if (Ci > 0) mma16_fwd(tm, aT2, wi2, 64, 64, 64, false);
            mb.commit();
        }
        mb.wait();
        const int64_t rows_left = M - (tile * 128 + q * 32);
        const int nrows = rows_left >= 32 ? 32 : (rows_left > 0 ? (int)rows_left : 0);
        uint32_t bmask;
        {   // ray boundaries inside this quadrant's 32 rows
            const int rv = wr[lane], pv = __shfl_up_sync(0xffffffffu, rv, 1);
            bmask = __ballot_sync(0xffffffffu, lane > 0 && rv != pv);
        }
        if (Ci > 0) {
            epi_relu16(tl + c16, bi2 + c16, T1 + 2 * cg * TCH, row);
            sync_to_mma();
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm, aT1, wi3, l.CiP, l.CiP, 64, false); mb.commit(); }
            mb.wait();
            // 32-column block b2 belongs to column group b2 % 4 (two blocks per group at most: CiP <= 208).
            // Pass 1 (softmax only): block-wise online max / sum with ONE exp2 per logit; the exponentials, taken
            // relative to the running maximum bref[.] of their 16-column block, go back into TMEM over the logits.
            float bref[4] = {0.f, 0.f, 0.f, 0.f};
            float inv = 1.f, gm = 0.f;
            if (inst_softmax) {
                float mx = -INFINITY, sum = 0.f;
#pragma unroll
                for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int c0 = 32 * cg + 128 * kk + 16 * h;
                        if (c0 < l.CiP) {
                            float v[16];
                            tmem_ld16(tl + c0, v);
                            float bm = -INFINITY;
#pragma unroll
                            for (int i = 0; i < 16; i += 4) {
                                const float4 b4 = *reinterpret_cast<const float4*>(bi3 + c0 + i);   // pre-scaled, -inf on padding
                                v[i] = fmaf(v[i], s2, b4.x); v[i + 1] = fmaf(v[i + 1], s2, b4.y);
                                v[i + 2] = fmaf(v[i + 2], s2, b4.z); v[i + 3] = fmaf(v[i + 3], s2, b4.w);
                                bm = fmaxf(fmaxf(bm, fmaxf(v[i], v[i + 1])), fmaxf(v[i + 2], v[i + 3]));
                            }
                            const float nm = fmaxf(mx, bm);
                            sum *= fast_exp2(mx - nm);
#pragma unroll
                            for (int i = 0; i < 16; ++i) { v[i] = fast_exp2(v[i] - nm); sum += v[i]; }
                            mx = nm; bref[2 * kk + h] = nm;
                            tmem_st16(tl + c0, v);
                        }
                    }
                }
                part_s[cg][row][0] = mx; part_s[cg][row][1] = sum;
                __syncthreads();
                gm = -INFINITY;
#pragma unroll
                for (int k = 0; k < PCF_NCG; ++k) gm = fmaxf(gm, part_s[k][row][0]);
                float gs = 0.f;
#pragma unroll
                for (int k = 0; k < PCF_NCG; ++k) gs = fmaf(part_s[k][row][1], fast_exp2(part_s[k][row][0] - gm), gs);
                inv = 1.f / gs;
                if (cg == 0 && valid && inst_lse) inst_lse[m] = gm + fast_log2(gs);   // log2-domain logsumexp for the backward
            }
            // Pass 2: probabilities -> fp16 transpose buffer -> weighted segment sums
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const int c0 = 32 * cg + 128 * kk;
                if (c0 < l.CiP) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        if (c0 + 16 * h < l.CiP) {
                            float v[16];
                            tmem_ld16(tl + c0 + 16 * h, v);
                            if (inst_softmax) {
                                const float f = fast_exp2(bref[2 * kk + h] - gm) * inv;
#pragma unroll
                                for (int i = 0; i < 16; ++i) v[i] *= f;
                            } else {
#pragma unroll
                                for (int i = 0; i < 16; ++i) v[i] = fmaf(v[i], s2, bi3[c0 + 16 * h + i]);
                            }
#pragma unroll
                            for (int i = 0; i < 16; i += 2)
                                *reinterpret_cast<__half2*>(stage + lane * STG_LD + 16 * h + i) = __floats2half2_rn(v[i], v[i + 1]);
                        }
                    }
                    __syncwarp();
                    comp_block(stage, wc, wr, bmask, nrows, out_inst, Ci, c0, lane);
                    __syncwarp();
                }
            }
        }
        if (Cs > 0 && cg == 0) {   // semantic head: 16 columns, one column group
            float z[16];
            tmem_ld16(tl + semcol, z);
            float mx = -INFINITY, sum = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) { z[j] += bs2[j]; if (j < Cs) mx = fmaxf(mx, z[j]); }
#pragma unroll
            for (int j = 0; j < 16; ++j) { z[j] = (j < Cs) ? (sem_softmax ? __expf(z[j] - mx) : z[j]) : 0.f; sum += z[j]; }
            const float inv = sem_softmax ? 1.f / sum : 1.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) stage[lane * STG_LD + j] = __float2half_rn(z[j] * inv);
            __syncwarp();
            comp_block(stage, wc, wr, bmask, nrows, out_sem, Cs, 0, lane);
            __syncwarp();
        }
        tc_fence_before();
        __syncthreads();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 256);
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
// TMEM columns (512).  The instance logits / probabilities [0,208) alias the scratch accumulators S0 / S1 / SEMLOG.
// Bias gradients of the wide layers come out of the tensor core: a constant "ones" tile is the B operand of an extra
// 16 columns of the layer-2 / layer-3 weight-gradient chains (B = H1 | ones, ones | H2), so the per-tile warp
// reduce-scatter is only left on the two first-layer gradients.
#define PCB_S0 0
#define PCB_S1 64
#define PCB_SEMLOG 128   // 16 columns, consumed before the instance logits are produced
#define PCB_DW1J 208     // [128 = (sem L1 | inst L1) x <=48]: both first-layer weight gradients from ONE chain
#define PCB_DWS2T 256    // [64(h) x 16(classes)] transposed
#define PCB_DWI2 272     // [64 x (64 + 16)]: column 64 = bias gradient (ones trick)
#define PCB_DWI3 352     // [Ci(<=208) x (16 + 64)] as two 128-row blocks: column 0 = bias gradient (ones trick), 16.. = weights

#define PCB_THREADS 512
#define PCB_NCG 4    // column groups per row
#define PCB_MAXK 3   // input quads (float4) per thread: IN <= 48
#define PCB_NGC 16   // rays whose output gradients are cached (fp16, pre-scaled) per tile
// The semantic head (one 16-column block per row, ~250 dependent instructions = ~1.5 k cycles for a warp running alone on its
// scheduler) belongs to the column group that owns the FEWEST instance-logit blocks (13 blocks: group 0 has 4, groups 1-3 have 3)
#define PCB_SEM_CG 3

struct PanCompBwdLayout {
    int INP, nXc, CsP, CiP, nGi;
    int oGs, oX, oHs, oH1, oOnes, oH2, oGi, oW1, oWs2, oWi2, oWi3, oBias, oGC, oGSC, oPF, total;
};
__host__ __device__ inline PanCompBwdLayout pan_comp_bwd_layout(int IN, int Cs, int Ci, bool img = false) {
    PanCompBwdLayout l;
    l.INP = (IN + 15) & ~15; l.nXc = l.INP / 8;
    l.CsP = 16; l.CiP = Ci > 0 ? ((Ci + 15) & ~15) : 16; l.nGi = l.CiP / 8;
    int o = 0;
    l.oGs = o; o += 2 * TCH;
    l.oX = o; o += l.nXc * TCH;
    l.oHs = o; o += 8 * TCH;        // Hs | H1 adjacent: one MN-major A operand covers both first-layer gradients
    l.oH1 = o; o += 8 * TCH;
    l.oOnes = o; o += 2 * TCH;      // H1 | ones: B operand of the layer-2 weight gradient (N = 80)
    l.oH2 = o; o += 8 * TCH;
    l.oGi = o; o += l.nGi * TCH;
    l.oW1 = o; o += l.nXc * 128 * 16;   // joint [Ws1; Wi1] image, 128 output rows
    l.oWs2 = o; o += 8 * l.CsP * 16;
    l.oWi2 = o; o += 8 * 64 * 16;
    l.oWi3 = o; o += 8 * l.CiP * 16;
    l.oBias = o; o += (64 + l.CsP + 64 + 64 + l.CiP) * 4;
    const int need = l.oGi + (l.nGi > 16 ? 32 : 16) * TCH;   // MN-major A operands read 16 chunks from their base
    if (o < need) o = need;
    o = (o + 15) & ~15;
    l.oGC = o; o += PCB_NGC * l.CiP * 2;                       // fp16 cache of g_inst rows (6.5 KB)
    o = (o + 15) & ~15;
    l.oGSC = o; o += img ? PCB_NGC * 16 * 4 : 0;                // f32 cache of g_sem rows (1 KB; image mode only: the f32-row
                                                                // variant has no shared memory left)
    o = (o + 127) & ~127;
    // next tile's inputs: cp.async slots (48 KB, f32 rows) or the two bulk-copy landing tiles (fp16 images, 24 KB)
    l.oPF = o; o += img ? 2 * l.nXc * TCH : 2 * PCB_MAXK * PCB_THREADS * 16;
    l.total = o;
    return l;
}

// per-CTA partial weight gradients (floats): [Ws1 64xIN | Ws2 Csx64 | Wi1 64xIN | Wi2 64x64 | Wi3 Cix64], 16-byte aligned segments
struct PanWsLayout { int oWs1, oWs2, oWi1, oWi2, oWi3, total; };
__host__ __device__ inline PanWsLayout pan_ws_layout(int IN, int Cs, int Ci) {
    PanWsLayout w;
    int o = 0;
    w.oWs1 = o; o += 64 * IN;
    w.oWs2 = o; o += (Cs * 64 + 3) & ~3;
    w.oWi1 = o; o += 64 * IN;
    w.oWi2 = o; o += 64 * 64;
    w.oWi3 = o; o += (Ci * 64 + 3) & ~3;
    w.total = o;
    return w;
}
// rows [row0, row0 + rows) of a joint weight image with OUTP output rows; W == nullptr stages zeros
__device__ __forceinline__ void stage_w16_part(__half* img, const float* __restrict__ W, int OUT, int IN, int rows, int row0, int OUTP, int INP,
                                               const float* __restrict__ colscale) {
    const int n = (INP / 8) * rows * 8;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int e = i & 7, r = (i >> 3) % rows, c = (i >> 3) / rows, in = c * 8 + e;
        float v = 0.f;
        if (W && r < OUT && in < IN) { v = __ldg(W + (size_t)r * IN + in); if (colscale) v *= __ldg(colscale + in); }
        img[((size_t)c * OUTP + row0 + r) * 8 + e] = __float2half_rn(v);
    }
}

// 16 consecutive (pre-scaled) per-ray output gradients: from the tile's fp16 cache when the ray is one of the first
// PCB_NGC of the tile, else straight from global memory
__device__ __forceinline__ void load_g16(const __half* __restrict__ gc_row, const float* __restrict__ grow, int c0, int C, bool vec4,
                                         float scale, float (&g)[16]) {
    if (gc_row) {
        const uint4 a = *reinterpret_cast<const uint4*>(gc_row + c0), b = *reinterpret_cast<const uint4*>(gc_row + c0 + 8);
        const uint32_t u[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u[i]));
            g[2 * i] = f.x; g[2 * i + 1] = f.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
            float4 t;
            if (vec4) t = (c0 + i < C) ? __ldg(reinterpret_cast<const float4*>(grow + c0 + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
            else t = make_float4(c0 + i < C ? __ldg(grow + c0 + i) : 0.f, c0 + i + 1 < C ? __ldg(grow + c0 + i + 1) : 0.f,
                                 c0 + i + 2 < C ? __ldg(grow + c0 + i + 2) : 0.f, c0 + i + 3 < C ? __ldg(grow + c0 + i + 3) : 0.f);
            // same fp16 rounding as the cached rows: the result must not depend on which rays of a tile were cached
            g[i] = __half2float(__float2half_rn(t.x * scale)); g[i + 1] = __half2float(__float2half_rn(t.y * scale));
            g[i + 2] = __half2float(__float2half_rn(t.z * scale)); g[i + 3] = __half2float(__float2half_rn(t.w * scale));
        }
    }
}

template <bool IMG>
__global__ void __launch_bounds__(PCB_THREADS) pan_comp_bwd_kernel(
    const float* __restrict__ feats, const float* __restrict__ dfeats, const float* __restrict__ lodw, int64_t M, int IN,
    PanParams p, int Cs, int Ci, int sem_softmax, int inst_softmax, float inst_inv_temp,
    const float* __restrict__ w, const float* __restrict__ alpha, const int64_t* __restrict__ ridx,
    const float* __restrict__ g_sem, const float* __restrict__ g_inst, int64_t R, const float* __restrict__ inst_lse,
    const float* __restrict__ scale_ptr, float* __restrict__ g_panop, const int64_t* __restrict__ m_dev, float* __restrict__ ws,
    float* __restrict__ gw_sem, float* __restrict__ gw_inst) {
    if (m_dev) M = min(M, __ldg(m_dev));
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ uint64_t bar_s;
    __shared__ uint64_t xbar_s;
    __shared__ uint32_t tmem_s;
    __shared__ float part_s[PCB_NCG][128];      // per column group: partial <p, g> of the row
    const PanCompBwdLayout l = pan_comp_bwd_layout(IN, Cs, Ci, IMG);
    const int tid = threadIdx.x, warp = warp_id_uniform(), lane = tid & 31;
    const int q = warp & 3, cg = warp >> 2;       // TMEM lane quadrant, column group
    const int row = 32 * q + lane;
    const bool do_sem = (Cs > 0) && g_sem, do_inst = (Ci > 0) && g_inst;
    const float s2 = inst_softmax ? inst_inv_temp * LOG2E_F : inst_inv_temp;
    uint8_t *Gs = sm + l.oGs, *X = sm + l.oX, *Hs = sm + l.oHs, *H1 = sm + l.oH1, *H2 = sm + l.oH2, *Gi = sm + l.oGi;
    {
        float* b = reinterpret_cast<float*>(sm + l.oBias);
        __half* w1 = reinterpret_cast<__half*>(sm + l.oW1);
        stage_w16_part(w1, do_sem ? p.Ws1 : nullptr, 64, IN, 64, 0, 128, l.INP, lodw);
        stage_w16_part(w1, do_inst ? p.Wi1 : nullptr, 64, IN, 64, 64, 128, l.INP, lodw);
        if (do_sem) {
            stage_w16(reinterpret_cast<__half*>(sm + l.oWs2), p.Ws2, Cs, 64, l.CsP, 64);
            stage_b32(b, p.bs1, 64, 64); stage_b32(b + 64, p.bs2, Cs, l.CsP);
        }
        if (do_inst) {
            stage_w16(reinterpret_cast<__half*>(sm + l.oWi2), p.Wi2, 64, 64, 64, 64);
            stage_w16(reinterpret_cast<__half*>(sm + l.oWi3), p.Wi3, Ci, 64, l.CiP, 64);
            stage_b32(b + 64 + l.CsP, p.bi1, 64, 64); stage_b32(b + 128 + l.CsP, p.bi2, 64, 64);
            stage_bi3_scaled(b + 192 + l.CsP, p.bi3, Ci, l.CiP, s2, inst_softmax);
        }
        // constant tiles: ones column (feature 0 of a 16-feature tile); the gradient tile of a disabled head stays zero
        for (int i = tid; i < 2 * TCH / 16; i += PCB_THREADS) {
            uint4 u = make_uint4(0u, 0u, 0u, 0u);
            if (i < TCH / 16) u.x = 0x00003C00u;   // half(1.0) in element 0 of chunk 0
            reinterpret_cast<uint4*>(sm + l.oOnes)[i] = u;
        }
        for (int i = tid; i < PCB_NGC * l.CiP / 8; i += PCB_THREADS)      // the padded classes of the gradient cache stay zero
            reinterpret_cast<uint4*>(sm + l.oGC)[i] = make_uint4(0u, 0u, 0u, 0u);
        if (!do_sem) for (int i = tid; i < 8 * TCH / 16; i += PCB_THREADS) reinterpret_cast<uint4*>(Hs)[i] = make_uint4(0u, 0u, 0u, 0u);
        if (!do_inst) for (int i = tid; i < 8 * TCH / 16; i += PCB_THREADS) reinterpret_cast<uint4*>(H1)[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (tid == 0) { mbar_init(&bar_s, 1); mbar_init(&xbar_s, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_s, 512);
    sync_to_mma();
    tc_fence_after();
    const uint32_t tm = tmem_s, tl = tm + ((uint32_t)(q * 32) << 16);
    MmaBar mb{&bar_s, 0};
    const float* bias = reinterpret_cast<const float*>(sm + l.oBias);
    const float *bs1 = bias, *bs2 = bias + 64, *bi1 = bias + 64 + l.CsP, *bi2 = bi1 + 64, *bi3 = bi2 + 64;
    const uint32_t aGs = smem_u32(Gs), aX = smem_u32(X), aHs = smem_u32(Hs), aH1 = smem_u32(H1), aH2 = smem_u32(H2), aGi = smem_u32(Gi),
                   aOnes = smem_u32(sm + l.oOnes);
    const uint32_t w1j = smem_u32(sm + l.oW1), ws2 = smem_u32(sm + l.oWs2), wi2 = smem_u32(sm + l.oWi2), wi3 = smem_u32(sm + l.oWi3);
    __half* gcache = reinterpret_cast<__half*>(sm + l.oGC);
    float* gsc = reinterpret_cast<float*>(sm + l.oGSC);
    const float scale = scale_ptr ? __ldg(scale_ptr) : 1.f;
    const float inv_scale = 1.f / scale;
    const int c16 = 16 * cg;                       // this thread's 16 hidden columns
    const bool vec4 = !(Ci & 3);
    float db_s1 = 0.f, db_i1 = 0.f, db_s2 = 0.f;
    const int64_t ntiles = (M + 127) / 128;
    float4* pf = reinterpret_cast<float4*>(sm + l.oPF);
    int64_t n_ray = 0, n_ray0 = 0;
    float n_w = 0.f, n_lse = 0.f;
    // image mode: the landing buffers of the bulk copies (feats tile, delta tile) live where the cp.async slots are
    const uint32_t xbytes = (uint32_t)l.nXc * TCH;
    uint8_t *XL = sm + l.oPF, *DL = sm + l.oPF + xbytes;
    const uint8_t *fimg = reinterpret_cast<const uint8_t*>(feats), *dimg = reinterpret_cast<const uint8_t*>(dfeats);
    uint32_t xpar = 0;
    if ((int64_t)blockIdx.x < ntiles) {
        const int64_t m0 = min((int64_t)blockIdx.x * 128 + row, M - 1);
        if (IMG) {
            if (warp == 0 && elect_one()) {
                mbar_expect_tx(&xbar_s, dimg ? 2 * xbytes : xbytes);
                bulk_g2s(XL, fimg + (size_t)blockIdx.x * xbytes, xbytes, &xbar_s);
                if (dimg) bulk_g2s(DL, dimg + (size_t)blockIdx.x * xbytes, xbytes, &xbar_s);
            }
        } else {
            xpfc_issue<PCB_MAXK>(pf, feats, dfeats, IN, (int64_t)blockIdx.x * 128, M);
        }
        n_ray = ridx[m0]; n_w = __ldg(w + m0); n_ray0 = ridx[(int64_t)blockIdx.x * 128];
        if (inst_lse) n_lse = __ldg(inst_lse + m0);
    }
    const int ci1 = Ci > 0 ? Ci : 1;
    const int gc_r0 = tid / ci1, gc_c0 = tid % ci1, gc_dr = PCB_THREADS / ci1, gc_dc = PCB_THREADS % ci1;
    bool first = true;
    // dX staging [128][IN + 4] f32 (<= 26 KB) aliases Hs | H1 (32 KB): both are dead once the stage-6 MMAs have completed and are
    // first rewritten after the next tile's stage-1 barrier, i.e. after every thread has finished the copy-out
    float* dxs = reinterpret_cast<float*>(Hs);
    int64_t dx_tile = -1;
    PAG_PHASE_INIT();
    if (!IMG) cp_async_wait_all();
    __syncthreads();
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, first = false) {
        const int64_t m = tile * 128 + row;
        const bool valid = m < M;
        const int64_t mm = valid ? m : M - 1;
        // per-row scalars were loaded one tile ahead; the dependent alpha[ray] load has the whole MLP forward to land
        const int64_t ray = n_ray, ray0 = n_ray0;
        const float w_row = n_w, lse_row = n_lse;
        const float a_row = __ldg(alpha + ray);
        if (IMG) {
            if (g_panop && dx_tile >= 0 && warp == 0 && elect_one()) bulk_wait_read_all();    // dX staging (Hs) stored: free again
            PAG_PHASE(0);
            mbar_wait(&xbar_s, xpar);
            xpar ^= 1u;
            tile_add16(X, XL, dimg ? DL : nullptr, (int)xbytes);       // X = feats + delta (fp16), LOD weights live in W1
        } else {
            if (g_panop && dx_tile >= 0) dx_copy_out(dxs, g_panop, IN, dx_tile * 128, M);      // previous tile's dX
            PAG_PHASE(0);
            // ---------------- stage 1 ----------------
            xpfc_consume<PCB_NCG, PCB_MAXK>(pf, dfeats != nullptr, IN, l.INP, X, row, cg);   // LOD weights live in W1
        }
        PAG_PHASE(1);
        {   // row scalars of the next tile into registers
            const int64_t tn = tile + gridDim.x;
            if (tn < ntiles) {
                const int64_t mn = min(tn * 128 + row, M - 1);
                n_ray = ridx[mn]; n_w = __ldg(w + mn); n_ray0 = ridx[tn * 128];
                if (inst_lse) n_lse = __ldg(inst_lse + mn);
            }
        }
        sync_to_mma(); PAG_PHASE(2);
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            mma16_fwd(tm + PCB_S0, aX, w1j, 128, 128, l.INP, false);     // sem | inst first layers in one chain
            mb.commit();
        }
        PAG_PHASE(17);
        if (tile + gridDim.x < ntiles) {     // every thread is past its slot / landing-buffer reads: the next tile streams in from here
            if (IMG) {
                if (warp == 0 && elect_one()) {
                    mbar_expect_tx(&xbar_s, dimg ? 2 * xbytes : xbytes);
                    bulk_g2s(XL, fimg + (size_t)(tile + gridDim.x) * xbytes, xbytes, &xbar_s);
                    if (dimg) bulk_g2s(DL, dimg + (size_t)(tile + gridDim.x) * xbytes, xbytes, &xbar_s);
                }
            } else {
                xpfc_issue<PCB_MAXK>(pf, feats, dfeats, IN, (tile + gridDim.x) * 128, M);
            }
        }
        PAG_PHASE(18);
        // while the MMAs run: the tile's per-ray output gradients (first PCB_NGC rays) -> registers, coalesced
        float gpre[7], gspre = 0.f;
        const int ngc_elems = PCB_NGC * Ci;
        if (IMG && do_sem && tid < PCB_NGC * Cs) {      // g_sem rows of the same rays: PCB_NGC * Cs <= 256 values
            const int64_t src = ray0 * Cs + tid;
            gspre = (src < R * Cs) ? __ldg(g_sem + src) : 0.f;
        }
        if (do_inst) {
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                const int e = tid + PCB_THREADS * k;
                const int64_t src = ray0 * Ci + e;
                gpre[k] = (e < ngc_elems && src < R * Ci) ? __ldg(g_inst + src) : 0.f;
            }
        }
        PAG_PHASE(19);
        mb.wait(); PAG_PHASE(3);
        const float cs = valid ? a_row * w_row : 0.f;     // the loss scale rides on the cached gradients
        uint32_t mask_s = 0, mask_1 = 0, mask_2 = 0;
        if (do_sem) {
            mask_s = epi_relu16(tl + PCB_S0 + c16, bs1 + c16, Hs + 2 * cg * TCH, row);
            if (IMG && tid < PCB_NGC * Cs) gsc[(tid / Cs) * 16 + (tid % Cs)] = gspre;
        }
        if (do_inst) {
            mask_1 = epi_relu16(tl + PCB_S1 + c16, bi1 + c16, H1 + 2 * cg * TCH, row);
            int gr = gc_r0, gc = gc_c0;      // (ray slot, class) of element tid + 512 k, advanced without divisions
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                if (gr < PCB_NGC) gcache[gr * l.CiP + gc] = __float2half_rn(gpre[k] * scale);
                gr += gc_dr; gc += gc_dc;
                if (gc >= Ci) { gc -= Ci; ++gr; }
            }
        }
        // ---------------- stage 2 ----------------
        sync_to_mma(); PAG_PHASE(4);
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (do_inst) mma16_fwd(tm + PCB_S0, aH1, wi2, 64, 64, 64, false);
            if (do_sem) mma16_fwd(tm + PCB_SEMLOG, aHs, ws2, l.CsP, l.CsP, 64, false);
            mb.commit();
        }
        mb.wait(); PAG_PHASE(5);
        if (do_inst) mask_2 = epi_relu16(tl + PCB_S0 + c16, bi2 + c16, H2 + 2 * cg * TCH, row);
        float zs[16];
        if (do_sem && cg == PCB_SEM_CG) tmem_ld16(tl + PCB_SEMLOG, zs);     // before the instance logits overwrite the column range
        // ---------------- stage 3: instance logits + head gradient; 16-column block b belongs to group b % 4 ----------------
        if (do_inst) {
            sync_to_mma(); PAG_PHASE(6);
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm, aH2, wi3, l.CiP, l.CiP, 64, false); mb.commit(); }
            PAG_PHASE(20);
        }
        if (do_sem && cg == PCB_SEM_CG) {   // semantic head gradient (<= 16 classes), while the logits MMA runs
            float g[16];
            float mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < 16; ++j) { zs[j] += bs2[j]; if (j < Cs) mx = fmaxf(mx, zs[j]); }
            const int64_t sslot = ray - ray0;
            if (IMG && sslot < PCB_NGC) {      // this ray's output gradient is in the tile's cache (filled while the first MMA ran)
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                    const float4 t = *reinterpret_cast<const float4*>(gsc + sslot * 16 + j);
                    g[j] = t.x; g[j + 1] = t.y; g[j + 2] = t.z; g[j + 3] = t.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) g[j] = (j < Cs) ? __ldg(g_sem + ray * Cs + j) : 0.f;
            }
            float Z = 0.f, E = 0.f, ZG = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float e = (j < Cs) ? (sem_softmax ? fast_exp2((zs[j] - mx) * LOG2E_F) : 1.f) : 0.f;
                if (j < Cs) ZG = fmaf(zs[j], g[j], ZG);
                zs[j] = e;
                Z += e; E = fmaf(e, (j < Cs) ? g[j] : 0.f, E);
            }
            const float iz = 1.f / Z, dot = E * iz, css = cs * scale;
            // <p_s, g_ray>: d out / d weight of this sample (DD tracer: weights carry gradient); p_s = the logits without softmax
            if (gw_sem && valid) gw_sem[m] = sem_softmax ? dot : ZG;
#pragma unroll
            for (int j = 0; j < 16; ++j) g[j] = (j < Cs) ? (sem_softmax ? css * zs[j] * iz * (g[j] - dot) : css * g[j]) : 0.f;
            grad16_store(g, Gs, row, lane, db_s2);
            PAG_PHASE(21);
        }
        if (do_inst) {
            mb.wait(); PAG_PHASE(7);
            // d logit_j = c * p_j * (g_j - <p, g>) / T with p_j = 2^(z_j - lse) from the forward's log-sum-exp: one
            // exp2 per logit; the probabilities go back into TMEM over the logits for the second pass.
            const float* grow = g_inst + ray * Ci;
            const int64_t slot = ray - ray0;
            const __half* gc_row = (slot < PCB_NGC) ? gcache + slot * l.CiP : nullptr;
            float dot = 0.f;
            if (inst_softmax) {
                const float nl = -lse_row;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c0 = 16 * (cg + PCB_NCG * k);
                    if (c0 < l.CiP) {
                        float v[16], g[16];
                        load_g16(gc_row, grow, c0, Ci, vec4, scale, g);
                        tmem_ld16(tl + c0, v);
#pragma unroll
                        for (int i = 0; i < 16; i += 4) {
                            const float4 b4 = *reinterpret_cast<const float4*>(bi3 + c0 + i);   // pre-scaled, -inf on padding
                            v[i] = fast_exp2(fmaf(v[i], s2, b4.x) + nl);         dot = fmaf(v[i], g[i], dot);
                            v[i + 1] = fast_exp2(fmaf(v[i + 1], s2, b4.y) + nl); dot = fmaf(v[i + 1], g[i + 1], dot);
                            v[i + 2] = fast_exp2(fmaf(v[i + 2], s2, b4.z) + nl); dot = fmaf(v[i + 2], g[i + 2], dot);
                            v[i + 3] = fast_exp2(fmaf(v[i + 3], s2, b4.w) + nl); dot = fmaf(v[i + 3], g[i + 3], dot);
                        }
                        tmem_st16_nowait(tl + c0, v);
                    }
                }
                tmem_wait_st();
                part_s[cg][row] = dot;
                __syncthreads(); PAG_PHASE(8);
                dot = (part_s[0][row] + part_s[1][row]) + (part_s[2][row] + part_s[3][row]);
                if (gw_inst && cg == 0 && valid) gw_inst[m] = dot * inv_scale;      // the cached gradients carry the loss scale
            } else if (gw_inst) {      // without softmax the sample's outputs are the scaled logits z / T: <z / T, g_ray>
                float zg = 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c0 = 16 * (cg + PCB_NCG * k);
                    if (c0 < l.CiP) {
                        float v[16], g[16];
                        load_g16(gc_row, grow, c0, Ci, vec4, scale, g);
                        tmem_ld16(tl + c0, v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) zg = fmaf(fmaf(v[i], s2, bi3[c0 + i]), g[i], zg);   // padded columns: g = 0
                    }
                }
                part_s[cg][row] = zg;
                __syncthreads();
                if (cg == 0 && valid) gw_inst[m] = ((part_s[0][row] + part_s[1][row]) + (part_s[2][row] + part_s[3][row])) * inv_scale;
            }
            const float c2 = cs * inst_inv_temp;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c0 = 16 * (cg + PCB_NCG * k);
                if (c0 < l.CiP) {
                    float v[16], g[16];
                    load_g16(gc_row, grow, c0, Ci, vec4, scale, g);
                    if (inst_softmax) {
                        tmem_ld16(tl + c0, v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = c2 * v[i] * (g[i] - dot);
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = c2 * g[i];
                    }
                    tile_store8(Gi + (c0 / 8) * TCH, 0, row, v);
                    tile_store8(Gi + (c0 / 8) * TCH, 1, row, v + 8);
                }
            }
        }
        // ---------------- stage 4 ----------------
        sync_to_mma(); PAG_PHASE(9);
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (do_inst) {
                mma16_bwd_weight(tm + PCB_DWI3, aGi, aOnes, 80, !first);      // B = ones | H2: column 0 = bias gradient
                if (l.CiP > 128) mma16_bwd_weight(tm + PCB_DWI3 + 80, aGi + 16 * TCH, aOnes, 80, !first);
                mma16_bwd_data(tm + PCB_S1, aGi, wi3, 64, l.CiP, l.CiP, false);
            }
            if (do_sem) {
                mma16_bwd_weight(tm + PCB_DWS2T, aHs, aGs, 16, !first);
                mma16_bwd_data(tm + PCB_S0, aGs, ws2, 64, l.CsP, l.CsP, false);
            }
            mb.commit();
        }
        mb.wait(); PAG_PHASE(10);
        if (do_inst) epi_grad16_nb(tl + PCB_S1 + c16, mask_2, H2 + 2 * cg * TCH, row);           // G2 overwrites H2
        if (do_sem) epi_grad16(tl + PCB_S0 + c16, mask_s, Hs + 2 * cg * TCH, row, lane, db_s1);  // Gs1 overwrites Hs
        // ---------------- stage 5 ----------------
        if (do_inst) {
            sync_to_mma(); PAG_PHASE(11);
            if (warp == 0 && elect_one()) {
                tc_fence_after();
                mma16_bwd_weight(tm + PCB_DWI2, aH2, aH1, 80, !first);      // B = H1 | ones: column 64 = bias gradient
                mma16_bwd_data(tm + PCB_S1, aH2, wi2, 64, 64, 64, false);
                mb.commit();
            }
            mb.wait(); PAG_PHASE(12);
            epi_grad16(tl + PCB_S1 + c16, mask_1, H1 + 2 * cg * TCH, row, lane, db_i1);           // G1 overwrites H1
        }
        // ---------------- stage 6: both first layers at once ----------------
        sync_to_mma(); PAG_PHASE(13);
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            mma16_bwd_weight(tm + PCB_DW1J, aHs, aX, l.INP, !first);                              // A = Gs1 | G1
            if (g_panop) mma16_bwd_data(tm + PCB_S0, aHs, w1j, l.INP, 128, 128, false);           // K = 128
            mb.commit();
        }
        mb.wait(); PAG_PHASE(14);
        if (IMG) {
            // dX as an fp16 operand-image tile (still carrying the loss scale), staged over Hs, stored with one bulk copy
            if (g_panop && c16 < l.INP) {
                float v[16];
                tmem_ld16(tl + PCB_S0 + c16, v);
                tile_store8(Hs, 2 * cg, row, v);
                tile_store8(Hs, 2 * cg + 1, row, v + 8);
                fence_async_smem();
            }
            dx_tile = tile;
            tc_fence_before();
            __syncthreads(); PAG_PHASE(15);
            if (g_panop && warp == 0 && elect_one()) bulk_s2g(reinterpret_cast<uint8_t*>(g_panop) + (size_t)tile * xbytes, Hs, xbytes);
        } else {
            if (g_panop && c16 < l.INP) dx_stage16(tl + PCB_S0, dxs, row, IN, c16, inv_scale);   // written out at the top of the next tile
            dx_tile = tile;
            cp_async_wait_all();      // own copies landed; the barrier publishes everybody's
            tc_fence_before();
            __syncthreads(); PAG_PHASE(15);
        }
    }
    if (IMG) {
        if (g_panop && dx_tile >= 0 && warp == 0 && elect_one()) bulk_wait_read_all();
    } else if (g_panop && dx_tile >= 0) dx_copy_out(dxs, g_panop, IN, dx_tile * 128, M);
    if (!first) {
        tc_fence_after();
        const int f1 = scatter_base(lane, 32) >> 1;     // feature (of 16) owned by this lane pair after grad16_store
        const bool own = !(lane & 1);
        // weight gradients: into this CTA's slice of the partial workspace when one is given (plain stores; 148 CTAs
        // hammering the same 94 KB with red.add serialise in the L2 atomic units), else straight into the gradients
        const bool plain = ws != nullptr;
        const PanWsLayout wl = pan_ws_layout(IN, Cs, Ci);
        float* wsb = plain ? ws + (size_t)blockIdx.x * wl.total : nullptr;
        float *dWs1 = plain ? wsb + wl.oWs1 : p.gWs1, *dWs2 = plain ? wsb + wl.oWs2 : p.gWs2, *dWi1 = plain ? wsb + wl.oWi1 : p.gWi1,
              *dWi2 = plain ? wsb + wl.oWi2 : p.gWi2, *dWi3 = plain ? wsb + wl.oWi3 : p.gWi3;
        if (c16 < l.INP) {      // joint first-layer gradient: lanes 0..63 semantic, 64..127 instance
            float* gW1 = (row < 64) ? (do_sem ? dWs1 : nullptr) : (do_inst ? dWi1 : nullptr);
            float v[16];
            tmem_ld16(tl + PCB_DW1J + c16, v);      // G^T X with X unweighted: the LOD weight of each input column applies here
            if (gW1) {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (c16 + i < IN) {
                        const float x = v[i] * inv_scale * (lodw ? __ldg(lodw + c16 + i) : 1.f);
                        float* d = gW1 + (size_t)(row & 63) * IN + c16 + i;
                        if (plain) *d = x; else red_add_f32(d, x);
                    }
            }
        }
        if (do_sem) {
            if (cg == 0) {
                float v[16];
                tmem_ld16(tl + PCB_DWS2T, v);      // transposed accumulator [lanes = hidden k][cols = classes j] -> gW[j][k]
                if (row < 64) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (j < Cs) { if (plain) dWs2[(size_t)j * 64 + row] = v[j] * inv_scale; else red_add_f32(dWs2 + (size_t)j * 64 + row, v[j] * inv_scale); }
                }
            }
            if (own) red_add_f32(p.gbs1 + c16 + f1, db_s1 * inv_scale);
            if (own && cg == PCB_SEM_CG && f1 < Cs) red_add_f32(p.gbs2 + f1, db_s2 * inv_scale);
        }
        if (do_inst) {
            flush_dw16(tl + PCB_DWI2, dWi2, row, 64, 64, c16, inv_scale, plain);
            flush_dw16(tl + PCB_DWI3 + 16, dWi3, row, Ci, 64, c16, inv_scale, plain);
            if (l.CiP > 128) flush_dw16(tl + PCB_DWI3 + 96, dWi3 + (size_t)128 * 64, row, Ci - 128, 64, c16, inv_scale, plain);
            if (own) red_add_f32(p.gbi1 + c16 + f1, db_i1 * inv_scale);
            if (cg == 0) {      // ones-trick bias gradients: column 0 of the extra accumulators
                float v[16];
                tmem_ld16(tl + PCB_DWI2 + 64, v);
                if (row < 64) red_add_f32(p.gbi2 + row, v[0] * inv_scale);
                tmem_ld16(tl + PCB_DWI3, v);
                if (row < Ci) red_add_f32(p.gbi3 + row, v[0] * inv_scale);
                if (l.CiP > 128) {
                    tmem_ld16(tl + PCB_DWI3 + 80, v);
                    if (128 + row < Ci) red_add_f32(p.gbi3 + 128 + row, v[0] * inv_scale);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    PAG_PHASE(40);
    PAG_PHASE_FLUSH();
    if (warp == 0) tmem_dealloc(tm, 512);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
extern int pag_reserved_sms;      // decoder_tc.cu, pag_set_reserved_sms
static int fused_num_sms() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    const int m = n - pag_reserved_sms;
    return m > 8 ? m : 8;
}
static void fill_pan_f(PanParams& p, const float* const* w, float* const* g) {
    p.Ws1 = w[0]; p.bs1 = w[1]; p.Ws2 = w[2]; p.bs2 = w[3]; p.Wi1 = w[4]; p.bi1 = w[5]; p.Wi2 = w[6]; p.bi2 = w[7]; p.Wi3 = w[8]; p.bi3 = w[9];
    if (g) { p.gWs1 = g[0]; p.gbs1 = g[1]; p.gWs2 = g[2]; p.gbs2 = g[3]; p.gWi1 = g[4]; p.gbi1 = g[5]; p.gWi2 = g[6]; p.gbi2 = g[7]; p.gWi3 = g[8]; p.gbi3 = g[9]; }
}
static bool fused_shape_ok(int IN, int hidden, int Cs, int Ci) {
    return hidden == H && IN >= 4 && IN <= 48 && !(IN & 3) && Cs >= 0 && Cs <= 16 && Ci >= 0 && Ci <= 208;
}

PAG_PHASE_READER(pag_debug_phase_read)

extern "C" {

// out_sem[N,Cs] / out_inst[N,Ci] must be zero-initialised by the caller; results are accumulated with red.add.
int pag_pan_composite_fwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                             const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                             float inst_temperature, const float* w, const float* alpha, const int64_t* ridx,
                             float* out_sem, float* out_inst, float* inst_lse, const int64_t* m_dev, int x_img16, void* stream) {
    if (!fused_shape_ok(IN, hidden, Cs, Ci)) return PAG_ERR_UNSUPPORTED;
    if (x_img16 && (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M == 0 || (Cs == 0 && Ci == 0)) return PAG_OK;
    PanParams p{};
    fill_pan_f(p, weights, nullptr);
    const PanCompFwdLayout l = pan_comp_fwd_layout(IN, Cs, Ci);
    if (l.total > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    const float it = inst_temperature > 0.f ? 1.f / inst_temperature : 1.f;
    const int64_t tiles = (M + 127) / 128;
    const int64_t cap = 2 * (int64_t)fused_num_sms();   // 97 KB smem + 256 TMEM columns per CTA: two CTAs per SM
    const int grid = (int)(tiles < cap ? tiles : cap);
    if (x_img16) {
        cudaError_t e = cudaFuncSetAttribute(pan_comp_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, l.total);
        if (e != cudaSuccess) return (int)e;
        pan_comp_fwd_kernel<true><<<grid, PCF_THREADS, l.total, (cudaStream_t)stream>>>(
            feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax, inst_softmax, it, w, alpha, ridx, out_sem, out_inst, inst_lse, m_dev);
    } else {
        cudaError_t e = cudaFuncSetAttribute(pan_comp_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, l.total);
        if (e != cudaSuccess) return (int)e;
        pan_comp_fwd_kernel<false><<<grid, PCF_THREADS, l.total, (cudaStream_t)stream>>>(
            feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax, inst_softmax, it, w, alpha, ridx, out_sem, out_inst, inst_lse, m_dev);
    }
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// g_sem[N,Cs] / g_inst[N,Ci]: per-RAY gradients of the composited outputs (nullable); g_panop[M,IN] nullable.
int pag_pan_composite_bwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                             const float* const* weights, float* const* grads, int hidden, int Cs, int Ci,
                             int sem_softmax, int inst_softmax, float inst_temperature, const float* w, const float* alpha,
                             const int64_t* ridx, int64_t R, const float* g_sem, const float* g_inst, const float* inst_lse,
                             const float* grad_scale, float* g_panop, const int64_t* m_dev, float* workspace,
                             int64_t workspace_bytes, int x_img16, float* gw_sem, float* gw_inst, void* stream) {
    if (!fused_shape_ok(IN, hidden, Cs, Ci)) return PAG_ERR_UNSUPPORTED;
    if (Ci > 0 && g_inst && inst_softmax && !inst_lse) return PAG_ERR_ARG;
    if (M == 0 || (Cs == 0 && Ci == 0)) return PAG_OK;
    PanParams p{};
    fill_pan_f(p, weights, grads);
    if (x_img16 && (IN & 3)) return PAG_ERR_UNSUPPORTED;
    const PanCompBwdLayout l = pan_comp_bwd_layout(IN, Cs, Ci, x_img16 != 0);
    if (l.total > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    const float it = inst_temperature > 0.f ? 1.f / inst_temperature : 1.f;
    const int64_t tiles = (M + 127) / 128;
    const int64_t cap = fused_num_sms();
    const int nblocks = (int)(tiles < cap ? tiles : cap);
    const PanWsLayout wl = pan_ws_layout(IN, Cs, Ci);
    float* ws = (workspace && workspace_bytes >= (int64_t)nblocks * wl.total * 4 && !(reinterpret_cast<uintptr_t>(workspace) & 15)) ? workspace : nullptr;
    if (x_img16) {
        cudaError_t e2 = cudaFuncSetAttribute(pan_comp_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, l.total);
        if (e2 != cudaSuccess) return (int)e2;
        pan_comp_bwd_kernel<true><<<nblocks, PCB_THREADS, l.total, (cudaStream_t)stream>>>(
            feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax, inst_softmax, it, w, alpha, ridx, g_sem, g_inst, R, inst_lse, grad_scale, g_panop, m_dev, ws, gw_sem, gw_inst);
    } else {
        cudaError_t e2 = cudaFuncSetAttribute(pan_comp_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, l.total);
        if (e2 != cudaSuccess) return (int)e2;
        pan_comp_bwd_kernel<false><<<nblocks, PCB_THREADS, l.total, (cudaStream_t)stream>>>(
            feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax, inst_softmax, it, w, alpha, ridx, g_sem, g_inst, R, inst_lse, grad_scale, g_panop, m_dev, ws, gw_sem, gw_inst);
    }
    PAG_LAUNCH_CHECK();
    if (ws) {
        const bool ds = Cs > 0 && g_sem, di = Ci > 0 && g_inst;
        WsSegs sg{5, {wl.oWs1, wl.oWs2, wl.oWi1, wl.oWi2, wl.oWi3}, {64 * IN, Cs * 64, 64 * IN, 64 * 64, Ci * 64},
                  {ds ? p.gWs1 : nullptr, ds ? p.gWs2 : nullptr, di ? p.gWi1 : nullptr, di ? p.gWi2 : nullptr, di ? p.gWi3 : nullptr}};
        ws_reduce_kernel<<<dim3((wl.total + 255) / 256, WS_GROUPS), 256, 0, (cudaStream_t)stream>>>(ws, nblocks, M, m_dev, wl.total, sg);
        PAG_LAUNCH_CHECK();
    }
    return PAG_OK;
}

// bytes of partial-gradient workspace pag_pan_composite_bwd_tc can use for M samples (0 rows -> 0)
int pag_pan_composite_bwd_workspace(int64_t M, int IN, int Cs, int Ci, int64_t* bytes) {
    if (!bytes) return PAG_ERR_ARG;
    const int64_t tiles = (M + 127) / 128, cap = fused_num_sms();
    *bytes = (tiles < cap ? tiles : cap) * (int64_t)pan_ws_layout(IN, Cs, Ci).total * 4;
    return PAG_OK;
}

}  // extern "C"
