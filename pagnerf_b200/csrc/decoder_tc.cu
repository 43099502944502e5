// Tensor-core (tcgen05 + TMEM) decoders: the training-mode path of the panoptic field's MLPs.
//
// Same math as decoder.cu, but every dense layer is a tcgen05.mma (kind::f16: fp16 operands, fp32
// accumulation in TMEM) -- the numerics of the reference's own training step, which runs these
// layers as fp16 GEMMs under torch.cuda.amp.autocast with a GradScaler (pc_nerf/trainer.py:429,582).
// ncu on the FP32-FMA kernels showed them issue/occupancy bound (profiles/r01_*): 85 GFLOP per
// 410 k-sample step cost 8.6 ms on the FMA pipe, i.e. the contraction, not memory, bounds the step.
//
// Mapping (density/colour kernels; the modular semantic/instance kernels further down keep the simpler 128-thread form):
//   * persistent CTAs (one per SM in the backward, two in the forward), one 128-sample tile at a time, 512 threads =
//     4 column groups x 128 rows: warps w, w+4, w+8, w+12 share TMEM lane quadrant w % 4 and split a row's columns,
//     which quadruples the warps that hide epilogue latency without more TMEM or shared memory;
//   * activations / gradients live in shared memory as fp16 "tile images" [F/8][128 rows][8 halfs]
//     (UMMA SWIZZLE_NONE canonical layout; a thread writes its row with conflict-free 16-byte stores);
//   * weights are staged once per CTA as fp16 images [IN/8][OUT rows][8 halfs]; the LOD weights of the feature vector are
//     folded into the first-layer image;
//   * ONE image serves every operand role:  Y = X W^T (tile K-major x weight K-major),
//     dX = G W (tile K-major x the same weight image read MN-major), dW += G^T X (tile MN-major x
//     tile MN-major, K = the tile's 128 samples);
//   * tcgen05.mma is issued from warp-uniform control flow (warp_id_uniform() == 0 && elect_one()): under a divergent
//     `threadIdx.x == 0` the compiler wraps every MMA in a per-lane loop (tools/mma_bench.py: 105 -> 77 cycles per MMA);
//   * the input tile arrives either as f32 rows (coalesced cp.async into rotation-swizzled slots, converted by the
//     threads) or, in the fused trace, as the encoder's fp16 operand image by ONE bulk (TMA) copy per tile into a
//     ping-pong buffer; dX leaves the same way (padded f32 staging + coalesced copy-out, or an fp16 image tile + bulk store);
//   * weight gradients never leave TMEM until the CTA has swept all its tiles (accumulate flag); a constant "ones" tile next
//     to each B operand adds 16 accumulator columns whose first column is the bias gradient; the CTA's partial sums go to
//     a private workspace slice (plain stores) and ws_reduce_kernel adds the slices (red.add without a workspace).
// Upstream gradients are multiplied by a power-of-two `grad_scale` before the fp16 repack and every
// result is unscaled in fp32 (the GradScaler trick, applied inside the kernel); dX images keep the scale and the encoder
// backward removes it.
#include "decoder_tc_common.cuh"

// ---------------------------------------------------------------------------------------------
// density + color
// ---------------------------------------------------------------------------------------------
#define DC_THREADS 512
#define DC_NCG 4     // column groups per sample row: warps w, w+4, w+8, w+12 share TMEM lane quadrant w % 4
#define DC_MAXK 4    // input quads per thread in the coalesced prefetch: 128 * (IN <= 64) / 4 / 512

struct DcTcLayout {  // byte offsets inside dynamic smem
    int INP, nXc;
    int oG3, oGy, oOnesA, oX, oHd, oOnesB, oCin, oH1, oOnesC, oH2, oWd1, oWd2, oWc1, oWc2, oWc3, oBias, oPF, oDX, oXI, total;
};
// Backward tile order: G3 Gy | onesA X | Hd onesB Cin | H1 onesC H2.  Each constant "ones" tile (feature 0 = 1) sits next
// to the B operands of two weight-gradient chains, which therefore also produce the bias gradients:
//   dWd1 = Gd^T [onesA | X]   dWd2 = Gy^T [Hd | onesB]   dWc1 = G1^T [onesB | Cin]   dWc2 = G2^T [H1 | onesC]   dWc3 = G3^T [onesC | H2]
__host__ __device__ inline DcTcLayout dc_tc_layout(int IN, bool bwd, bool img = false) {
    DcTcLayout l;
    l.INP = (IN + 15) & ~15;
    l.nXc = l.INP / 8;
    int o = 0;
    l.oG3 = o; o += bwd ? 2 * TCH : 0;
    l.oGy = o; o += bwd ? 2 * TCH : 0;
    l.oOnesA = o; o += bwd ? 2 * TCH : 0;
    l.oX = o; o += 8 * TCH;            // X (<= 64 feats); forward reuses it for Hc2
    l.oHd = o; o += 8 * TCH;
    l.oOnesB = o; o += bwd ? 2 * TCH : 0;
    l.oCin = o; o += bwd ? 6 * TCH : 0;
    l.oH1 = o; o += bwd ? 8 * TCH : 0;
    l.oOnesC = o; o += bwd ? 2 * TCH : 0;
    l.oH2 = o; o += bwd ? 8 * TCH : 0;
    l.oWd1 = o; o += l.nXc * 64 * 16;
    l.oWd2 = o; o += 8 * 16 * 16;
    l.oWc1 = o; o += 6 * 64 * 16;
    l.oWc2 = o; o += 8 * 64 * 16;
    l.oWc3 = o; o += 8 * 16 * 16;
    l.oBias = o; o += (64 + 16 + 64 + 64 + 16) * 4;
    if (bwd && o < l.oH2 + 16 * TCH) o = l.oH2 + 16 * TCH;  // MN-major A operands read 16 chunks from their base
    o = (o + 15) & ~15;
    l.oPF = o; o += (bwd && !img) ? 128 * (IN >> 2) * 16 : 0;   // cp.async slots of the next tile's inputs (f32 rows)
    l.oDX = o; o += bwd ? (img ? l.nXc * TCH : 128 * (IN + 4) * 4) : 0;   // dX tile staging: fp16 image tile / padded f32 rows
    // image mode: the input tile arrives by bulk copy straight into operand layout; two buffers (tile t+1 lands while tile t is
    // processed), each preceded by its own ones tile in the backward (B operand of dWd1 = [ones | X])
    o = (o + 127) & ~127;
    l.oXI = o; o += img ? 2 * ((bwd ? 2 : 0) + l.nXc) * TCH : 0;
    l.total = o;
    return l;
}

// lodw (nullable): per-feature LOD weights, folded into the first density layer (see stage_w16)
__device__ __forceinline__ void dc_tc_stage(uint8_t* sm, const DcTcLayout& l, const DcParams& p, int IN, const float* __restrict__ lodw) {
    stage_w16(reinterpret_cast<__half*>(sm + l.oWd1), p.Wd1, 64, IN, 64, l.INP, lodw);
    stage_w16(reinterpret_cast<__half*>(sm + l.oWd2), p.Wd2, 16, 64, 16, 64);
    stage_w16(reinterpret_cast<__half*>(sm + l.oWc1), p.Wc1, 64, CIN, 64, 48);
    stage_w16(reinterpret_cast<__half*>(sm + l.oWc2), p.Wc2, 64, 64, 64, 64);
    stage_w16(reinterpret_cast<__half*>(sm + l.oWc3), p.Wc3, 3, 64, 16, 64);
    float* b = reinterpret_cast<float*>(sm + l.oBias);
    stage_b32(b, p.bd1, 64, 64); stage_b32(b + 64, p.bd2, 16, 16); stage_b32(b + 80, p.bc1, 64, 64);
    stage_b32(b + 144, p.bc2, 64, 64); stage_b32(b + 208, p.bc3, 3, 16);
}

// 16 features [16*cg, 16*cg+16) of the color-decoder input row [y16 | PE(-d) 27 | 0 pad 5], cg = 1, 2
__device__ __forceinline__ void stage_cin_pe(uint8_t* tile, int row, int cg, float dx, float dy, float dz) {
    float pe[PE_DIM];
    view_embed(dx, dy, dz, pe);
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        v[i] = 0.f;
#pragma unroll
        for (int g = 1; g <= 2; ++g) {
            const int k = 16 * (g - 1) + i;      // PE index
            if (g == cg && k < PE_DIM) v[i] = pe[k];
        }
    }
    tile_store8(tile, 2 * cg, row, v);
    tile_store8(tile, 2 * cg + 1, row, v + 8);
}
// the same from the per-ray fp16 embedding image pe16[ray][32 halfs] (pag_view_pe16): two 16-byte copies
__device__ __forceinline__ void stage_cin_pe16(uint8_t* tile, int row, int cg, uint4 a, uint4 b) {
    *reinterpret_cast<uint4*>(tile + (2 * cg) * TCH + row * 16) = a;
    *reinterpret_cast<uint4*>(tile + (2 * cg + 1) * TCH + row * 16) = b;
}

// per-ray view embedding, fp16, padded to 32: the decoders copy it instead of evaluating 24 sin/cos per SAMPLE
__global__ void view_pe16_kernel(const float* __restrict__ ray_d, int64_t R, __half* __restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    float pe[32];
    view_embed(ray_d[3 * r], ray_d[3 * r + 1], ray_d[3 * r + 2], pe);
#pragma unroll
    for (int i = PE_DIM; i < 32; ++i) pe[i] = 0.f;
    uint4* o = reinterpret_cast<uint4*>(out + r * 32);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        uint4 u;
        u.x = pack_h2(pe[8 * c], pe[8 * c + 1]); u.y = pack_h2(pe[8 * c + 2], pe[8 * c + 3]);
        u.z = pack_h2(pe[8 * c + 4], pe[8 * c + 5]); u.w = pack_h2(pe[8 * c + 6], pe[8 * c + 7]);
        o[c] = u;
    }
}

// IMG: feats is the encoder's fp16 operand image (pag_permuto_fwd_img16_dyn): the input tile of a step is one 12 KB bulk copy
// into a ping-pong buffer, issued a tile ahead by one elected thread, and consumed by the tensor core as it is.
template <bool IMG>
__global__ void __launch_bounds__(DC_THREADS) dc_tc_fwd_kernel(const float* __restrict__ feats, const float* __restrict__ lodw,
                                                               const float* __restrict__ ray_d, int S, int64_t M, int IN,
                                                               DcParams p, int want_rgb, float* __restrict__ sigma,
                                                               float* __restrict__ rgb, const int64_t* __restrict__ m_dev,
                                                               const int64_t* __restrict__ ridx, const uint4* __restrict__ pe16,
                                                               float* __restrict__ y0_raw) {
    if (m_dev) M = min(M, __ldg(m_dev));
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ uint64_t bar_s;
    __shared__ uint64_t xbar_s[2];
    __shared__ uint32_t tmem_s;
    const DcTcLayout l = dc_tc_layout(IN, false, IMG);
    const int tid = threadIdx.x, warp = warp_id_uniform(), lane = tid & 31;
    const int q = warp & 3, cg = warp >> 2, row = 32 * q + lane, c16 = 16 * cg;
    dc_tc_stage(sm, l, p, IN, lodw);
    if (tid == 0) { mbar_init(&bar_s, 1); mbar_init(&xbar_s[0], 1); mbar_init(&xbar_s[1], 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_s, 128);
    sync_to_mma();
    tc_fence_after();
    const uint32_t tm = tmem_s, tl = tm + ((uint32_t)(q * 32) << 16);
    MmaBar mb{&bar_s, 0};
    const float* bias = reinterpret_cast<const float*>(sm + l.oBias);
    uint8_t *T0 = sm + l.oX, *T1 = sm + l.oHd;
    const uint32_t aT0 = smem_u32(T0), aT1 = smem_u32(T1);
    const uint32_t wd1 = smem_u32(sm + l.oWd1), wd2 = smem_u32(sm + l.oWd2), wc1 = smem_u32(sm + l.oWc1),
                   wc2 = smem_u32(sm + l.oWc2), wc3 = smem_u32(sm + l.oWc3);
    const int64_t ntiles = (M + 127) / 128;
    const uint32_t xbytes = (uint32_t)l.nXc * TCH;
    const uint8_t* fimg = reinterpret_cast<const uint8_t*>(feats);
    uint32_t xpar = 0;      // bit b = phase parity of xbar_s[b]
    int xb = 0;
    if (IMG && (int64_t)blockIdx.x < ntiles && warp == 0 && elect_one()) {
        mbar_expect_tx(&xbar_s[0], xbytes);
        bulk_g2s(sm + l.oXI, fimg + (size_t)blockIdx.x * xbytes, xbytes, &xbar_s[0]);
    }
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, xb ^= 1) {
        const int64_t m = tile * 128 + row;
        const bool valid = m < M;
        const int64_t mm = valid ? m : M - 1;
        if (!IMG) stage_x_coalesced(T0, feats, nullptr, IN, l.INP, tile * 128, M);
        // view embedding of this row's ray: issued now, consumed two MMA phases later
        uint4 pa = make_uint4(0u, 0u, 0u, 0u), pb = pa;
        int64_t r = 0;
        if (want_rgb && (cg == 1 || cg == 2)) {
            r = ridx ? ridx[mm] : mm / S;
            if (pe16) { pa = __ldg(pe16 + r * 4 + 2 * (cg - 1)); pb = __ldg(pe16 + r * 4 + 2 * (cg - 1) + 1); }
        }
        if (IMG) {
            // the other buffer was last read by the first MMA of the previous tile (completed): the next tile may land there
            if (tile + gridDim.x < ntiles && warp == 0 && elect_one()) {
                mbar_expect_tx(&xbar_s[xb ^ 1], xbytes);
                bulk_g2s(sm + l.oXI + (xb ^ 1) * xbytes, fimg + (size_t)(tile + gridDim.x) * xbytes, xbytes, &xbar_s[xb ^ 1]);
            }
            mbar_wait(&xbar_s[xb], (xpar >> xb) & 1u);
            xpar ^= 1u << xb;
        }
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            mma16_fwd(tm, IMG ? smem_u32(sm + l.oXI + xb * xbytes) : aT0, wd1, 64, 64, l.INP, false);
            mb.commit();
        }
        if (!IMG && tile + gridDim.x < ntiles) prefetch_x_l2(feats, nullptr, IN, l.nXc, min((tile + gridDim.x) * 128 + row, M - 1), cg, DC_NCG);
        mb.wait();
        epi_relu16(tl + c16, bias + c16, T1 + 2 * cg * TCH, row);
        sync_to_mma();
        if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + 64, aT1, wd2, 16, 16, 64, false); mb.commit(); }
        mb.wait();
        if (cg == 0) {
            float y[16];
            tmem_ld16(tl + 64, y);
#pragma unroll
            for (int i = 0; i < 16; ++i) y[i] += bias[64 + i];
            if (valid) { sigma[m] = fmaxf(y[0], 0.f); if (y0_raw) y0_raw[m] = y[0]; }   // y0_raw: pre-activation (DD field)
            if (want_rgb) { tile_store8(T0, 0, row, y); tile_store8(T0, 1, row, y + 8); }
        } else if (want_rgb && cg <= 2) {
            if (pe16) stage_cin_pe16(T0, row, cg, pa, pb);
            else stage_cin_pe(T0, row, cg, ray_d[3 * r], ray_d[3 * r + 1], ray_d[3 * r + 2]);
        }
        if (!want_rgb) { tc_fence_before(); __syncthreads(); continue; }
        sync_to_mma();
        if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm, aT0, wc1, 64, 64, 48, false); mb.commit(); }
        mb.wait();
        epi_relu16(tl + c16, bias + 80 + c16, T1 + 2 * cg * TCH, row);
        sync_to_mma();
        if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + 64, aT1, wc2, 64, 64, 64, false); mb.commit(); }
        mb.wait();
        epi_relu16(tl + 64 + c16, bias + 144 + c16, T0 + 2 * cg * TCH, row);
        sync_to_mma();
        if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm, aT0, wc3, 16, 16, 64, false); mb.commit(); }
        mb.wait();
        if (cg == 0) {
            float c[16];
            tmem_ld16(tl, c);
            if (valid) {
#pragma unroll
                for (int j = 0; j < 3; ++j) rgb[3 * m + j] = 1.f / (1.f + __expf(-(c[j] + bias[208 + j])));
            }
        }
        tc_fence_before();
        __syncthreads();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 128);
}

// TMEM columns of the backward kernel (512): two scratch accumulators + five weight-gradient accumulators, each with 16
// extra columns (from the ones tile next to its B operand) whose first column is the bias gradient
#define DCB_S0 0
#define DCB_S1 64
#define DCB_DWD1 128   // [64 x (16 + INP<=64)]   bias col 0,  weights col 16..
#define DCB_DWD2 208   // [16 x (64 + 16)]        weights col 0.., bias col 64
#define DCB_DWC1 288   // [64 x (16 + 48)]        bias col 0,  weights col 16..
#define DCB_DWC2 352   // [64 x (64 + 16)]        weights col 0.., bias col 64
#define DCB_DWC3 432   // [3  x (16 + 64)]        bias col 0,  weights col 16..   -> 512

// per-CTA partial weight gradients (floats): [Wd1 64xIN | Wd2 16x64 | Wc1 64x43 (+pad) | Wc2 64x64 | Wc3 3x64]
struct DcWsLayout { int oWd1, oWd2, oWc1, oWc2, oWc3, total; };
__host__ __device__ inline DcWsLayout dc_ws_layout(int IN) {
    DcWsLayout w;
    int o = 0;
    w.oWd1 = o; o += 64 * IN;
    w.oWd2 = o; o += 16 * 64;
    w.oWc1 = o; o += (64 * CIN + 3) & ~3;
    w.oWc2 = o; o += 64 * 64;
    w.oWc3 = o; o += 3 * 64;
    w.total = o;
    return w;
}

template <bool IMG>
__global__ void __maxnreg__(96) dc_tc_bwd_kernel(const float* __restrict__ feats, const float* __restrict__ lodw,
                                                               const float* __restrict__ ray_d, int S, int64_t M, int IN,
                                                               DcParams p, const float* __restrict__ g_sigma,
                                                               const float* __restrict__ g_rgb, const float* __restrict__ scale_ptr,
                                                               float* __restrict__ g_feats, float* __restrict__ g_dir,
                                                               const int64_t* __restrict__ m_dev, const int64_t* __restrict__ ridx,
                                                               const uint4* __restrict__ pe16, float* __restrict__ ws) {
    if (m_dev) M = min(M, __ldg(m_dev));
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ uint64_t bar_s;
    __shared__ uint64_t xbar_s[2];
    __shared__ uint32_t tmem_s;
    __shared__ float gdir_s[2][128][3];   // view-direction gradient partials of column groups 1 and 2
    const DcTcLayout l = dc_tc_layout(IN, true, IMG);
    const int tid = threadIdx.x, warp = warp_id_uniform(), lane = tid & 31;
    const int q = warp & 3, cg = warp >> 2, row = 32 * q + lane, c16 = 16 * cg;
    dc_tc_stage(sm, l, p, IN, lodw);
    for (int i = tid; i < 3 * 2 * TCH / 16; i += DC_THREADS) {      // the three ones tiles: half(1.0) in feature 0 of every row
        const int t = i / (2 * TCH / 16), j = i - t * (2 * TCH / 16);
        uint4 u = make_uint4(0u, 0u, 0u, 0u);
        if (j < TCH / 16) u.x = 0x00003C00u;
        reinterpret_cast<uint4*>(sm + (t == 0 ? l.oOnesA : (t == 1 ? l.oOnesB : l.oOnesC)))[j] = u;
        if (IMG && t < 2) reinterpret_cast<uint4*>(sm + l.oXI + t * (2 + l.nXc) * TCH)[j] = u;    // ones tile in front of each input buffer
    }
    if (tid == 0) { mbar_init(&bar_s, 1); mbar_init(&xbar_s[0], 1); mbar_init(&xbar_s[1], 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_s, 512);
    sync_to_mma();
    tc_fence_after();
    const uint32_t tm = tmem_s, tl = tm + ((uint32_t)(q * 32) << 16);
    MmaBar mb{&bar_s, 0};
    const float* bias = reinterpret_cast<const float*>(sm + l.oBias);
    uint8_t *G3 = sm + l.oG3, *Gy = sm + l.oGy, *X = sm + l.oX, *Cin = sm + l.oCin, *Hd = sm + l.oHd, *H1 = sm + l.oH1, *H2 = sm + l.oH2;
    const uint32_t aG3 = smem_u32(G3), aGy = smem_u32(Gy), aX = smem_u32(X), aCin = smem_u32(Cin), aHd = smem_u32(Hd),
                   aH1 = smem_u32(H1), aH2 = smem_u32(H2), aOnesA = smem_u32(sm + l.oOnesA), aOnesB = smem_u32(sm + l.oOnesB),
                   aOnesC = smem_u32(sm + l.oOnesC);
    const uint32_t wd1 = smem_u32(sm + l.oWd1), wd2 = smem_u32(sm + l.oWd2), wc1 = smem_u32(sm + l.oWc1),
                   wc2 = smem_u32(sm + l.oWc2), wc3 = smem_u32(sm + l.oWc3);
    float4* pf = reinterpret_cast<float4*>(sm + l.oPF);
    const float scale = scale_ptr ? __ldg(scale_ptr) : 1.f;
    const float inv_scale = 1.f / scale;
    const bool do_rgb = g_rgb != nullptr;
    const int64_t ntiles = (M + 127) / 128;
    const uint32_t xbytes = (uint32_t)l.nXc * TCH, xstride = (uint32_t)(2 + l.nXc) * TCH;
    const uint8_t* fimg = reinterpret_cast<const uint8_t*>(feats);
    uint32_t xpar = 0;
    int xb = 0;
    if (IMG) {
        if ((int64_t)blockIdx.x < ntiles && warp == 0 && elect_one()) {
            mbar_expect_tx(&xbar_s[0], xbytes);
            bulk_g2s(sm + l.oXI + 2 * TCH, fimg + (size_t)blockIdx.x * xbytes, xbytes, &xbar_s[0]);
        }
    } else {
        if ((int64_t)blockIdx.x < ntiles) xpfc_issue<DC_MAXK>(pf, feats, nullptr, IN, (int64_t)blockIdx.x * 128, M);
        cp_async_wait_all();
    }
    __syncthreads();
    bool first = true;
    float* dxs = reinterpret_cast<float*>(sm + l.oDX);
    int64_t dx_tile = -1;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, first = false, xb ^= 1) {
        const int64_t m = tile * 128 + row;
        const bool valid = m < M;
        const int64_t mm = valid ? m : M - 1;
        const uint32_t aXt = IMG ? smem_u32(sm + l.oXI + xb * xstride + 2 * TCH) : aX;      // this tile's input operand
        const uint32_t aOnesXt = IMG ? smem_u32(sm + l.oXI + xb * xstride) : aOnesA;        // ... and the ones tile in front of it
        if (IMG) {
            if (g_feats && dx_tile >= 0 && warp == 0 && elect_one()) bulk_wait_read_all();   // staging tile free again (stored last tile)
            if (tile + gridDim.x < ntiles && warp == 0 && elect_one()) {      // the other buffer's MMAs (previous tile) have completed
                mbar_expect_tx(&xbar_s[xb ^ 1], xbytes);
                bulk_g2s(sm + l.oXI + (xb ^ 1) * xstride + 2 * TCH, fimg + (size_t)(tile + gridDim.x) * xbytes, xbytes, &xbar_s[xb ^ 1]);
            }
            mbar_wait(&xbar_s[xb], (xpar >> xb) & 1u);
            xpar ^= 1u << xb;
        } else {
            if (g_feats && dx_tile >= 0) dx_copy_out(dxs, g_feats, IN, dx_tile * 128, M);      // previous tile's dX
            // ---------------- forward recompute ----------------
            xpfc_consume<DC_NCG, DC_MAXK>(pf, false, IN, l.INP, X, row, cg);
        }
        // this row's upstream gradients / view embedding: issued now, consumed several MMA phases later
        float gs_row = 0.f, gr0 = 0.f, gr1 = 0.f, gr2 = 0.f;
        uint4 pa = make_uint4(0u, 0u, 0u, 0u), pb = pa;
        int64_t r = 0;
        if (cg == 0) {
            if (g_sigma && valid) gs_row = __ldg(g_sigma + m);
            if (do_rgb && valid) { gr0 = __ldg(g_rgb + 3 * m); gr1 = __ldg(g_rgb + 3 * m + 1); gr2 = __ldg(g_rgb + 3 * m + 2); }
        } else if (do_rgb && cg <= 2) {
            r = ridx ? ridx[mm] : mm / S;
            if (pe16) { pa = __ldg(pe16 + r * 4 + 2 * (cg - 1)); pb = __ldg(pe16 + r * 4 + 2 * (cg - 1) + 1); }
        }
        sync_to_mma();
        if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + DCB_S0, aXt, wd1, 64, 64, l.INP, false); mb.commit(); }
        if (!IMG && tile + gridDim.x < ntiles)      // every thread is past its slot reads: the next tile's inputs stream in from here
            xpfc_issue<DC_MAXK>(pf, feats, nullptr, IN, (tile + gridDim.x) * 128, M);
        mb.wait();
        const uint32_t mask_d = epi_relu16(tl + DCB_S0 + c16, bias + c16, Hd + 2 * cg * TCH, row);
        sync_to_mma();
        if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + DCB_S1, aHd, wd2, 16, 16, 64, false); mb.commit(); }
        mb.wait();
        bool y0pos = false;
        float vdir[3] = {0.f, 0.f, 0.f};
        uint32_t mask_1 = 0, mask_2 = 0;
        float dy[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) dy[i] = 0.f;
        if (cg == 0) {
            float y[16];
            tmem_ld16(tl + DCB_S1, y);
#pragma unroll
            for (int i = 0; i < 16; ++i) y[i] += bias[64 + i];
            y0pos = y[0] > 0.f;
            if (do_rgb) { tile_store8(Cin, 0, row, y); tile_store8(Cin, 1, row, y + 8); }
        } else if (do_rgb && cg <= 2) {
            if (pe16 && !g_dir) stage_cin_pe16(Cin, row, cg, pa, pb);
            else {
                vdir[0] = -ray_d[3 * r]; vdir[1] = -ray_d[3 * r + 1]; vdir[2] = -ray_d[3 * r + 2];
                stage_cin_pe(Cin, row, cg, -vdir[0], -vdir[1], -vdir[2]);
            }
        }
        if (do_rgb) {
            sync_to_mma();
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + DCB_S0, aCin, wc1, 64, 64, 48, false); mb.commit(); }
            mb.wait();
            mask_1 = epi_relu16(tl + DCB_S0 + c16, bias + 80 + c16, H1 + 2 * cg * TCH, row);
            sync_to_mma();
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + DCB_S1, aH1, wc2, 64, 64, 64, false); mb.commit(); }
            mb.wait();
            mask_2 = epi_relu16(tl + DCB_S1 + c16, bias + 144 + c16, H2 + 2 * cg * TCH, row);
            sync_to_mma();
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + DCB_S0, aH2, wc3, 16, 16, 64, false); mb.commit(); }
            mb.wait();
            if (cg == 0) {   // d rgb_pre (sigmoid') -> G3 tile (16 features, 3 valid)
                float c[16], g[16];
                tmem_ld16(tl + DCB_S0, c);
#pragma unroll
                for (int j = 0; j < 16; ++j) g[j] = 0.f;
                if (valid) {
                    const float gr[3] = {gr0, gr1, gr2};
#pragma unroll
                    for (int j = 0; j < 3; ++j) {
                        const float sg = 1.f / (1.f + __expf(-(c[j] + bias[208 + j])));
                        g[j] = gr[j] * sg * (1.f - sg) * scale;
                    }
                }
                tile_store8(G3, 0, row, g); tile_store8(G3, 1, row, g + 8);
            }
            // ---------------- color backward ----------------
            sync_to_mma();
            if (warp == 0 && elect_one()) {
                tc_fence_after();
                mma16_bwd_weight(tm + DCB_DWC3, aG3, aOnesC, 80, !first);      // B = ones | H2
                mma16_bwd_data(tm + DCB_S1, aG3, wc3, 64, 16, 16, false);
                mb.commit();
            }
            mb.wait();
            epi_grad16_nb(tl + DCB_S1 + c16, mask_2, H2 + 2 * cg * TCH, row);     // G2 overwrites H2
            sync_to_mma();
            if (warp == 0 && elect_one()) {
                tc_fence_after();
                mma16_bwd_weight(tm + DCB_DWC2, aH2, aH1, 80, !first);         // B = H1 | ones
                mma16_bwd_data(tm + DCB_S0, aH2, wc2, 64, 64, 64, false);
                mb.commit();
            }
            mb.wait();
            epi_grad16_nb(tl + DCB_S0 + c16, mask_1, H1 + 2 * cg * TCH, row);     // G1 overwrites H1
            sync_to_mma();
            if (warp == 0 && elect_one()) {
                tc_fence_after();
                mma16_bwd_weight(tm + DCB_DWC1, aH1, aOnesB, 64, !first);      // B = ones | Cin
                mma16_bwd_data(tm + DCB_S1, aH1, wc1, 48, 64, 64, false);
                mb.commit();
            }
            mb.wait();
            if (cg == 0) {
                tmem_ld16(tl + DCB_S1, dy);      // d cin[0:16] = d y16
            } else if (cg <= 2 && g_dir) {      // d cin[16:43] -> view direction through the positional embedding
                float g[16];
                tmem_ld16(tl + DCB_S1 + c16, g);
                float gv[3] = {0.f, 0.f, 0.f};
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int k = 16 * (cg - 1) + i;      // PE index of this column (cg is warp-uniform)
                    if (k < 3) gv[k] += g[i];
                    else if (k < 3 + 3 * PE_F) { const int f = (k - 3) / 3, c = (k - 3) % 3; const float b = (float)(1 << f); gv[c] += b * cosf(vdir[c] * b) * g[i]; }
                    else if (k < PE_DIM) { const int f = (k - 3 - 3 * PE_F) / 3, c = (k - 3 - 3 * PE_F) % 3; const float b = (float)(1 << f); gv[c] -= b * sinf(vdir[c] * b) * g[i]; }
                }
                gdir_s[cg - 1][row][0] = gv[0]; gdir_s[cg - 1][row][1] = gv[1]; gdir_s[cg - 1][row][2] = gv[2];
            }
            if (g_dir) {
                __syncthreads();
                if (cg == 0 && valid) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) g_dir[3 * m + c] = -(gdir_s[0][row][c] + gdir_s[1][row][c]) * inv_scale;
                }
            }
        } else if (g_dir && valid && cg == 0) {
            g_dir[3 * m] = 0.f; g_dir[3 * m + 1] = 0.f; g_dir[3 * m + 2] = 0.f;
        }
        // ---------------- density backward ----------------
        if (cg == 0) {
            if (y0pos) dy[0] += gs_row * scale;
            if (!valid) {
#pragma unroll
                for (int i = 0; i < 16; ++i) dy[i] = 0.f;
            }
            tile_store8(Gy, 0, row, dy); tile_store8(Gy, 1, row, dy + 8);
        }
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            mma16_bwd_weight(tm + DCB_DWD2, aGy, aHd, 80, !first);             // B = Hd | ones
            mma16_bwd_data(tm + DCB_S0, aGy, wd2, 64, 16, 16, false);
            mb.commit();
        }
        mb.wait();
        epi_grad16_nb(tl + DCB_S0 + c16, mask_d, Hd + 2 * cg * TCH, row);         // Gd overwrites Hd
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            mma16_bwd_weight(tm + DCB_DWD1, aHd, aOnesXt, 16 + l.INP, !first);  // B = ones | X
            if (g_feats) mma16_bwd_data(tm + DCB_S1, aHd, wd1, l.INP, 64, 64, false);
            mb.commit();
        }
        mb.wait();
        if (IMG) {
            // dX leaves as an fp16 operand-image tile, still multiplied by the loss scale (the encoder backward unscales): staged
            // in shared memory in image order, then ONE bulk store of the 12 KB tile by an elected thread
            if (g_feats && c16 < l.INP) {
                float v[16];
                tmem_ld16(tl + DCB_S1 + c16, v);
                tile_store8(sm + l.oDX, 2 * cg, row, v);
                tile_store8(sm + l.oDX, 2 * cg + 1, row, v + 8);
                fence_async_smem();
            }
            dx_tile = tile;
            tc_fence_before();
            __syncthreads();
            if (g_feats && warp == 0 && elect_one()) bulk_s2g(reinterpret_cast<uint8_t*>(g_feats) + (size_t)tile * xbytes, sm + l.oDX, xbytes);
        } else {
            if (g_feats && c16 < l.INP) dx_stage16(tl + DCB_S1, dxs, row, IN, c16, inv_scale);   // W1 carries the LOD weights; written out next tile
            dx_tile = tile;
            cp_async_wait_all();      // own copies landed; the barrier publishes everybody's
            tc_fence_before();
            __syncthreads();
        }
    }
    if (IMG) {
        if (g_feats && dx_tile >= 0 && warp == 0 && elect_one()) bulk_wait_read_all();
    } else if (g_feats && dx_tile >= 0) dx_copy_out(dxs, g_feats, IN, dx_tile * 128, M);
    // ---------------- flush weight / bias gradients (once per CTA) ----------------
    if (!first) {
        tc_fence_after();
        const bool plain = ws != nullptr;      // private partial slice + reduce kernel instead of contended atomics
        const DcWsLayout wl = dc_ws_layout(IN);
        float* wsb = plain ? ws + (size_t)blockIdx.x * wl.total : nullptr;
        float *dWd1 = plain ? wsb + wl.oWd1 : p.gWd1, *dWd2 = plain ? wsb + wl.oWd2 : p.gWd2, *dWc1 = plain ? wsb + wl.oWc1 : p.gWc1,
              *dWc2 = plain ? wsb + wl.oWc2 : p.gWc2, *dWc3 = plain ? wsb + wl.oWc3 : p.gWc3;
        if (c16 < l.INP) {      // G^T X with X unweighted: the LOD weight of each input column applies here
            float v[16];
            tmem_ld16(tl + DCB_DWD1 + 16 + c16, v);
            if (row < 64) {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (c16 + i < IN) {
                        const float x = v[i] * inv_scale * (lodw ? __ldg(lodw + c16 + i) : 1.f);
                        float* d = dWd1 + (size_t)row * IN + c16 + i;
                        if (plain) *d = x; else red_add_f32(d, x);
                    }
            }
        }
        flush_dw16(tl + DCB_DWD2, dWd2, row, 16, 64, c16, inv_scale, plain);
        if (do_rgb) {
            if (c16 < 48) flush_dw16(tl + DCB_DWC1 + 16, dWc1, row, 64, CIN, c16, inv_scale, plain);
            flush_dw16(tl + DCB_DWC2, dWc2, row, 64, 64, c16, inv_scale, plain);
            flush_dw16(tl + DCB_DWC3 + 16, dWc3, row, 3, 64, c16, inv_scale, plain);
        }
        if (cg == 0) {      // bias gradients: the ones-tile column of each accumulator
            float v[16];
            tmem_ld16(tl + DCB_DWD1, v);
            if (row < 64) red_add_f32(p.gbd1 + row, v[0] * inv_scale);
            tmem_ld16(tl + DCB_DWD2 + 64, v);
            if (row < 16) red_add_f32(p.gbd2 + row, v[0] * inv_scale);
            if (do_rgb) {
                tmem_ld16(tl + DCB_DWC1, v);
                if (row < 64) red_add_f32(p.gbc1 + row, v[0] * inv_scale);
                tmem_ld16(tl + DCB_DWC2 + 64, v);
                if (row < 64) red_add_f32(p.gbc2 + row, v[0] * inv_scale);
                tmem_ld16(tl + DCB_DWC3, v);
                if (row < 3) red_add_f32(p.gbc3 + row, v[0] * inv_scale);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 512);
}

// ---------------------------------------------------------------------------------------------
// semantics + instance
// ---------------------------------------------------------------------------------------------
// logits row in TMEM [ncols] (+bias) -> optional softmax with temperature -> global rows.
// `stage` (per-warp [32][33] floats) transposes 32-column blocks so that every global store instruction
// writes one full 128-byte row segment (lanes = columns) instead of 32 strided 4-byte words.
__device__ __forceinline__ void epi_head_out(uint32_t taddr, const float* __restrict__ bias, int C, int CP, bool softmax,
                                             float inv_temp, float* __restrict__ out_tile /* row 0 of this warp */,
                                             int64_t rows_valid /* rows of this warp that exist */, float* stage, int lane) {
    float mx = -INFINITY, sum = 0.f;
    if (softmax) {
        for (int c0 = 0; c0 < CP; c0 += 16) {
            float v[16];
            tmem_ld16(taddr + c0, v);
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (c0 + i < C) {
                    const float z = (v[i] + bias[c0 + i]) * inv_temp;
                    const float nm = fmaxf(mx, z);
                    sum = sum * expf(mx - nm) + expf(z - nm);
                    mx = nm;
                }
        }
    }
    const float inv = softmax ? 1.f / sum : 1.f;
    for (int c0 = 0; c0 < CP; c0 += 32) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (c0 + 16 * h < CP) {
                float v[16];
                tmem_ld16(taddr + c0 + 16 * h, v);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int j = c0 + 16 * h + i;
                    const float z = (v[i] + (j < C ? bias[j] : 0.f)) * inv_temp;
                    stage[lane * 33 + 16 * h + i] = softmax ? expf(z - mx) * inv : z;
                }
            }
        }
        __syncwarp();
        if (c0 + lane < C) {
            for (int r = 0; r < 32 && r < rows_valid; ++r) out_tile[(int64_t)r * C + c0 + lane] = stage[r * 33 + lane];
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128) pan_tc_fwd_kernel(const float* __restrict__ feats, const float* __restrict__ dfeats,
                                                         const float* __restrict__ lodw, int64_t M, int IN, PanParams p,
                                                         int Cs, int Ci, int sem_softmax, int inst_softmax, float inst_inv_temp,
                                                         float* __restrict__ sem, float* __restrict__ inst) {
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ uint64_t bar_s;
    __shared__ uint32_t tmem_s;
    const PanTcLayout l = pan_tc_layout(IN, Cs, Ci, false);
    const int tid = threadIdx.x, warp = warp_id_uniform();
    pan_tc_stage(sm, l, p, IN, Cs, Ci);
    if (tid == 0) { mbar_init(&bar_s, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_s, 256);
    sync_to_mma();
    tc_fence_after();
    const uint32_t tm = tmem_s, tl = tm + ((uint32_t)(warp * 32) << 16);
    MmaBar mb{&bar_s, 0};
    const float* bias = reinterpret_cast<const float*>(sm + l.oBias);
    const float *bs1 = bias, *bs2 = bias + 64, *bi1 = bias + 64 + l.CsP, *bi2 = bi1 + 64, *bi3 = bi2 + 64;
    uint8_t *X = sm + l.oX, *T1 = sm + l.oHs, *T2 = sm + l.oH1;
    const uint32_t aX = smem_u32(X), aT1 = smem_u32(T1), aT2 = smem_u32(T2);
    const uint32_t ws1 = smem_u32(sm + l.oWs1), ws2 = smem_u32(sm + l.oWs2), wi1 = smem_u32(sm + l.oWi1),
                   wi2 = smem_u32(sm + l.oWi2), wi3 = smem_u32(sm + l.oWi3);
    const uint32_t semcol = (Ci > 0) ? (uint32_t)(l.CiP > 64 ? l.CiP : 64) : 128u;   // behind the instance logits and the Hi2 accumulator
    const int64_t ntiles = (M + 127) / 128;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t m = tile * 128 + tid;
        const bool valid = m < M;
        const int64_t mm = valid ? m : M - 1;
        stage_x(X, tid, feats, dfeats, lodw, IN, l.nXc, mm);
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (Cs > 0) mma16_fwd(tm, aX, ws1, 64, 64, l.INP, false);
            if (Ci > 0) mma16_fwd(tm + 64, aX, wi1, 64, 64, l.INP, false);
            mb.commit();
        }
        mb.wait();
        if (Cs > 0) epi_relu64(tl, bs1, T1, tid);
        if (Ci > 0) epi_relu64(tl + 64, bi1, T2, tid);
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (Cs > 0) mma16_fwd(tm + semcol, aT1, ws2, l.CsP, l.CsP, 64, false);
            if (Ci > 0) mma16_fwd(tm, aT2, wi2, 64, 64, 64, false);
            mb.commit();
        }
        mb.wait();
        float* stage = reinterpret_cast<float*>(sm + l.oHs) + warp * (32 * 33);   // T1|T2 (32 KB) are free in the final epilogues
        const int64_t row0 = tile * 128 + warp * 32;
        const int64_t rows_valid = M - row0;
        if (Ci > 0) {
            epi_relu64(tl, bi2, T1, tid);
            sync_to_mma();
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm, aT1, wi3, l.CiP, l.CiP, 64, false); mb.commit(); }
            mb.wait();
            epi_head_out(tl, bi3, Ci, l.CiP, inst_softmax, inst_inv_temp, inst + row0 * Ci, rows_valid, stage, tid & 31);
        }
        if (Cs > 0) {   // semantic head last: the transpose buffer is only free after the instance chain consumed T1/T2
            epi_head_out(tl + semcol, bs2, Cs, l.CsP, sem_softmax, 1.f, sem + row0 * Cs, rows_valid, stage, tid & 31);
        }
        tc_fence_before();
        __syncthreads();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 256);
}

#define PNB_S0 0
#define PNB_S1 64
#define PNB_DWS1 128   // [64 x <=64]
#define PNB_DWS2 192   // [Cs x 64]
#define PNB_DWI1 256   // [64 x <=64]
#define PNB_DWI2 320   // [64 x 64]
#define PNB_DWI3 384   // [Ci(<=256) x 64] as two 128-row blocks -> 512 columns

// d logits of one head from the saved probabilities: g_z = p*(g - <p,g>) / T  (or g / T without softmax).
// prob / g rows are fetched with coalesced 128-byte row segments (lanes = columns) into a per-warp transpose
// buffer `stage` (2 x [32][33] floats) and consumed thread-per-row from there.
__device__ __forceinline__ void head_grad_tile(uint8_t* tile, int row, int lane, const float* __restrict__ prob_w0,
                                               const float* __restrict__ g_w0, int64_t rows_valid, int C, int CP,
                                               bool softmax, float inv_temp, float scale, float* stage,
                                               float* dbacc /* CP/32 rounded up, per lane */) {
    float* sp = stage;
    float* sg = stage + 32 * 33;
    float dot = 0.f;
    if (softmax) {
        for (int c0 = 0; c0 < C; c0 += 32) {
            const bool cok = c0 + lane < C;
            for (int r = 0; r < 32; ++r) {
                const bool ok = cok && r < rows_valid;
                sp[r * 33 + lane] = ok ? __ldg(prob_w0 + (int64_t)r * C + c0 + lane) : 0.f;
                sg[r * 33 + lane] = ok ? __ldg(g_w0 + (int64_t)r * C + c0 + lane) : 0.f;
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 32; ++i) dot = fmaf(sp[lane * 33 + i], sg[lane * 33 + i], dot);
            __syncwarp();
        }
    }
#pragma unroll
    for (int c0 = 0; c0 < 256; c0 += 32) {   // 32 features per pass (one per lane after the scatter); CP <= 256
        if (c0 < CP) {
            const bool cok = c0 + lane < C;
            for (int r = 0; r < 32; ++r) {
                const bool ok = cok && r < rows_valid;
                sp[r * 33 + lane] = ok ? __ldg(prob_w0 + (int64_t)r * C + c0 + lane) : 0.f;
                sg[r * 33 + lane] = ok ? __ldg(g_w0 + (int64_t)r * C + c0 + lane) : 0.f;
            }
            __syncwarp();
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const float pj = sp[lane * 33 + i], gj = sg[lane * 33 + i];
                v[i] = (softmax ? pj * (gj - dot) : gj) * inv_temp * scale;   // zero for padded columns / rows
            }
            __syncwarp();
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c0 + 8 * c < CP) tile_store8(tile, c0 / 8 + c, row, v + 8 * c);
            warp_reduce_scatter<32>(v, lane);   // lane keeps feature c0 + lane
            dbacc[c0 / 32] += v[0];
        }
    }
}

__global__ void __launch_bounds__(128) pan_tc_bwd_kernel(const float* __restrict__ feats, const float* __restrict__ dfeats,
                                                         const float* __restrict__ lodw, int64_t M, int IN, PanParams p,
                                                         int Cs, int Ci, int sem_softmax, int inst_softmax, float inst_inv_temp,
                                                         const float* __restrict__ sem, const float* __restrict__ inst,
                                                         const float* __restrict__ g_sem, const float* __restrict__ g_inst,
                                                         const float* __restrict__ scale_ptr, float* __restrict__ g_panop) {
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ uint64_t bar_s;
    __shared__ uint32_t tmem_s;
    const PanTcLayout l = pan_tc_layout(IN, Cs, Ci, true);
    const int tid = threadIdx.x, warp = warp_id_uniform(), lane = tid & 31;
    pan_tc_stage(sm, l, p, IN, Cs, Ci);
    if (tid == 0) { mbar_init(&bar_s, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc(&tmem_s, 512);
    sync_to_mma();
    tc_fence_after();
    const uint32_t tm = tmem_s, tl = tm + ((uint32_t)(warp * 32) << 16);
    MmaBar mb{&bar_s, 0};
    const float* bias = reinterpret_cast<const float*>(sm + l.oBias);
    const float *bs1 = bias, *bi1 = bias + 64 + l.CsP, *bi2 = bi1 + 64;
    uint8_t *Gs = sm + l.oGs, *X = sm + l.oX, *Hs = sm + l.oHs, *H1 = sm + l.oH1, *H2 = sm + l.oH2, *Gi = sm + l.oGi;
    const uint32_t aGs = smem_u32(Gs), aX = smem_u32(X), aHs = smem_u32(Hs), aH1 = smem_u32(H1), aH2 = smem_u32(H2), aGi = smem_u32(Gi);
    const uint32_t ws1 = smem_u32(sm + l.oWs1), ws2 = smem_u32(sm + l.oWs2), wi1 = smem_u32(sm + l.oWi1),
                   wi2 = smem_u32(sm + l.oWi2), wi3 = smem_u32(sm + l.oWi3);
    const float scale = scale_ptr ? __ldg(scale_ptr) : 1.f;
    const float inv_scale = 1.f / scale;
    const bool do_sem = (Cs > 0) && g_sem, do_inst = (Ci > 0) && g_inst;
    float db_s1[2] = {0.f, 0.f}, db_i1[2] = {0.f, 0.f}, db_i2[2] = {0.f, 0.f}, db_s2[1] = {0.f}, db_i3[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) db_i3[i] = 0.f;
    const int64_t ntiles = (M + 127) / 128;
    bool first = true;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, first = false) {
        const int64_t m = tile * 128 + tid;
        const bool valid = m < M;
        const int64_t mm = valid ? m : M - 1;
        // ---------------- forward recompute of the hidden layers ----------------
        stage_x(X, tid, feats, dfeats, lodw, IN, l.nXc, mm);
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (do_sem) mma16_fwd(tm + PNB_S0, aX, ws1, 64, 64, l.INP, false);
            if (do_inst) mma16_fwd(tm + PNB_S1, aX, wi1, 64, 64, l.INP, false);
            mb.commit();
        }
        mb.wait();
        uint64_t mask_s = 0, mask_1 = 0, mask_2 = 0;
        if (do_sem) mask_s = epi_relu64(tl + PNB_S0, bs1, Hs, tid);
        if (do_inst) mask_1 = epi_relu64(tl + PNB_S1, bi1, H1, tid);
        if (do_inst) {
            sync_to_mma();
            if (warp == 0 && elect_one()) { tc_fence_after(); mma16_fwd(tm + PNB_S0, aH1, wi2, 64, 64, 64, false); mb.commit(); }
            mb.wait();
            mask_2 = epi_relu64(tl + PNB_S0, bi2, H2, tid);
        }
        // ---------------- head gradients from the saved outputs ----------------
        {
            float* stage = reinterpret_cast<float*>(sm + l.oStage) + warp * (2 * 32 * 33);
            const int64_t row0 = tile * 128 + warp * 32;
            const int64_t rows_valid = M - row0;
            if (do_sem) head_grad_tile(Gs, tid, lane, sem + row0 * Cs, g_sem + row0 * Cs, rows_valid, Cs, l.CsP, sem_softmax, 1.f, scale, stage, db_s2);
            if (do_inst) head_grad_tile(Gi, tid, lane, inst + row0 * Ci, g_inst + row0 * Ci, rows_valid, Ci, l.CiP, inst_softmax, inst_inv_temp, scale, stage, db_i3);
        }
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (do_sem) {
                mma16_bwd_weight(tm + PNB_DWS2, aGs, aHs, 64, !first);
                mma16_bwd_data(tm + PNB_S0, aGs, ws2, 64, l.CsP, l.CsP, false);
            }
            if (do_inst) {
                mma16_bwd_weight(tm + PNB_DWI3, aGi, aH2, 64, !first);
                if (l.CiP > 128) mma16_bwd_weight(tm + PNB_DWI3 + 64, aGi + 16 * TCH, aH2, 64, !first);
                mma16_bwd_data(tm + PNB_S1, aGi, wi3, 64, l.CiP, l.CiP, false);
            }
            mb.commit();
        }
        mb.wait();
        if (do_sem) epi_grad64(tl + PNB_S0, mask_s, Hs, tid, lane, db_s1);     // Gs1 overwrites Hs
        if (do_inst) epi_grad64(tl + PNB_S1, mask_2, H2, tid, lane, db_i2);    // Gi2 overwrites H2
        sync_to_mma();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            if (do_sem) {
                mma16_bwd_weight(tm + PNB_DWS1, aHs, aX, l.INP, !first);
                if (g_panop) mma16_bwd_data(tm + PNB_S0, aHs, ws1, l.INP, 64, 64, false);
            }
            if (do_inst) {
                mma16_bwd_weight(tm + PNB_DWI2, aH2, aH1, 64, !first);
                mma16_bwd_data(tm + PNB_S1, aH2, wi2, 64, 64, 64, false);
            }
            mb.commit();
        }
        mb.wait();
        if (do_inst) {
            epi_grad64(tl + PNB_S1, mask_1, H1, tid, lane, db_i1);             // Gi1 overwrites H1
            sync_to_mma();
            if (warp == 0 && elect_one()) {
                tc_fence_after();
                mma16_bwd_weight(tm + PNB_DWI1, aH1, aX, l.INP, !first);
                if (g_panop) mma16_bwd_data(tm + PNB_S0, aH1, wi1, l.INP, 64, 64, do_sem);   // accumulates onto the semantic dX
                mb.commit();
            }
            mb.wait();
        }
        if (g_panop) store_dx(tl + PNB_S0, g_panop + mm * IN, lodw, IN, l.INP, inv_scale, valid);
        tc_fence_before();
        __syncthreads();
    }
    if (!first) {
        tc_fence_after();
        const int f2 = scatter_base(lane, 64), f32i = scatter_base(lane, 32);
        if (do_sem) {
            flush_dw(tl + PNB_DWS1, p.gWs1, tid, 64, IN, l.INP, inv_scale);
            flush_dw(tl + PNB_DWS2, p.gWs2, tid, Cs, 64, 64, inv_scale);
            red_add_f32(p.gbs1 + f2, db_s1[0] * inv_scale); red_add_f32(p.gbs1 + f2 + 1, db_s1[1] * inv_scale);
            if (f32i < Cs) red_add_f32(p.gbs2 + f32i, db_s2[0] * inv_scale);
        }
        if (do_inst) {
            flush_dw(tl + PNB_DWI1, p.gWi1, tid, 64, IN, l.INP, inv_scale);
            flush_dw(tl + PNB_DWI2, p.gWi2, tid, 64, 64, 64, inv_scale);
            flush_dw(tl + PNB_DWI3, p.gWi3, tid, Ci, 64, 64, inv_scale);
            if (l.CiP > 128) flush_dw(tl + PNB_DWI3 + 64, p.gWi3 + (size_t)128 * 64, tid, Ci - 128, 64, 64, inv_scale);
            red_add_f32(p.gbi1 + f2, db_i1[0] * inv_scale); red_add_f32(p.gbi1 + f2 + 1, db_i1[1] * inv_scale);
            red_add_f32(p.gbi2 + f2, db_i2[0] * inv_scale); red_add_f32(p.gbi2 + f2 + 1, db_i2[1] * inv_scale);
            for (int c = 0; c * 32 < l.CiP; ++c)
                if (c * 32 + f32i < Ci) red_add_f32(p.gbi3 + c * 32 + f32i, db_i3[c] * inv_scale);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 512);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// SMs the persistent decoder kernels leave free (pag_set_reserved_sms): with one CTA per SM holding ~all of its shared memory
// and registers nothing else can run beside them -- in particular not the NCCL kernels of a gradient all-reduce that is
// supposed to overlap the backward (measured at 8 GPUs: both 50 MB all-reduces fully exposed, 77 % scaling efficiency)
int pag_reserved_sms = 0;
static int tc_num_sms() {
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
template <typename K>
static int tc_set_smem(K kernel, size_t bytes) {
    if (bytes > 227 * 1024) return PAG_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return e == cudaSuccess ? PAG_OK : (int)e;
}
static void fill_dc(DcParams& p, const float* const* w, float* const* g) {
    p.Wd1 = w[0]; p.bd1 = w[1]; p.Wd2 = w[2]; p.bd2 = w[3]; p.Wc1 = w[4]; p.bc1 = w[5]; p.Wc2 = w[6]; p.bc2 = w[7]; p.Wc3 = w[8]; p.bc3 = w[9];
    if (g) { p.gWd1 = g[0]; p.gbd1 = g[1]; p.gWd2 = g[2]; p.gbd2 = g[3]; p.gWc1 = g[4]; p.gbc1 = g[5]; p.gWc2 = g[6]; p.gbc2 = g[7]; p.gWc3 = g[8]; p.gbc3 = g[9]; }
}
static void fill_pan(PanParams& p, const float* const* w, float* const* g) {
    p.Ws1 = w[0]; p.bs1 = w[1]; p.Ws2 = w[2]; p.bs2 = w[3]; p.Wi1 = w[4]; p.bi1 = w[5]; p.Wi2 = w[6]; p.bi2 = w[7]; p.Wi3 = w[8]; p.bi3 = w[9];
    if (g) { p.gWs1 = g[0]; p.gbs1 = g[1]; p.gWs2 = g[2]; p.gbs2 = g[3]; p.gWi1 = g[4]; p.gbi1 = g[5]; p.gWi2 = g[6]; p.gbi2 = g[7]; p.gWi3 = g[8]; p.gbi3 = g[9]; }
}

extern "C" {

int pag_decode_dc_fwd_tc(const float* feats, const float* lodw, const float* ray_d, int S, int64_t M, int IN,
                         const float* const* weights, int hidden, int view_dim, int want_rgb, float* sigma, float* rgb,
                         void* stream) {
    if (hidden != H || view_dim != PE_DIM || IN < 1 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M == 0) return PAG_OK;
    DcParams p{};
    fill_dc(p, weights, nullptr);
    const DcTcLayout l = dc_tc_layout(IN, false);
    int rc = tc_set_smem(dc_tc_fwd_kernel<false>, l.total);
    if (rc) return rc;
    const int64_t tiles = (M + 127) / 128;
    const int64_t cap = 2 * (int64_t)tc_num_sms();
    dc_tc_fwd_kernel<false><<<(int)(tiles < cap ? tiles : cap), DC_THREADS, l.total, (cudaStream_t)stream>>>(feats, lodw, ray_d, S, M, IN, p, want_rgb, sigma, rgb, nullptr, nullptr, nullptr, nullptr);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// device-side sample count (m_dev[0] <= M_max) and per-sample ray index: sample m uses ray_d[ridx[m]]
int pag_decode_dc_fwd_tc_dyn(const float* feats, const float* lodw, const float* ray_d, const int64_t* ridx, int64_t M_max,
                             const int64_t* m_dev, int IN, const float* const* weights, int hidden, int view_dim,
                             int want_rgb, float* sigma, float* rgb, float* y0_raw, const void* view_pe16, int feats_img16,
                             void* stream) {
    if (hidden != H || view_dim != PE_DIM || IN < 1 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (feats_img16 && (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M_max == 0) return PAG_OK;
    DcParams p{};
    fill_dc(p, weights, nullptr);
    const DcTcLayout l = dc_tc_layout(IN, false, feats_img16 != 0);
    const int64_t tiles = (M_max + 127) / 128;
    const int64_t cap = 2 * (int64_t)tc_num_sms();
    const int grid = (int)(tiles < cap ? tiles : cap);
    const uint4* pe = reinterpret_cast<const uint4*>(view_pe16);
    if (feats_img16) {
        int rc = tc_set_smem(dc_tc_fwd_kernel<true>, l.total);
        if (rc) return rc;
        dc_tc_fwd_kernel<true><<<grid, DC_THREADS, l.total, (cudaStream_t)stream>>>(feats, lodw, ray_d, 1, M_max, IN, p, want_rgb, sigma, rgb, m_dev, ridx, pe, y0_raw);
    } else {
        int rc = tc_set_smem(dc_tc_fwd_kernel<false>, l.total);
        if (rc) return rc;
        dc_tc_fwd_kernel<false><<<grid, DC_THREADS, l.total, (cudaStream_t)stream>>>(feats, lodw, ray_d, 1, M_max, IN, p, want_rgb, sigma, rgb, m_dev, ridx, pe, y0_raw);
    }
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

// grad_scale: device pointer to one float (power of two) or NULL (= 1)
int pag_decode_dc_bwd_tc(const float* feats, const float* lodw, const float* ray_d, int S, int64_t M, int IN,
                         const float* const* weights, float* const* grads, int hidden, int view_dim,
                         const float* g_sigma, const float* g_rgb, const float* grad_scale, float* g_feats, float* g_dir,
                         void* stream) {
    if (hidden != H || view_dim != PE_DIM || IN < 1 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M == 0) return PAG_OK;
    DcParams p{};
    fill_dc(p, weights, grads);
    const DcTcLayout l = dc_tc_layout(IN, true);
    int rc = tc_set_smem(dc_tc_bwd_kernel<false>, l.total);
    if (rc) return rc;
    const int64_t tiles = (M + 127) / 128;
    const int64_t cap = tc_num_sms();
    dc_tc_bwd_kernel<false><<<(int)(tiles < cap ? tiles : cap), DC_THREADS, l.total, (cudaStream_t)stream>>>(
        feats, lodw, ray_d, S, M, IN, p, g_sigma, g_rgb, grad_scale, g_feats, g_dir, nullptr, nullptr, nullptr, nullptr);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

int pag_decode_dc_bwd_tc_dyn(const float* feats, const float* lodw, const float* ray_d, const int64_t* ridx, int64_t M_max,
                             const int64_t* m_dev, int IN, const float* const* weights, float* const* grads, int hidden,
                             int view_dim, const float* g_sigma, const float* g_rgb, const float* grad_scale, float* g_feats,
                             float* g_dir, const void* view_pe16, float* workspace, int64_t workspace_bytes, int img16,
                             void* stream) {
    if (hidden != H || view_dim != PE_DIM || IN < 1 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (img16 && (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M_max == 0) return PAG_OK;
    DcParams p{};
    fill_dc(p, weights, grads);
    const DcTcLayout l = dc_tc_layout(IN, true, img16 != 0);
    const int64_t tiles = (M_max + 127) / 128;
    const int64_t cap = tc_num_sms();
    const int nblocks = (int)(tiles < cap ? tiles : cap);
    const DcWsLayout wl = dc_ws_layout(IN);
    float* ws = (workspace && workspace_bytes >= (int64_t)nblocks * wl.total * 4 && !(reinterpret_cast<uintptr_t>(workspace) & 15)) ? workspace : nullptr;
    const uint4* pe = reinterpret_cast<const uint4*>(view_pe16);
    if (img16) {
        int rc = tc_set_smem(dc_tc_bwd_kernel<true>, l.total);
        if (rc) return rc;
        dc_tc_bwd_kernel<true><<<nblocks, DC_THREADS, l.total, (cudaStream_t)stream>>>(
            feats, lodw, ray_d, 1, M_max, IN, p, g_sigma, g_rgb, grad_scale, g_feats, g_dir, m_dev, ridx, pe, ws);
    } else {
        int rc = tc_set_smem(dc_tc_bwd_kernel<false>, l.total);
        if (rc) return rc;
        dc_tc_bwd_kernel<false><<<nblocks, DC_THREADS, l.total, (cudaStream_t)stream>>>(
            feats, lodw, ray_d, 1, M_max, IN, p, g_sigma, g_rgb, grad_scale, g_feats, g_dir, m_dev, ridx, pe, ws);
    }
    PAG_LAUNCH_CHECK();
    if (ws) {
        const bool rgb = g_rgb != nullptr;
        WsSegs sg{5, {wl.oWd1, wl.oWd2, wl.oWc1, wl.oWc2, wl.oWc3}, {64 * IN, 16 * 64, 64 * CIN, 64 * 64, 3 * 64},
                  {p.gWd1, p.gWd2, rgb ? p.gWc1 : nullptr, rgb ? p.gWc2 : nullptr, rgb ? p.gWc3 : nullptr}};
        ws_reduce_kernel<<<dim3((wl.total + 255) / 256, WS_GROUPS), 256, 0, (cudaStream_t)stream>>>(ws, nblocks, M_max, m_dev, wl.total, sg);
        PAG_LAUNCH_CHECK();
    }
    return PAG_OK;
}

// bytes of partial-gradient workspace pag_decode_dc_bwd_tc_dyn can use for M_max samples
int pag_decode_dc_bwd_workspace(int64_t M_max, int IN, int64_t* bytes) {
    if (!bytes) return PAG_ERR_ARG;
    const int64_t tiles = (M_max + 127) / 128, cap = tc_num_sms();
    *bytes = (tiles < cap ? tiles : cap) * (int64_t)dc_ws_layout(IN).total * 4;
    return PAG_OK;
}

// n SMs stay free of persistent decoder CTAs (0 = use all); returns the previous value
int pag_set_reserved_sms(int n, int* previous) {
    if (n < 0 || n > 120) return PAG_ERR_ARG;
    if (previous) *previous = pag_reserved_sms;
    pag_reserved_sms = n;
    return PAG_OK;
}

// per-ray view embedding image pe16[R][32] (fp16: 27 values of PE(-d), 5 zeros) for the *_dyn decoders
int pag_view_pe16(const float* ray_d, int64_t R, void* pe16, void* stream) {
    if (R == 0) return PAG_OK;
    view_pe16_kernel<<<(unsigned)((R + 127) / 128), 128, 0, (cudaStream_t)stream>>>(ray_d, R, reinterpret_cast<__half*>(pe16));
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

int pag_decode_pan_fwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                          const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                          float inst_temperature, float* sem, float* inst, void* stream) {
    if (hidden != H || Cs < 0 || Ci < 0 || Cs > 32 || Ci > 224 || IN < 1 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M == 0 || (Cs == 0 && Ci == 0)) return PAG_OK;
    PanParams p{};
    fill_pan(p, weights, nullptr);
    const PanTcLayout l = pan_tc_layout(IN, Cs, Ci, false);
    int rc = tc_set_smem(pan_tc_fwd_kernel, l.total);
    if (rc) return rc;
    const float it = inst_temperature > 0.f ? 1.f / inst_temperature : 1.f;
    const int64_t tiles = (M + 127) / 128;
    const int64_t cap = 2 * (int64_t)tc_num_sms();
    pan_tc_fwd_kernel<<<(int)(tiles < cap ? tiles : cap), 128, l.total, (cudaStream_t)stream>>>(
        feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax, inst_softmax, it, sem, inst);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

int pag_decode_pan_bwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                          const float* const* weights, float* const* grads, int hidden, int Cs, int Ci, int sem_softmax,
                          int inst_softmax, float inst_temperature, const float* sem, const float* inst,
                          const float* g_sem, const float* g_inst, const float* grad_scale, float* g_panop, void* stream) {
    if (hidden != H || Cs < 0 || Ci < 0 || Cs > 32 || Ci > 256 || IN < 1 || IN > 64 || (IN & 3)) return PAG_ERR_UNSUPPORTED;
    if (M == 0 || (Cs == 0 && Ci == 0)) return PAG_OK;
    PanParams p{};
    fill_pan(p, weights, grads);
    const PanTcLayout l = pan_tc_layout(IN, Cs, Ci, true);
    int rc = tc_set_smem(pan_tc_bwd_kernel, l.total);
    if (rc) return rc;
    const float it = inst_temperature > 0.f ? 1.f / inst_temperature : 1.f;
    const int64_t tiles = (M + 127) / 128;
    const int64_t cap = tc_num_sms();
    pan_tc_bwd_kernel<<<(int)(tiles < cap ? tiles : cap), 128, l.total, (cudaStream_t)stream>>>(
        feats, dfeats, lodw, M, IN, p, Cs, Ci, sem_softmax, inst_softmax, it, sem, inst, g_sem, g_inst, grad_scale, g_panop);
    PAG_LAUNCH_CHECK();
    return PAG_OK;
}

}  // extern "C"
