/* pagnerf_b200 -- C ABI of the B200-native PAg-NeRF per-ray hot path (libpagnerf_b200.so).
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); kernels never allocate/free;
 *   - sizes are int64_t, small dims int; `stream` is a cudaStream_t passed as void*;
 *   - return 0 on success, <0 argument/unsupported-shape error (PAG_ERR_*), >0 a cudaError_t;
 *   - no host synchronisation, no global state, re-entrant per stream;
 *   - "nullable" arguments may be NULL to skip the corresponding channel.
 * The reference is pure Python on top of kaolin / kaolin-wisp / permutohedral_encoding / tiny-cuda-nn;
 * each entry below cites the reference call site (file:line under the reference tree) whose
 * third-party kernel(s) it replaces.  The Python binding a maintainer adds is in INTEGRATION.md.
 */
#ifndef PAGNERF_B200_H
#define PAGNERF_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PAG_OK 0
#define PAG_ERR_ARG (-1)
#define PAG_ERR_UNSUPPORTED (-2)

/* ---- occupancy octree: grids/occtree.py:85-91 -> wisp OctreeAS.{query,raytrace,raymarch} ------------- */

/* kaolin.ops.spc.unbatched_query: coords f32[P,3] in [-1,1] -> point-hierarchy index (or -1). */
int pag_octree_query(const uint8_t* octree, const int32_t* prefix, const float* coords, int64_t P, int level,
                     int32_t* pidx, void* stream);

/* exclusive scan of int32 counts; out has N+1 entries, out[N] = total. */
int pag_exclusive_scan_i32(const int32_t* in, int64_t N, int64_t* out, void* stream);
/* ---- live-sample compaction (training hot path; no reference counterpart: the reference decodes every packed sample) ----
 * Samples with density exactly 0 have integration weight 0 and receive gradient 0, so removing them from the packed list
 * before the remaining decoders / the delta-grid encode / the backward is exact.  offsets i64[N+1] describes the packed list
 * (ray r owns [offsets[r], offsets[r+1])); pag_compact_count writes counts i32[N] and the compacted offsets_c i64[N+1]
 * (offsets_c[N] = number of live samples, stays on the device); pag_compact_emit copies the survivors in order. */
int pag_compact_count(const float* sigma, const int64_t* offsets, int64_t N, int32_t* counts, int64_t* offsets_c, void* stream);
int pag_compact_emit(const float* sigma, const int64_t* offsets, const int64_t* offsets_c, int64_t N, const float* samples,
                     const float* depths, const float* deltas, const float* feats, int F, int64_t* ridx_c, float* samples_c,
                     float* depths_c, float* deltas_c, float* feats_c, void* stream);

/* 'ray' raymarch, pass 1 (tracers/panoptic_packed_rf_tracer.py:85 with raymarch_type='ray'):
 * S jittered steps per ray, octree lookup per step.  Writes pidx_tmp[N*S], counts[N], offsets[N+1].
 * jitter f32[N,S] nullable (then the counter RNG with `seed` is used); linspace = torch.linspace(0,1,S).
 * seed_dev (nullable): device word overriding `seed`, so that CUDA-graph replays can advance the jitter stream. */
int pag_march_ray_count(const float* origins, const float* dirs, int64_t N, int S, const float* linspace,
                        const float* jitter, uint32_t seed, float dist_min, float dist_range,
                        const uint8_t* octree, const int32_t* prefix, int level,
                        int32_t* pidx_tmp, int32_t* counts, int64_t* offsets, const uint32_t* seed_dev, void* stream);
/* pass 2: packed outputs of size M = offsets[N]: ridx/pidx i64[M], samples f32[M,3], depths/deltas f32[M],
 * boundary u8[M]. */
int pag_march_ray_emit(const float* origins, const float* dirs, int64_t N, int S, const float* linspace,
                       const float* jitter, uint32_t seed, float dist_min, float dist_range,
                       const int32_t* pidx_tmp, const int64_t* offsets,
                       int64_t* ridx, int64_t* pidx, float* samples, float* depths, float* deltas,
                       uint8_t* boundary, const uint32_t* seed_dev, void* stream);

/* 'ray' raymarch against an occupancy BIT FIELD of the marching level, without point indices (the fused training trace
 * never reads pidx).  pag_octree_level_bits derives bits u32[8^level / 32] (bit (ix*res + iy)*res + iz) from the octree once
 * per octree change; the count pass leaves step masks u32[N * ceil(S/32)] for the emit pass.  Same kept set, same
 * ridx / samples / depths / deltas as pag_march_ray_{count,emit}. */
int pag_octree_level_bits(const uint8_t* octree, const int32_t* prefix, int level, uint32_t* bits, void* stream);
int pag_march_ray_bits_count(const float* origins, const float* dirs, int64_t N, int S, const float* linspace,
                             const float* jitter, uint32_t seed, float dist_min, float dist_range, const uint32_t* bits, int level,
                             uint32_t* masks, int32_t* counts, int64_t* offsets, const uint32_t* seed_dev, void* stream);
int pag_march_ray_bits_emit(const float* origins, const float* dirs, int64_t N, int S, const float* linspace,
                            const float* jitter, uint32_t seed, float dist_min, float dist_range, const uint32_t* masks,
                            const int64_t* offsets, int64_t* ridx, float* samples, float* depths, float* deltas,
                            const uint32_t* seed_dev, void* stream);

/* kaolin.render.spc.unbatched_raytrace(return_depth, with_exit): count pass then emit pass;
 * nuggets (ridx,pidx,[entry,exit]) in kaolin's order.  offsets[N+1] doubles as the per-ray first-nugget index. */
int pag_raytrace_count(const uint8_t* octree, const int32_t* prefix, const float* origins, const float* dirs,
                       int64_t N, int level, int32_t* counts, int64_t* offsets, void* stream);
int pag_raytrace_emit(const uint8_t* octree, const int32_t* prefix, const float* origins, const float* dirs,
                      int64_t N, int level, const int64_t* offsets, int64_t* ridx, int64_t* pidx, float* depth,
                      void* stream);
/* 'voxel' raymarch sampling (wisp sample_from_depth_intervals + addcmul + expand_pack_boundary):
 * samples f32[K,S,3], depths f32[K,S], deltas f32[K*S], boundary u8[K*S]. */
int pag_voxel_samples(const float* origins, const float* dirs, const int64_t* ridx, const float* depth, int64_t K,
                      int S, const float* jitter, uint32_t seed, float* samples, float* depths, float* deltas,
                      uint8_t* boundary, void* stream);
/* max-travel filter, tracers/panoptic_packed_rf_tracer.py:88-99: keep[k] u8. */
int pag_max_travel_mask(const int64_t* ridx, const float* depths, int64_t K, int S, const int64_t* ray_first,
                        float max_travel, uint8_t* keep, void* stream);
/* kaolin.render.spc.mark_pack_boundaries, tracers/panoptic_packed_rf_tracer.py:114. */
/* Sync-free 'voxel' marching for the fused training trace (configs/bup20/best.yaml:34 switches the trainer to voxel marching at
 * epoch 201, pc_nerf/trainer.py:362-366): after pag_raytrace_count / pag_raytrace_emit into worst-case nugget buffers, the max-travel
 * filter of tracers/panoptic_packed_rf_tracer.py:88-108 is folded into the kept-nugget count (rel i32[K_max]: rank among the ray's kept
 * nuggets or -1; offsets i64[N+1]: packed SAMPLE offsets, offsets[N] = M stays on the device) and the emit pass writes the S samples
 * of every kept nugget into the packed list.  Jitter index = k*S + s with k the unfiltered nugget index (== pag_voxel_samples). */
int pag_voxel_filter_count(const float* nug_depth, const int64_t* nug_offsets, int64_t N, int S, uint32_t seed, const uint32_t* seed_dev,
                           float max_travel, int apply_filter, int32_t* rel, int32_t* counts, int64_t* offsets, void* stream);
int pag_voxel_emit_dyn(const float* origins, const float* dirs, const int64_t* nug_ridx, const float* nug_depth, const int32_t* rel,
                       const int64_t* nug_offsets, const int64_t* offsets, int64_t N, int64_t K_max, int S, uint32_t seed,
                       const uint32_t* seed_dev, int64_t* ridx, float* samples, float* depths, float* deltas, void* stream);
/* One-traversal variant of the sync-free voxel chain: the raytrace stages every ray's nuggets in its own row of
 * stage_depth f32[N, stage_cap, 2] (stage_cap >= 3 * 2^level - 2) while counting; filter and emit read the rows (rel i32[N, stage_cap]).
 * With slot_counts (and level >= 2) the traversal is split 64 ways per ray: thread (ray, i1, i2) walks the i2-th child of the i1-th
 * child of the root in the ray's own visiting order; a count pass and a write pass, both 64x wider than the per-ray DFS. */
int pag_raytrace_stage(const uint8_t* octree, const int32_t* prefix, const float* origins, const float* dirs, int64_t N, int level,
                       int64_t stage_cap, int32_t* counts, int64_t* nug_offsets, float* stage_depth, int32_t* slot_counts /* i32[N*64], nullable */,
                       void* stream);
int pag_voxel_filter_count_staged(const float* stage_depth, const int64_t* nug_offsets, int64_t N, int64_t stage_cap, int S, uint32_t seed,
                                  const uint32_t* seed_dev, float max_travel, int apply_filter, int32_t* rel, int32_t* counts,
                                  int64_t* offsets, void* stream);
int pag_voxel_emit_staged(const float* origins, const float* dirs, const float* stage_depth, const int32_t* rel, const int64_t* nug_offsets,
                          const int64_t* offsets, int64_t N, int64_t stage_cap, int S, uint32_t seed, const uint32_t* seed_dev,
                          int64_t* ridx, float* samples, float* depths, float* deltas, void* stream);
/* Octree rebuild on the device (prune(): pc_nerf/panoptic_delta_nef.py:63-104, pc_nerf/panoptic_nef.py:207-237 -> kaolin
 * unbatched_points_to_octree + wisp OctreeAS.init, SURVEY 3.4 / 8f rank 4): from the dense leaf-occupancy mask u8[8^level] in Morton
 * order to the SPC layout the marcher consumes.  Workspaces and outputs hold F = (8^(level+1)-1)/7 entries (see csrc/octree.cu);
 * pyramid i32[2, level+2] stays on the device: n_nodes = pyramid[1][level], n_points = pyramid[1][level+1]. */
int pag_octree_from_mask(const uint8_t* mask, int level, int32_t* exists, uint8_t* bytes, int64_t* pos, int32_t* popc, int64_t* prefix64,
                         uint8_t* octree, int16_t* points, int32_t* prefix, int32_t* pyramid, void* stream);
int pag_mark_pack_boundaries(const int64_t* ids, int64_t M, uint8_t* boundary, void* stream);

/* ---- permutohedral encoding: grids/permuto_grid.py:57-62,71 -> PermutoEncoding fwd / bwd ------------- */
/* pos f32[M,3]; table f32[L,capacity,F]; scale_factor/shift f32[L,3]; anneal f32[L]; out f32[M,L*F]. F must be 2. */
int pag_permuto_fwd(const float* pos, int64_t M, const float* table, int64_t capacity, int L, int F,
                    const float* scale_factor, const float* shift, const float* anneal, float* out, void* stream);
/* grad_table f32[L,capacity,F] is accumulated into; grad_pos f32[M,3] nullable (delta grid: NULL,
 * pc_nerf/panoptic_delta_nef.py:215). n_agg_levels = number of coarse levels scattered with warp aggregation. */
int pag_permuto_bwd(const float* pos, int64_t M, const float* table, int64_t capacity, int L, int F,
                    const float* scale_factor, const float* shift, const float* anneal, const float* grad_out,
                    float* grad_table, float* grad_pos, int n_agg_levels, void* stream);
/* variants for the sync-free fused trace: the packed-sample count is read on the device (m_dev[0] <= M_max, written by
 * the marcher's scan), pos_half rounds positions to fp16 first (autocast, grids/permuto_grid.py:65,71). */
int pag_permuto_fwd_dyn(const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table,
                        int64_t capacity, int L, int F, const float* scale_factor, const float* shift, const float* anneal,
                        float* out, void* stream);
int pag_permuto_bwd_dyn(const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table,
                        int64_t capacity, int L, int F, const float* scale_factor, const float* shift, const float* anneal,
                        const float* grad_out, float* grad_table, float* grad_pos, int n_agg_levels, void* stream);
/* fp16 operand-image interchange with the tensor-core decoders (fused trace): features / feature gradients as tiles of 128
 * samples, each [2L/8 chunks][128 rows][8 halfs] (the UMMA operand image, 12 KB for L = 24) -- one bulk copy per tile on the
 * decoder side, coalesced 16-byte accesses on the encoder side, half the bytes.  img16 holds ceil(M_max/128) tiles; rows past the
 * sample count in the last tile are zero-filled.  grad_img16 is still multiplied by the decoders' loss scale *img_scale. L % 4 == 0. */
int pag_permuto_fwd_img16_dyn(const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table,
                              int64_t capacity, int L, int F, const float* scale_factor, const float* shift, const float* anneal,
                              void* img16, void* stream);
int pag_permuto_bwd_img16_dyn(const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table,
                              int64_t capacity, int L, int F, const float* scale_factor, const float* shift, const float* anneal,
                              const void* grad_img16, const float* img_scale, float* grad_table, float* grad_pos, int n_agg_levels,
                              int level_begin, int level_end, void* stream);
/* [level_begin, level_end): the levels this launch scatters (0, L for all).  Splitting the table into level ranges lets the
 * all-reduce of a finished range overlap the scatter of the next; grad_pos is written by the range starting at 0 and
 * accumulated by the others. */
/* parity probe: lattice vertex hash indices u32[L,M,4], ranks i32[L,M,4], barycentric f32[L,M,4]. */
int pag_permuto_indices(const float* pos, int64_t M, int64_t capacity, int L, const float* scale_factor,
                        const float* shift, uint32_t* idx, int32_t* rank, float* bary, void* stream);

/* ---- hash grids: flavour 0 = tiny-cuda-nn (grids/hash_grid_tinycudann.py:24-34,41),
 *                  flavour 1 = HashNeRF torch grid (grids/hash_grid_torch.py:13-108) ------------------- */
int pag_hash_fwd(int flavour, const float* pos, int64_t M, const float* table, int L, int F, const float* fparam,
                 const uint32_t* res, const uint32_t* offset, const uint32_t* size, float* out, int round_half,
                 void* stream);
int pag_hash_bwd(int flavour, const float* pos, int64_t M, const float* table, int L, int F, const float* fparam,
                 const uint32_t* res, const uint32_t* offset, const uint32_t* size, const float* grad_out,
                 float* grad_table, float* grad_pos, int n_agg_levels, void* stream);
/* variants for the sync-free fused trace (device-side sample count, optional fp16 rounding of the positions) */
int pag_hash_fwd_dyn(int flavour, const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table, int L,
                     int F, const float* fparam, const uint32_t* res, const uint32_t* offset, const uint32_t* size, float* out,
                     int round_half, void* stream);
int pag_hash_bwd_dyn(int flavour, const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table, int L,
                     int F, const float* fparam, const uint32_t* res, const uint32_t* offset, const uint32_t* size,
                     const float* grad_out, float* grad_table, float* grad_pos, int n_agg_levels, void* stream);
/* fp16 operand-image interchange with the tensor-core decoders inside the fused trace (same layout as
 * pag_permuto_fwd_img16_dyn: tiles of 128 samples, ceil(2L/16)*2 chunks [128 rows][8 halfs], zero padded); the gradient image is
 * scaled by *img_scale (device float, nullable = 1).  Replaces grids/hash_grid_tinycudann.py:41 / grids/hash_grid_torch.py:95-108
 * on the training path (the reference's autocast hands the decoders half features as well). */
int pag_hash_fwd_img16_dyn(int flavour, const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table, int L,
                           int F, const float* fparam, const uint32_t* res, const uint32_t* offset, const uint32_t* size, void* img16,
                           void* stream);
int pag_hash_bwd_img16_dyn(int flavour, const float* pos, int64_t M_max, const int64_t* m_dev, int pos_half, const float* table, int L,
                           int F, const float* fparam, const uint32_t* res, const uint32_t* offset, const uint32_t* size,
                           const void* grad_img16, const float* img_scale, float* grad_table, float* grad_pos, int n_agg_levels,
                           void* stream);
int pag_hash_indices(int flavour, const float* pos, int64_t M, int L, const float* fparam, const uint32_t* res,
                     const uint32_t* offset, const uint32_t* size, uint32_t* idx, void* stream);

/* ---- decoders: pc_nerf/panoptic_nef.py:114-164,309-361; pc_nerf/panoptic_delta_nef.py:184-257 -------- */
/* density IN->64->16 (+relu on ch0) and color [16|PE(-d)]->64->64->3 sigmoid.
 * weights: Wd1,bd1,Wd2,bd2,Wc1,bc1,Wc2,bc2,Wc3,bc3 (torch Linear [out][in]); sample m uses ray_d[m / S]. */
int pag_decode_dc_fwd(const float* feats, const float* lodw, const float* ray_d, int S, int64_t M, int IN,
                      const float* const* weights, int hidden, int view_dim, int want_rgb, float* sigma, float* rgb,
                      void* stream);
int pag_decode_dc_bwd(const float* feats, const float* lodw, const float* ray_d, int S, int64_t M, int IN,
                      const float* const* weights, float* const* grads, int hidden, int view_dim,
                      const float* g_sigma, const float* g_rgb, float* g_feats, float* g_dir, void* stream);
/* semantics IN->64->Cs and instance IN->64->64->Ci on panop = (feats + dfeats) * lodw, optional softmax / temperature.
 * weights: Ws1,bs1,Ws2,bs2,Wi1,bi1,Wi2,bi2,Wi3,bi3. */
int pag_decode_pan_fwd(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                       const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                       float inst_temperature, float* sem, float* inst, void* stream);
int pag_decode_pan_bwd(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                       const float* const* weights, float* const* grads, int hidden, int Cs, int Ci, int sem_softmax,
                       int inst_softmax, float inst_temperature, const float* sem, const float* inst,
                       const float* g_sem, const float* g_inst, float* g_panop, void* stream);
/* linear scalar head y[m] = b + sum_k (feats + dfeats)[m,k] * lodw[k] * w[k]: PanopticDDensityNeF's delta-density decoder
 * (pc_nerf/panoptic_dd_nef.py:41-58, BasicDecoder with activation 'none' = one linear map, collapsed on the host).
 * dfeats / lodw / g_x nullable; g_w f32[IN] and g_b f32[1] accumulate (caller zeroes). */
int pag_linear_head_fwd(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN, const float* w,
                        const float* b, float* y, void* stream);
int pag_linear_head_bwd(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN, const float* w,
                        const float* g, float* g_x, float* g_w, float* g_b, void* stream);
/* fused-trace variants (device-side sample count): y = post * relu?(pre + head(x)) -- the DD field's tau_p =
 * relu(y0.detach() + delta_density) * delta in one pass; the backward gates g with the forward output `gate` (ReLU), multiplies
 * it by post and can accumulate into g_x. */
int pag_linear_head_fwd_dyn(const float* feats, const float* dfeats, const float* lodw, int64_t M_max, const int64_t* m_dev, int IN,
                            const float* w, const float* b, const float* pre, int relu, const float* post, float* y, int x_img16,
                            void* stream);
int pag_linear_head_bwd_dyn(const float* feats, const float* dfeats, const float* lodw, int64_t M_max, const int64_t* m_dev, int IN,
                            const float* w, const float* g, const float* gate, const float* post, float* g_x, int accumulate_x,
                            float* g_w, float* g_b, int x_img16, const float* img_scale, void* stream);
/* x_img16 != 0: feats / dfeats / g_x are fp16 operand images (g_x accumulated, multiplied by *img_scale like the heads' dX). */
/* DD tracer backward glue (tracers/panoptic_dd_packed_rf_tracer.py:128-162): gw[s] = alpha_p[ray] * (gw_sem + gw_inst)[s]
 * + sum_c g[ray][c] out[ray][c] / alpha_p[ray], the gradient of the loss w.r.t. the panoptic integration weights. */
int pag_dd_weight_grads(const float* g_sem, const float* out_sem, int Cs, const float* g_inst, const float* out_inst, int Ci,
                        const float* alpha_p, const float* gw_sem, const float* gw_inst, const int64_t* offsets, int64_t R,
                        float* gw, void* stream);

/* tensor-core (tcgen05, fp16 operands / fp32 accumulate) variants of the four decoder entry points: the numerics of
 * the reference's autocast training step (pc_nerf/trainer.py:429).  grad_scale: device pointer to one power-of-two
 * float applied to the upstream gradients before the fp16 repack and divided out of every result (NULL = 1). */
int pag_decode_dc_fwd_tc(const float* feats, const float* lodw, const float* ray_d, int S, int64_t M, int IN,
                         const float* const* weights, int hidden, int view_dim, int want_rgb, float* sigma, float* rgb,
                         void* stream);
int pag_decode_dc_bwd_tc(const float* feats, const float* lodw, const float* ray_d, int S, int64_t M, int IN,
                         const float* const* weights, float* const* grads, int hidden, int view_dim,
                         const float* g_sigma, const float* g_rgb, const float* grad_scale, float* g_feats, float* g_dir,
                         void* stream);
int pag_decode_dc_fwd_tc_dyn(const float* feats, const float* lodw, const float* ray_d, const int64_t* ridx, int64_t M_max,
                             const int64_t* m_dev, int IN, const float* const* weights, int hidden, int view_dim,
                             int want_rgb, float* sigma, float* rgb, float* y0_raw /* nullable: density pre-activation */,
                             const void* view_pe16, int feats_img16, void* stream);
int pag_decode_dc_bwd_tc_dyn(const float* feats, const float* lodw, const float* ray_d, const int64_t* ridx, int64_t M_max,
                             const int64_t* m_dev, int IN, const float* const* weights, float* const* grads, int hidden,
                             int view_dim, const float* g_sigma, const float* g_rgb, const float* grad_scale, float* g_feats,
                             float* g_dir, const void* view_pe16, float* workspace, int64_t workspace_bytes, int img16, void* stream);
/* feats_img16 / img16 != 0: `feats` (and `g_feats`, then still multiplied by *grad_scale) are fp16 operand images, see
 * pag_permuto_fwd_img16_dyn; IN % 8 == 0. */
/* view_pe16 (nullable): per-ray fp16 view embedding [R][32] from pag_view_pe16 -- the decoders copy it instead of evaluating
 * the positional embedding per sample.  workspace (nullable, device, 16-byte aligned): see pag_pan_composite_bwd_tc. */
int pag_view_pe16(const float* ray_d, int64_t R, void* pe16, void* stream);
int pag_decode_dc_bwd_workspace(int64_t M_max, int IN, int64_t* bytes /* host */);
int pag_decode_pan_fwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                          const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                          float inst_temperature, float* sem, float* inst, void* stream);
int pag_decode_pan_bwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                          const float* const* weights, float* const* grads, int hidden, int Cs, int Ci, int sem_softmax,
                          int inst_softmax, float inst_temperature, const float* sem, const float* inst,
                          const float* g_sem, const float* g_inst, const float* grad_scale, float* g_panop, void* stream);

/* exact-FP32 decoders for inference, register-tiled (csrc/decoder_tiled.cu; forward only).  pag_decode_dc_fwd_tiled has the
 * contract of pag_decode_dc_fwd (pc_nerf/panoptic_nef.py:274-300); pag_pan_composite_fwd_f32 has the contract of
 * pag_pan_composite_fwd_tc without the saved log-sum-exp (pc_nerf/panoptic_nef.py:302-363 fused with
 * tracers/panoptic_packed_rf_tracer.py:148-178): out_sem[N,Cs] / out_inst[N,Ci] zeroed by the caller, ridx i64[M] ascending. */
int pag_decode_dc_fwd_tiled(const float* feats, const float* lodw, const float* ray_d, int samples_per_ray, int64_t M, int IN,
                            const float* const* weights, int hidden, int view_dim, int want_rgb, float* sigma, float* rgb,
                            void* stream);
int pag_pan_composite_fwd_f32(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                              const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                              float inst_temperature, const float* w, const float* alpha, const int64_t* ridx,
                              float* out_sem, float* out_inst, void* stream);
/* labels of the semantic / instance heads for the point-map export (utils/render_map.py, which calls the nef on every map point and
 * takes the argmax on the host): same inputs, checks and error codes as pag_pan_composite_fwd_f32, but per sample the argmax class of
 * the head's logits (lowest index on ties) -> *_label i64[M], and that class's value of the channel the nef returns -> *_score f32[M]
 * (softmax ? 1 / sum_c exp((z_c - z_max) * s) : z_max * s, s = 1 / inst_temperature for the instance head when > 0, else 1).
 * No per-class output; nullable pairs skip their head (Cs / Ci = 0). */
int pag_pan_labels_fwd_f32(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN, const float* const* weights,
                           int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax, float inst_temperature, int64_t* sem_label,
                           float* sem_score, int64_t* inst_label, float* inst_score, void* stream);

/* panoptic heads fused with their compositing (training mode): out[ray] = alpha_ray * sum_s w_s * head(panop_s) with
 * alpha, w detached (tracers/panoptic_packed_rf_tracer.py:148-155,178-205); the [M,C] probabilities never reach HBM.
 * out_sem[N,Cs] / out_inst[N,Ci] must be zeroed by the caller (accumulated with red.add). ridx i64[M] ascending.
 * R = number of rays (rows of g_sem / g_inst). inst_lse f32[M] (nullable in forward): per-sample log2-domain log-sum-exp of the instance logits / T, written by
 * the forward and required by the backward when inst_softmax is set (the backward recomputes the logits with the same
 * tensor-core instructions and turns them into probabilities with one exp2 each). */
int pag_pan_composite_fwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                             const float* const* weights, int hidden, int Cs, int Ci, int sem_softmax, int inst_softmax,
                             float inst_temperature, const float* w, const float* alpha, const int64_t* ridx,
                             float* out_sem, float* out_inst, float* inst_lse, const int64_t* m_dev, int x_img16, void* stream);
int pag_pan_composite_bwd_tc(const float* feats, const float* dfeats, const float* lodw, int64_t M, int IN,
                             const float* const* weights, float* const* grads, int hidden, int Cs, int Ci,
                             int sem_softmax, int inst_softmax, float inst_temperature, const float* w, const float* alpha,
                             const int64_t* ridx, int64_t R, const float* g_sem, const float* g_inst, const float* inst_lse,
                             const float* grad_scale, float* g_panop, const int64_t* m_dev, float* workspace,
                             int64_t workspace_bytes, int x_img16, float* gw_sem, float* gw_inst, void* stream);
/* gw_sem / gw_inst f32[M] (nullable, softmax heads only): <p_s, g_ray> per sample = d out / d weight_s / alpha -- what a
 * tracer whose panoptic weights carry gradient (PanopticDDensityPackedRFTracer) needs to continue the chain rule. */
/* x_img16 != 0: feats / dfeats (and g_panop, then still multiplied by *grad_scale) are fp16 operand images, see
 * pag_permuto_fwd_img16_dyn; IN % 8 == 0. */
/* workspace (nullable, device): *bytes of pag_pan_composite_bwd_workspace(M, IN, Cs, Ci, &bytes), 16-byte aligned.  With it every CTA stores its
 * partial weight gradients privately and a second kernel sums them; without it they are accumulated with red.add. */
int pag_pan_composite_bwd_workspace(int64_t M, int IN, int Cs, int Ci, int64_t* bytes /* host */);

/* ---- packed compositing: tracers/panoptic_packed_rf_tracer.py:134-205 ------------------------------- */
/* offsets[r] = first packed index with ridx >= r (ridx ascending), offsets[R] = M. */
int pag_ray_offsets(const int64_t* ridx, int64_t M, int64_t R, int64_t* offsets, void* stream);
/* fused exponential integration + all channel reductions + alpha-on-top + background, dense [R,*] outputs. */
int pag_composite_fwd(const float* sigma, const float* deltas, const float* depths, const float* rgb,
                      const float* sem, int Cs, const float* inst, int Ci, const int64_t* offsets, int64_t R,
                      int bg_white, float* w, float* T, float* alpha, uint8_t* hit, float* rgb_out, float* rgbsum_out,
                      float* depth_out, float* sem_out, float* inst_out, void* stream);
int pag_composite_bwd(const float* sigma, const float* deltas, const float* depths, const float* rgb,
                      const int64_t* offsets, int64_t R, int bg_white, const float* w, const float* T,
                      const float* alpha, const float* rgbsum, const float* g_alpha, const float* g_rgb,
                      const float* g_depth, const float* g_sem, int Cs, const float* g_inst, int Ci, float* g_sigma,
                      float* g_rgb_s, float* g_sem_s, float* g_inst_s, void* stream);
/* Gradient tables on the wire as halfs for the multi-GPU all-reduce (SURVEY 8e; the reference reduces its grid gradients through
 * DistributedDataParallel-style fp32 all-reduce -- here the two 50 MB tables can travel as fp16 under a shared power-of-two scale):
 * out16[n] = half(x[n] * scale[0]);  x[n] = float(in16[n]) * mult / scale[0].  n % 4 == 0, 16-byte aligned. */
int pag_pack_f16(const float* x, int64_t n, const float* scale, void* out16, void* stream);
int pag_unpack_f16(const void* in16, int64_t n, const float* scale, float mult, float* x, void* stream);
/* debugging aid: cudaStreamCaptureStatus of `stream` (0 none, 1 active, 2 invalidated), negative on error. */
int pag_capture_status(void* stream);
/* power-of-two loss scale for the fp16 tensor-core backward (the GradScaler of pc_nerf/trainer.py:582, on the device).
 * scratch: two uint32, zero on entry, left zero by the kernel (one launch: the last block finalises and resets). */
int pag_grad_scale(const float* a, int64_t na, int wa, const float* b, int64_t nb, int wb, const int64_t* m_dev,
                   float target, uint32_t* scratch, float* out_scale, void* stream);
/* kaolin.render.spc.sum_reduce / exponential_integration (weights only), packs given by offsets[R+1]. */
int pag_sum_reduce_fwd(const float* x, int64_t C, const int64_t* offsets, int64_t R, float* out, void* stream);
int pag_sum_reduce_bwd(const float* g, int64_t C, const int64_t* offsets, int64_t R, float* gx, void* stream);
int pag_expint_fwd(const float* tau, const int64_t* offsets, int64_t R, float* w, float* T, void* stream);
int pag_expint_bwd(const float* gw, const float* w, const float* T, const int64_t* offsets, int64_t R, float* gtau,
                   void* stream);

/* The persistent tensor-core decoder kernels normally occupy every SM (one CTA per SM holding nearly all of its shared memory
 * and registers); reserve n SMs so that concurrently running kernels of other libraries -- the NCCL all-reduce that overlaps
 * the backward in multi-GPU training -- can make progress.  previous (host, nullable) receives the old value. */
int pag_set_reserved_sms(int n, int* previous /* host */);

/* ---- camera-pose transform of the base rays (bundle adjustment, SURVEY 8f rank 1) ----
 * Replaces BAPipeline.transform_rays (pc_nerf/ba_pipeline.py:85-92; kaolin Camera.extrinsics 'matrix_6dof_rotation' backend :44,
 * inv_transform_rays + renormalised directions :88-89) and its autograd backward into the 9 pose parameters per camera
 * (a1, a2: 6-D rotation, Gram-Schmidt rows of the view rotation; t: view translation).  Rays are grouped by camera, B per group;
 * cam_idx (nullable = identity) maps group -> parameter row; g_params is accumulated into. */
int pag_pose_transform_fwd(const float* params, const int64_t* cam_idx, const float* base_o, const float* base_d, int64_t C, int64_t B,
                           float* out_o, float* out_d, void* stream);
int pag_pose_transform_bwd(const float* params, const int64_t* cam_idx, const float* base_o, const float* base_d, const float* g_o,
                           const float* g_d, int64_t C, int64_t B, float* g_params, void* stream);

/* ---- gradient all-reduce over NVLink / NVSwitch peer memory (ray-sharded data parallelism, SURVEY 8e; no reference counterpart:
 * the reference is single-GPU, its DDP equivalent would all-reduce the grid tables of grids/permuto_grid.py:57-62 with NCCL) ----
 * In-place x <- mult * sum_ranks x on elements [offset, offset+n) of a SYMMETRIC float buffer: through the NVSwitch multicast
 * address (multimem.ld_reduce / multimem.st: the sum is formed inside the switch) or, when multicast is NULL, with explicit loads
 * from / stores to the `world` peer copies.  Rank r reduces the r-th slice.  The cross-rank ordering is pag_symm_barrier on the same
 * stream before and after: one CTA exchanging epochs through int32 flags [channels][16] kept at flag_offset of the same buffer. */
int pag_symm_barrier(float* const* peers, int64_t flag_offset, int* epoch, int rank, int world, int channel, void* stream);
int pag_allreduce_symm(float* multicast, float* const* peers, int rank, int world, int64_t offset, int64_t n, float mult, int max_ctas,
                       void* stream);

/* ---- instance loss with linear assignment, on the device (SURVEY 8f rank 3) ----
 * Replaces LinAssignmentThingsLoss (loss/lin_assignment_things.py:13-89, called at pc_nerf/trainer.py:484-520: Python loops over the
 * labels with a .cpu() each, scipy.optimize.linear_sum_assignment on the host, utils/outlier_rejection.py:8-52 id-range rejection):
 * sorted unique labels + per-ray ranks, label x id cost matrix, shortest-augmenting-path assignment (one CTA per image), virtual
 * labels, arg-max check and the NLL -- five launches, no host synchronisation.  Workspace shapes in csrc/loss.cu. */
int pag_inst_assignment_loss_fwd(const float* p, const int64_t* gt, const uint8_t* stuff, const float* points, int64_t B, int64_t R, int C,
                                 float frame_min_length, int max_num_inst_at_x, int id_margin, int32_t* labels, int32_t* n_labels, int32_t* rank,
                                 float* csum, float* cnt, float* xsum, int32_t* assign, int32_t* virt, int32_t* flag, float* loss, void* stream);
int pag_inst_assignment_loss_bwd(const float* p, const int32_t* virt, const int32_t* flag, const float* g_loss, int64_t B, int64_t R, int C,
                                 float* gp, void* stream);

/* Photometric + panoptic NLL loss of a training step (pc_nerf/trainer.py:442-480: L1 rgb, NLL of log(p + 1e-27) on the composited
 * semantic / instance probabilities) as one forward and one backward launch instead of ~20 torch kernels.
 * partials f32[>= 592], ticket u32[1] zero on entry (left zero), loss f32[1]; g_loss f32[1] on the device. */
int pag_panoptic_loss_fwd(const float* rgb, const float* sem, const float* inst, const float* t_rgb, const int64_t* t_sem, const int64_t* t_inst,
                          int64_t N, int Cs, int Ci, float w_rgb, float w_sem, float w_inst, float eps, float* partials, uint32_t* ticket,
                          float* loss, void* stream);
int pag_panoptic_loss_bwd(const float* rgb, const float* sem, const float* inst, const float* t_rgb, const int64_t* t_sem, const int64_t* t_inst,
                          int64_t N, int Cs, int Ci, float w_rgb, float w_sem, float w_inst, float eps, const float* g_loss, float* g_rgb,
                          float* g_sem, float* g_inst, void* stream);

/* ---- panoptic quality update on the device (validation metric) ----
 * Replaces the update of the vendored torchmetrics PanopticQuality (utils/metrics/panoptic_quality.py; called from evaluate_metrics,
 * pc_nerf/trainer.py:651-941: torch.unique per image, a device-to-host copy per segment colour, Python loops over segment pairs).
 * preds / target i64[B, P, 2] (category, instance), 16-byte aligned.  cat_ids i32[K] sorted ascending, cat_code i32[K] = continuous id
 * (| 0x100 for a thing) of each; K <= 256.  Accumulates iou_sum f64[K] and counts i64[3][K] (tp | fp | fn), and into errors i64[2] the
 * number of prediction pixels of an unknown category (unless allow_unknown_preds) and of thing pixels whose instance id lies outside
 * [0, 2^31).  Three launches (histogram, match, unmatched), no host synchronisation, geometry from (B, P) only; B <= 65535,
 * P <= 2^30.  workspace: pag_pq_workspace(B, P, &bytes) bytes = 44 * B * C with C the smallest power of two >= 2P (hash tables of
 * 2+ slots per pixel: never full, whatever the data), zero-filled by the caller ONCE -- every update leaves it zeroed again.
 * Layout in csrc/metrics.cu. */
int pag_pq_workspace(int64_t B, int64_t P, int64_t* bytes /* host */);
int pag_pq_update(const int64_t* preds, const int64_t* target, int64_t B, int64_t P, const int32_t* cat_ids, const int32_t* cat_code,
                  int K, int allow_unknown_preds, void* workspace, int64_t workspace_bytes, double* iou_sum, int64_t* counts,
                  int64_t* errors, void* stream);

/* ---- scene-level panoptic quality on the device: one segment per id across all frames of a sequence ----
 * Same rules as the per-image update above (evaluate_metrics, pc_nerf/trainer.py:651-941, scores each image on its own), applied to
 * ONE image made of every pixel of every update: tables that persist across updates.  Three open-addressing tables (prediction
 * segments, target segments, same-category pairs) of C = smallest power of two >= 2 * capacity slots, u64 areas; each admits at most
 * `capacity` keys and counts the pixels of refused keys; capacity in [1, 2^26].  workspace: pag_scene_pq_workspace(capacity, &bytes)
 * bytes = 64 * C + 128, zero-filled by the caller ONCE; it persists across updates (layout and counters in csrc/metrics.cu).
 * update: preds / target i64[N, 2] (all pixels of the call), 16-byte aligned, categories as pag_pq_update; errors i64[2] as there.
 *         One launch, no host synchronisation, geometry from N only.
 * stats:  accumulates iou_sum f64[K] and counts i64[3][K] (tp | fp | fn) of the scene so far into caller-zeroed arrays; two launches;
 *         the tables are left as found.
 * merge:  inserts another workspace of the same capacity (another rank's tables) into `workspace`; two launches. */
int pag_scene_pq_workspace(int64_t capacity, int64_t* bytes /* host */);
int pag_scene_pq_update(const int64_t* preds, const int64_t* target, int64_t N, const int32_t* cat_ids, const int32_t* cat_code, int K,
                        int allow_unknown_preds, void* workspace, int64_t capacity, int64_t workspace_bytes, int64_t* errors, void* stream);
int pag_scene_pq_stats(void* workspace, int64_t capacity, int64_t workspace_bytes, int K, double* iou_sum, int64_t* counts, void* stream);
int pag_scene_pq_merge(void* workspace, const void* other, int64_t capacity, int64_t workspace_bytes, void* stream);

/* ---- panoptic point-map export (utils/render_map.py: the nef evaluated on the occupied octree cells, labelled, exported) ----
 * pag_map_cell_points: cells i16[C,3] (leaf cells of `level`, e.g. the octree's level points) -> xyz f32[C*k^3, 3], k in [1, 8]:
 * sub-point s = (ix*k + iy)*k + iz of cell c at row c*k^3 + s, coordinate (2*(p*k + i) + 1) / (k << level) - 1 in fp32 (IEEE division).
 * pag_map_instance_stats: per-instance statistics of labelled points (xyz f32[P,3], rgb f32[P,3], semantic / instance i64[P]); a point
 * counts toward its instance only when bit `semantic` of thing_mask is set (Cs <= 32).  Accumulates count i64[Ci], sum_xyz / sum_rgb
 * f64[Ci,3] and votes i64[Ci,Cs] (zeroed by the caller) and bbox_min / bbox_max f32[Ci,3] (set to +inf / -inf by the caller); points
 * with a label outside [0, Cs) / [0, Ci) are skipped and counted in errors i64[1].  Label counts whose per-CTA slots fit in shared
 * memory accumulate there; larger ones accumulate in global memory, runs of equal labels reduced per warp first. */
int pag_map_cell_points(const int16_t* cells, int64_t C, int level, int k, float* xyz, void* stream);
int pag_map_instance_stats(const float* xyz, const float* rgb, const int64_t* semantic, const int64_t* instance, int64_t P, int Cs, int Ci,
                           uint32_t thing_mask, int64_t* count, double* sum_xyz, double* sum_rgb, int64_t* votes, float* bbox_min,
                           float* bbox_max, int64_t* errors, void* stream);
/* ---- connected components of a labelled map (no reference counterpart: objects of the exported map) ----
 * pag_map_components: xyz f32[P,3] on the lattice of (k, level), D = k << level (a coordinate is bit for bit
 * fl(fl((2j+1)/D) - 1), j in [0, D)), semantic / instance i64[P].  A point is active iff its labels are in [0, Cs) / [0, Ci) and bit
 * `semantic` of thing_mask is set; two active points are adjacent iff their lattice indices differ by a vector of {-1,0,1}^3 \ {0}
 * (connectivity 26) or by one unit step (connectivity 6) and their instance labels are equal.  Writes component i64[P]: the object
 * of each point, numbered 0..K-1 in the order of each object's smallest point index, -1 for inactive points and for objects of
 * fewer than min_points points.  info i64[4] (set by the call) = K | points off the lattice | points repeating the lattice index of
 * another point | points with a label out of range; component is meaningful only when the three counts are 0.  Seven launches,
 * no host synchronisation; P <= 2^30, Cs <= 32.  workspace: pag_map_components_workspace(P, &bytes) bytes = 12 C + 16 P +
 * 12 ceil(P / 1024) + 8, C = the smallest power of two >= 2P (hash table key u64 | point u32, never full), 8-byte aligned, no
 * initialisation needed.  Layout in csrc/mapping.cu.
 * pag_map_component_stats: pag_map_instance_stats per object (K labels, points with component -1 skipped, no thing mask, no error
 * count) plus object_instance i64[K], the instance label of each object. */
int pag_map_components_workspace(int64_t P, int64_t* bytes /* host */);
int pag_map_components(const float* xyz, const int64_t* semantic, const int64_t* instance, int64_t P, int level, int k, int Cs, int Ci,
                       uint32_t thing_mask, int connectivity, int64_t min_points, void* workspace, int64_t workspace_bytes,
                       int64_t* component, int64_t* info, void* stream);
int pag_map_component_stats(const float* xyz, const float* rgb, const int64_t* semantic, const int64_t* instance, const int64_t* component,
                            int64_t P, int Cs, int K, int64_t* count, double* sum_xyz, double* sum_rgb, int64_t* votes, float* bbox_min,
                            float* bbox_max, int64_t* object_instance, void* stream);
/* ---- lattice index of a map, and which map point / object a 3-D point or a rendered pixel lies on ----
 * pag_map_index: every point of xyz f32[P,3] (on the lattice of (k, level), D = k << level, as for pag_map_components; labels are not
 * read) into an open-addressing table: keys i64[C] (packed lattice index (jx << 42 | jy << 21 | jz) + 1, 0 = empty slot, linear
 * probing from fmix64(key) & (C-1)) and points i32[C] (the point of each filled slot).  C = pag_map_index_bytes(P, &bytes) / 12 = the
 * smallest power of two >= 2P; the call zero-fills keys itself.  info i64[4] (set by the call) = points inserted | points off the
 * lattice | points repeating the lattice index of another point | 0; the index is meaningful only when the two counts are 0.  One
 * launch, no host synchronisation; P <= 2^30.
 * pag_map_lookup_points: per query xyz f32[Q,3], per axis in float64 with explicitly rounded operations: t = ((x + 1) D) 0.5 - 0.5,
 * j0 = floor(t + 0.5).  point i64[Q] = the map point with lattice index j in [0, D)^3, |j - j0| <= radius per axis (radius in [0, 4])
 * and the smallest ((tx-jx)^2 + (ty-jy)^2) + (tz-jz)^2, then the smallest point index; -1 with no candidate, for a non-finite
 * coordinate and for t outside [-radius - 0.5, D - 0.5 + radius].  object i64[Q] (with component i64[P], nullable) = component[point],
 * -1 where point is -1.
 * pag_map_lookup_rays: the same for the surface point of each rendered ray: s = depth[i] / alpha[i] (fp32 IEEE), x = o + d s per axis
 * (fp32, separately rounded mul and add); origins / dirs f32[Q,3], depth / alpha f32[Q].  Rays with alpha < min_alpha (min_alpha in
 * (0, 1]) or a non-finite s get -1.
 * Lookups: one launch each, geometry from (Q, radius) only, no host synchronisation (graph capturable), results independent of
 * query order. */
int pag_map_index_bytes(int64_t P, int64_t* bytes /* host */);
int pag_map_index(const float* xyz, int64_t P, int level, int k, int64_t* keys, int32_t* points, int64_t C, int64_t* info, void* stream);
int pag_map_lookup_points(const int64_t* keys, const int32_t* points, int64_t C, int level, int k, const float* xyz, int64_t Q,
                          int radius, const int64_t* component, int64_t* point, int64_t* object, void* stream);
int pag_map_lookup_rays(const int64_t* keys, const int32_t* points, int64_t C, int level, int k, const float* origins,
                        const float* dirs, const float* depth, const float* alpha, float min_alpha, int64_t Q, int radius,
                        const int64_t* component, int64_t* point, int64_t* object, void* stream);
/* ---- projection of a map into camera views: which map point, at what depth, and which object each pixel sees ----
 * pag_map_project: xyz f32[P,3] (P <= 2^30), view f32[B,4,4] world-to-camera (rows 0..2 read), intrinsics f32[B,4] = (fx, fy, cx, cy)
 * in pixels; the camera looks down -z, pixel (row r, column c) has the camera-space direction ((c + 0.5 - cx) / fx,
 * (r + 0.5 - cy) / fy, -1).  In fp32, every operation separately rounded: p_q = ((V[q,0] x + V[q,1] y) + V[q,2] z) + V[q,3],
 * z = -p_2, u = fx (p_0 / z) + cx, v = fy (p_1 / z) + cy, su = min((fx h) / z, max_radius), sv = min((fy h) / z, max_radius) (h =
 * the lattice half-size 1 / D, passed by the caller).  A point is splatted iff z > near, u and v are finite and su, sv >= 0 (false
 * for NaN); it covers columns floor(u - su) .. floor(u + su) and rows floor(v - sv) .. floor(v + sv), clipped to the image.  Each
 * pixel keeps the covering point of smallest z, then of smallest index: point i64[B,H,W] (-1 if none), depth f32[B,H,W] (+inf if
 * none), object i64[B,H,W] = component[point] (object nullable; component i64[P] required with object when P > 0; -1 where point is -1).  zbuf u64[B*H*W]:
 * caller-owned depth buffer, filled by the call.  B <= 65535, H and W in [1, 16384], max_radius in [0, 32], near > 0.  A fill and
 * two launches, geometry from (P, B, H, W) only, no host synchronisation (graph capturable), deterministic. */
int pag_map_project(const float* xyz, int64_t P, const float* view, const float* intrinsics, int B, int H, int W, float h, float near,
                    int max_radius, int64_t* zbuf, const int64_t* component, int64_t* point, float* depth, int64_t* object,
                    void* stream);
/* ---- per-object visibility of a map in camera views: visible area, unoccluded silhouette and visible box per (view, object) ----
 * Cameras, footprints and the front point of each pixel exactly as pag_map_project; component i64[P] (required when P > 0), K
 * objects (K <= 2^30), N = B K pairs n = b K + o.  Points with component -1 occlude but own no pair; components outside [-1, K) are
 * skipped and counted.  Two calls, with one host read between them:
 * pag_map_visibility: fills the depth buffer zbuf u64[B*H*W] (not read, may be null, when P = 0) and splats the map (pag_map_project's kernel), then writes
 * visible i64[N] (pixels whose front point has object o), bbox i32[N,4] = (col_min, row_min, col_max, row_max) of those pixels
 * (-1s where visible is 0), box i32[N,4] (the union of the footprints of the pair's points, clipped to the image; (2^31-1,
 * 2^31-1, -1, -1) when empty), words i32[N] (the size of the pair's silhouette bitmap: box rows times the 32-bit words of the
 * image its columns touch) and offset i64[N+2]: exclusive scan of words (offset[N] = total words) and offset[N+1] = points with a
 * component outside [-1, K).  Sets silhouette i64[N] to 0.  Five launches and a scan, no host synchronisation.
 * pag_map_visibility_silhouette: silhouette[n] = pixels covered by a footprint of the pair's points, at any depth: the pairs'
 * bitmaps are OR-splatted in rounds into bits i32[bits_words] and popcounted.  A round takes the pairs whose offset lies in
 * [lo, lo + step), step = total_words when it fits bits_words, else bits_words - H ceil(W / 32) (the largest bitmap), which must be
 * > 0.  Two launches and a fill per round. */
int pag_map_visibility(const float* xyz, int64_t P, const float* view, const float* intrinsics, int B, int H, int W, float h, float near,
                       int max_radius, const int64_t* component, int K, int64_t* zbuf, int32_t* box, int32_t* words, int64_t* offset,
                       int64_t* visible, int64_t* silhouette, int32_t* bbox, void* stream);
int pag_map_visibility_silhouette(const float* xyz, int64_t P, const float* view, const float* intrinsics, int B, int H, int W, float h,
                                  float near, int max_radius, const int64_t* component, int K, const int32_t* box, const int32_t* words,
                                  const int64_t* offset, int64_t total_words, int32_t* bits, int64_t bits_words, int64_t* silhouette,
                                  void* stream);

/* ---- fused multi-tensor Adam (BASELINE config 4: "+ Adam"; SURVEY 8e "a single fused unscale + Adam kernel") ----
 * Replaces torch.optim.Adam.step() as the reference's trainer runs it (pc_nerf/trainer.py:229-300 parameter groups, :590 step;
 * configs/bup20/best.yaml:114 optimizer_type adam): n_tensors <= 48 fp32 tensors in one launch, host arrays of device pointers,
 * step count and optional inverse loss scale in device memory (graph capturable).  amsgrad off, L2 weight decay. */
int pag_adam_step(float* const* p, const float* const* g, float* const* m, float* const* v, const int64_t* numel, const float* lr,
                  const float* weight_decay, int n_tensors, float beta1, float beta2, float eps, int* step, const float* inv_scale,
                  void* stream);

/* ---- L2 persisting window for a grid table (north_star: "per-level tables staged in shared memory or L2-persisting windows";
 * the tables of grids/permuto_grid.py:57-62 are 50 MB each, the B200 L2 126 MB) ----
 * Kernels launched on `stream` afterwards treat [base, base+bytes) as persisting with probability hit_ratio, everything else as
 * streaming; bytes = 0 clears.  pag_l2_limits: the device's maximum persisting carve-out and window size. */
int pag_set_l2_window(const void* base, int64_t bytes, float hit_ratio, void* stream);
int pag_l2_limits(int64_t* max_persisting /* host */, int64_t* max_window /* host */);

/* ---- achievable-gather-bandwidth probe (bench.py: denominator of the encoder's roofline fraction, SURVEY 8d) ----
 * threads x loads_per_thread (multiple of 16, 16 in flight per thread) uniformly random 8-byte loads from table[entries] float2; sink f32[threads]. */
int pag_gather_probe(const float* table, int64_t entries, int64_t threads, int loads_per_thread, float* sink, void* stream);
/* L2 read bandwidth: all CTAs together stream buf[bytes] (multiple of 16; <= the 126 MB L2 to stay resident) iters times with
 * coalesced 16-byte loads; sink f32[148 * 8 * 256].  Peak of the "l2" roofline of the gather-bound encoders (SURVEY 8d). */
int pag_l2_stream_probe(const void* buf, int64_t bytes, int iters, float* sink, void* stream);

/* ---- tcgen05 building-block probe (tests only): one 128-row tile through the tensor-core operand images ---- */
int pag_tc_gemm_test(int mode, const float* A, const float* B, float* D, int N, int K, int FA, int reps, void* stream);
int pag_tc_gemm_test16(int mode, const float* A, const float* B, float* D, int N, int K, int FA, int reps, void* stream);
/* timing probe: mode 0/1/2 = forward / backward-data / backward-weight operand roles; cycles i64[2] = {total, issue} */
int pag_tc_mma_bench(int mode, int N, int K, int chains, int reps, int64_t* cycles, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PAGNERF_B200_H */
