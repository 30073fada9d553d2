/* libhnr -- C ABI of the B200-native per-ray sample pipeline (drop-in boundary, SURVEY.md 8b).
 *
 * The reference (CVMI-Lab/HybridNeuralRendering) has no FFI layer: its seam is the Python module
 * API (lighting_fast_querier, NeuralPoints, PointAggregator, ray_march, blur_update_output).  The
 * host package `hybridneuralrendering_b200` mirrors that API and calls the entry points below
 * through ctypes.  Each entry point cites the reference code it replaces (paths relative to the
 * reference repository root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to caller-owned memory (torch-allocated); the library
 *     allocates nothing and keeps no pointers between calls;  fp32 / int32 / uint8 only;
 *   - tensors are dense row-major; sizes are int64_t; `stream` is a cudaStream_t passed as void*;
 *   - return 0 on success, negative on error (-1 CUDA error, -2 bad argument, -3 unsupported);
 *     hnr_last_error() returns the message (thread-local);  functions never throw;
 *   - kernels are compiled for sm_100a only; there is no CPU fallback.
 */
#ifndef HNR_H
#define HNR_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

int hnr_abi_version(void);
const char* hnr_last_error(void);
int hnr_device_arch(void); /* major*10+minor of the current device (100 on B200) */

/* ---------------------------------------------------------------------------------------------
 * Voxel-grid neural-point query: models/neural_points/query_point_indices_worldcoords.py
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    float origin[3];     /* ranges[:3] after padding         (get_hyperparameters :46-77) */
    float cell[3];       /* vsize * vscale                                                 */
    int32_t dims[3];     /* scaled_vdim                                                    */
    float radius2;       /* (radius_limit_scale * max(vsize.x, vsize.y))^2 ; 0 = unlimited */
    int64_t n_cells;     /* dims[0]*dims[1]*dims[2]                                        */
    int32_t P;           /* max stored points consulted per voxel (opt.P)                  */
    int32_t layers;      /* (kernel_size[0]+1)/2 shells walked by the neighbour search     */
    int32_t qhalf_lo[3]; /* occupancy dilation reach below: query_size/2                   */
    int32_t qhalf_hi[3]; /* and above: (query_size+1)/2 - 1                                */
} hnr_grid_t;

int64_t hnr_scan_scratch_elems(int64_t n);
int hnr_exclusive_scan_i32(const int32_t* in, int32_t* out /* n+1 */, int64_t n, int32_t* scratch, void* stream);

/* Occupancy-grid build; replaces build_occ_vox + claim_occ/map_coor2occ/fill_occ2pnts (:237-381, :540-602).
 * Called once per point-set change (the reference rebuilds per forward, :616).
 * skip_cell: -1 none, -2 voxel of the first in-grid point (stand-in for the reference's
 * "occupied slot 0 stores no points" quirk, :366), >=0 explicit linear voxel id.
 * info int32[8]: [0] occupied voxels [1] max points/voxel [2] skip voxel [3] points dropped with it
 *                [4] first in-grid point id [5] points stored. */
int hnr_grid_build(const float* xyz, int64_t N, const hnr_grid_t* g, int32_t skip_cell, int32_t* cell_of_pt /* N */,
                   int32_t* counts /* n_cells */, int32_t* cell_start /* n_cells+1 */, int32_t* tmp_idx /* N */,
                   void* pts_sorted /* float4[N] */, uint32_t* occ_bits /* ceil(n_cells/32) */, int32_t* scan_scratch,
                   int32_t* info /* 8 */, void* stream);

/* One query over R rays; replaces mask_raypos, get_shadingloc, query_neigh_along_ray_layered and
 * the torch compaction between them (:384-522, :605-711) plus w2pers / ray-dir expansion (:80-103).
 * ts = the D candidate parameters of near_far_linear_ray_generation
 * (models/rendering/diff_ray_marching.py:349-392), shared by all rays (ts_stride 0) or per ray
 * (ts_stride D).  Outputs are sized for R rays; counts_out = {R'' kept rays, Nv valid samples}. */
int hnr_query(const float* campos, const float* camrot /* c2w rotation 3x3 */, const float* raydir /* R,3 */, const float* ts,
              int64_t ts_stride, int64_t R, int64_t D, int64_t SR, int64_t K, const hnr_grid_t* g, const int32_t* cell_start,
              const void* pts_sorted, const uint32_t* occ_bits, float* sample_loc_full /* R,SR,3 zeroed */,
              int32_t* pidx_full /* R,SR,K */, int32_t* nsamp /* R */, int32_t* nvalid /* R */, int32_t* keep /* R */,
              int32_t* ray_off /* R+1 */, int32_t* val_off /* R+1 */, int32_t* scan_scratch, int32_t* out_pidx /* R,SR,K */,
              float* out_loc_pers /* R,SR,3 */, float* out_loc_w, float* out_dirs, int8_t* ray_mask /* R */, int32_t* ray_ids /* R */,
              int32_t* vlist /* R*SR */, int32_t* counts_out /* 2 */, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Aggregation: models/aggregators/point_aggregators.py, models/neural_points/neural_points.py
 * ------------------------------------------------------------------------------------------- */
/* camera block `cam`: 21 floats in DEVICE memory = campos[3], camrot[9] (c2w rotation, row-major),
 * rt[9] (Rw2c^T row-major, identity unless normview).  Device-resident so no host sync is needed. */

/* inverse-distance weights + confidence clamp for ALL S samples; PointAggregator.linear (:825-833),
 * normalisation (:1500-1501), gradiant_clamp (:1422-1424).  mask may be NULL (then pidx<0 = masked). */
int hnr_nbr_weights(const float* xyz, const float* conf, const int32_t* pidx, const uint8_t* mask, const float* loc_w, int64_t S,
                    int64_t K, float* weight, float* confc, uint8_t* valid, void* stream);
/* per-neighbour MLP input rows for the Nv valid samples: gather (neural_points.py:708-720), dists
 * (:1472-1480), positional encodings (helpers/networks.py:175-189), block3 extras (:957-971). */
int hnr_nbr_features(const float* xyz, const float* xyz_pers /* may be NULL */, const float* emb, const float* color,
                     const float* dir, const int32_t* pidx, const int32_t* vlist, const float* loc_w, const float* loc_pers,
                     const float* raydirs, const float* cam, int64_t Nv, int64_t K, int64_t emb_dim, float* X0 /* Nv*K,284 */,
                     float* E /* Nv*K,7 */, void* stream);
int hnr_nbr_features_bwd(const float* dX0, const float* dE, const float* emb, const int32_t* pidx, const uint8_t* mask,
                         const int32_t* vlist, const float* raydirs, const float* cam, int64_t Nv, int64_t K, float* d_emb,
                         float* d_color, float* d_dir, void* stream);
/* density head + weighted K-sum + view-dir encoding (:1002-1036) */
int hnr_alpha_ksum_fwd(const float* H, const float* weight, const float* confc, const int32_t* vlist, const float* w_alpha,
                       const float* b_alpha, const float* raydirs, const float* cam, int64_t Nv, int64_t K, int64_t hidden,
                       float* sigma, float* X5 /* Nv,280 */, float* alpha_raw /* Nv*K */, void* stream);
int hnr_alpha_ksum_bwd(const float* H, const float* weight, const float* confc, const int32_t* vlist, const float* w_alpha,
                       const float* alpha_raw, const float* d_sigma, const float* dX5, int64_t Nv, int64_t K, int64_t hidden,
                       float* dH, float* d_wc, float* d_walpha, float* d_balpha, void* stream);
int hnr_conf_bwd(const float* d_wc, const float* weight, const int32_t* vlist, const int32_t* pidx, const float* d_confc, int64_t Nv,
                 int64_t S, int64_t K, float* d_conf, void* stream);
/* w2iproject + delta view dirs (models/neural_points_volumetric_model.py:248-255, :287-310) */
int hnr_project_views(const float* loc_w, const float* w2c /* V,4,4 */, const float* Kmat /* 3,3 */, const float* campos,
                      const float* campos_n /* V,3 */, int64_t V, int64_t S, float* xy /* V,S,2 */, float* delta /* V,S,3 */,
                      void* stream);
/* pyramid lookup == F.interpolate(bilinear) to full res, zero pixel (0,0), truncated nearest pixel
 * (:1064-1096, :1193); levels are NHWC: (V,H,W,3),(V,h1,w1,6),(V,h2,w2,12),(V,h3,w3,24) */
int hnr_image_gather_fwd(const float* const* levels, const int64_t* level_hw /* 8 */, const float* xy, const int32_t* vlist,
                         int64_t V, int64_t S, int64_t Nv, float* aux /* V,Nv,aux_ld */, float* ok /* V,Nv */,
                         int64_t aux_ld /* 45, or 48 = 16-byte aligned rows */, const float* delta /* V,S,3 or NULL: copied into columns
                         45..47 of a 48-wide row (the blend-weight net's input [aux | dview] in one aligned block) */, void* stream);
int hnr_image_gather_bwd(float* const* level_grads, const int64_t* level_hw, const float* xy, const int32_t* vlist, const float* d_aux,
                         int64_t V, int64_t S, int64_t Nv, void* stream);
/* same with a row stride for d_aux (48 = the aligned training rows [aux 45 | dview 3]; columns >= 45 are ignored) */
int hnr_image_gather_bwd_ld(float* const* level_grads, const int64_t* level_hw, const float* xy, const int32_t* vlist, const float* d_aux,
                            int64_t d_ld, int64_t V, int64_t S, int64_t Nv, void* stream);
/* multi-view blend (:1199-1217) + train-time drop (:1222-1237) */
int hnr_blend_fwd(const float* aux, const float* sig, const float* ok, const uint8_t* keep, int64_t V, int64_t Nv, int64_t aux_ld,
                  float* merged, int64_t merged_ld /* 45, or 48 with zero padding */, void* stream);
int hnr_blend_bwd(const float* aux, const float* sig, const float* ok, const uint8_t* keep, const float* d_merged, int64_t V,
                  int64_t Nv, float* d_aux, float* d_sig, void* stream);
/* same with row strides for aux and d_aux (45..64; padding columns of d_aux are zero-filled) */
int hnr_blend_bwd_ld(const float* aux, int64_t aux_ld, const float* sig, const float* ok, const uint8_t* keep, const float* d_merged,
                     int64_t V, int64_t Nv, float* d_aux, int64_t d_aux_ld, float* d_sig, void* stream);

/* dense layers: y = act(concat(A0,A1,A2) W^T + b [+res]); W (N,K) row-major as nn.Linear
 * (layers built at point_aggregators.py:484-683).  act: 0 none, 1 LeakyReLU(0.01), 2 sigmoid,
 * 3 sigmoid*1.002-0.001 (raw2out_color :478-482).  a_mod[i] > 0: source i has a_mod[i] rows, shared
 * by row blocks (the per-sample feature reused for each of the V views). */
int hnr_linear_fwd(const float* const* a_ptr, const int64_t* a_ld, const int64_t* a_k, const int64_t* a_mod, const float* W,
                   const float* bias, const float* res, int64_t ldres, float* Y, int64_t ldy, int64_t M, int64_t N, int64_t K, int act,
                   void* stream);
int hnr_linear_bwd_data(const float* dY, int64_t lddy, const float* Y, int64_t ldy, const float* W, float* const* da_ptr,
                        const int64_t* da_ld, const int64_t* a_k, int64_t M, int64_t N, int64_t K, int act, void* stream);
int hnr_linear_bwd_weight(const float* dY, int64_t lddy, const float* Y, int64_t ldy, const float* const* a_ptr, const int64_t* a_ld,
                          const int64_t* a_k, const int64_t* a_mod, float* dW, float* db, int64_t M, int64_t N, int64_t K, int act,
                          void* stream);
/* backward of a ONE-output layer h = act(y.w + b) in one pass (csrc/linear_simt.cu; the sigmoid head of the blend-weight net,
 * point_aggregators.py:1199-1217): dY[m,:] = dH[m] act'(h[m]) w, dW (K) += sum_m s_m y[m,:], db (1) += sum_m s_m.  K = 64 or 128. */
int hnr_linear_head_bwd(const float* dH, const float* Hout, int act, const float* w, const float* Y, int64_t ldy, int64_t M, int64_t K,
                        float* dY, int64_t lddy, float* dW, float* db, void* stream);
/* data gradient of a narrow column slice [k0, k0+kn), kn <= 8, of a layer with N = 128 or 256 outputs: dA (M, kn) =
 * (dY * act'(Y)) (M,N) . W[:, k0:k0+kn]; W (N, ldw) row-major.  HBM-bound (one read of dY and Y); dY / Y rows 16-byte aligned. */
int hnr_linear_bwd_data_narrow(const float* dY, int64_t lddy, const float* Y, int64_t ldy, int act, const float* W, int64_t ldw,
                               int64_t k0, int64_t kn, float* dA, int64_t ldda, int64_t M, int64_t N, void* stream);

/* one dense layer on tcgen05 tensor cores (3xTF32, fp32 accuracy): same semantics as hnr_linear_fwd; wpack is
 * the host-packed TF32 hi/lo image of W zero-padded to (Npad % 16 == 0 <= 256, Kp % 8 == 0) (csrc/linear_tc.cu) */
int64_t hnr_linear_tc_packed_bytes(int64_t Npad, int64_t Kp);
int hnr_linear_tc_fwd(const float* const* a_ptr, const int64_t* a_ld, const int64_t* a_k, const int64_t* a_mod, const void* wpack,
                      int64_t Npad, int64_t Kp, const float* bias, const float* res, int64_t ldres, float* Y /* may be NULL */,
                      int64_t ldy, int64_t M, int64_t N, int64_t K, int act, const float* head_w /* N or NULL */,
                      const float* head_b, int head_act, float* out_head /* M */, void* stream);

/* Tensor-core backward of a dense layer (training path), 3xTF32 -- autograd of the nn.Linear layers of
 * models/aggregators/point_aggregators.py:484-754 as called at :921-1026 (per-neighbour) and :1028-1037, :1188-1217, :1285-1334:
 *   hnr_linear_tc_bwd_data:   dX (M, Kout <= 256 columns per call) = (dY * act'(Y)) (M,N) . W (N, K-slice); wpackT = image of
 *                             the transposed weight slice (csrc/linear_tc.cu; replaces hnr_linear_bwd_data)
 *   hnr_linear_tc_bwd_weight: dW (N,K) += (dY * act'(Y))^T . concat(X), db += column sums; reduction over the M rows with the
 *                             accumulator resident in TMEM (csrc/wgrad_tc.cu; replaces hnr_linear_bwd_weight) */
int hnr_linear_tc_bwd_data(const float* dY, int64_t lddy, const float* Y, int64_t ldy, int act, const void* wpackT, int64_t Kpad,
                           int64_t Np, float* dX, int64_t lddx, int64_t M, int64_t N, int64_t Kout, void* stream);
int hnr_linear_tc_bwd_weight(const float* dY, int64_t lddy, const float* Y, int64_t ldy, const float* const* a_ptr, const int64_t* a_ld,
                             const int64_t* a_k, const int64_t* a_mod, float* dW, float* db, int64_t M, int64_t N, int64_t K, int act,
                             void* stream);

/* Fused per-neighbour stage (gather, encodings, block1, block3, density head, weighted K-sum; SURVEY 8a rows G1 + A1-A3;
 * reference: models/neural_points/neural_points.py:708-720, models/aggregators/point_aggregators.py:921-1026): 3xFP16 split on tcgen05.mma.kind::f16 (twice the TF32 rate, fp32
 * accuracy: 22 mantissa bits), activations kept in shared memory directly in the UMMA operand layout, two TMEM
 * accumulators so that epilogue l overlaps the MMAs of layer l+1 (csrc/nbr_mlp_f16.cu).  wpack: 67 chunk images in
 * consumption order; bias (4,256) with rows 0..2 pre-multiplied by the next layer's input scale; mul[4]: accumulator ->
 * pre-activation factors; scale0/scale2: input scales of the generated features / the block3 extras (all built by
 * hybridneuralrendering_b200/mlp_tc.py: pack_mlp_f16).  dbg: optional (4, Nv*8, 256) per-layer activations (saved by the
 * training forward for the backward pass, and the taps of the parity test), else NULL. */
int64_t hnr_nbr_mlp_f16_packed_bytes(void);
int hnr_nbr_mlp_f16_forward(const float* xyz, const float* xyz_pers, const float* emb, const float* color, const float* dir,
                            const int32_t* pidx, const int32_t* vlist, const float* loc_w, const float* loc_pers,
                            const float* raydirs, const float* cam, const float* weight, const float* confc, const void* wpack,
                            const float* bias, const float* walpha, const float* balpha, const float* mul /* host, 4 */,
                            float scale0, float scale2, float inv_act, int64_t Nv, int64_t K, float* sigma /* Nv */,
                            float* X5 /* Nv,280 */, float* dbg, float* araw /* Nv*8, with dbg */,
                            int32_t* status /* optional device word: |= 1 when an activation saturated fp16 */, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused TRAINING path of the per-neighbour MLP (round 2).  The reference's backward is autograd over
 * models/aggregators/point_aggregators.py:921-972, :1002-1026; here three kernels replace the 4 x (data gradient + weight
 * gradient) layer launches.  Everything that crosses HBM between them is a "split image" (csrc/img_common.cuh): bf16 hi | lo
 * planes per 32-row slab, which is simultaneously the canonical MN-major UMMA operand of the weight gradient and a
 * thread-per-row coalesced format.  All images have ceil(Nv*8 / 128) * 128 rows.
 * ------------------------------------------------------------------------------------------- */
/* forward that saves its operands: x0img 288 columns (layer-0 input, kernel column order = mlp_tc.layer1_column_order_f16),
 * eimg 16 columns (block3 extras), h0..h3img 256 columns (layer outputs), araw (Nv*8) density pre-activations. */
/* hnr_nbr_mlp_f16_forward with the per-point layer-0 partial (inference): 224 of block1[0]'s 284 inputs -- the embedding and its
 * positional encoding (point_aggregators.py:931-939) -- depend on the POINT only, and a point is the neighbour of many samples.
 * pp (N_points, 256) fp32 = block1[0].weight[:, :224] . [emb | PE(emb)] per point (unscaled), computed once per (weights, point
 * set); the kernel generates only the 4 distance-encoding chunks of layer 0 and adds pp[point] in the layer-0 epilogue.  Same
 * wpack / bias / mul as hnr_nbr_mlp_f16_forward; the embedding table is not read. */
int hnr_nbr_mlp_f16_forward_pp(const float* xyz, const float* xyz_pers, const float* pp, const float* color, const float* dir,
                               const int32_t* pidx, const int32_t* vlist, const float* loc_w, const float* loc_pers, const float* raydirs,
                               const float* cam, const float* weight, const float* confc, const void* wpack, const float* bias,
                               const float* walpha, const float* balpha, const float* mul /* host, 4 */, float scale0, float scale2,
                               float inv_act, int64_t Nv, int64_t K, float* sigma, float* X5, int32_t* status, void* stream);
int hnr_nbr_mlp_f16_forward_train(const float* xyz, const float* xyz_pers, const float* emb, const float* color, const float* dir,
                                  const int32_t* pidx, const int32_t* vlist, const float* loc_w, const float* loc_pers,
                                  const float* raydirs, const float* cam, const float* weight, const float* confc, const void* wpack,
                                  const float* bias, const float* walpha, const float* balpha, const float* mul /* host, 4 */,
                                  float scale0, float scale2, float inv_act, int64_t Nv, int64_t K, float* sigma, float* X5,
                                  void* x0img, void* eimg, void* h0img, void* h1img, void* h2img, void* h3img, float* araw,
                                  int32_t* status, void* stream);
/* backward of the density head + weighted K-sum (:1002-1036) from / to images: reads h3img, writes dz3img = dH * act'(H_3);
 * d_confc (S,K; pre-zeroed) or NULL: the gradient of conf_coefficient, d_wc * weight, written at the valid samples' rows */
int hnr_alpha_ksum_bwd_img(const void* h3img, const float* weight, const float* confc, const int32_t* vlist, const float* w_alpha,
                           const float* alpha_raw, const float* d_sigma, const float* dX5, int64_t Nv, int64_t K, void* dz3img,
                           float* d_wc, float* d_walpha, float* d_balpha, float* d_confc, void* stream);
/* fused data-gradient chain dZ_3 -> dZ_2 -> dZ_1 -> dZ_0 -> dX0 (csrc/nbr_bwd_f16.cu; 3 x bf16 split on tcgen05, gradient
 * tile resident in shared memory / TMEM across the four layers).  wpackT: hnr_nbr_bwd_f16_packed_bytes() bytes built by
 * mlp_tc.pack_mlp_bwd.  dX0 (rows, ldx): the first nx0 input-gradient columns of layer 0. */
int64_t hnr_nbr_bwd_f16_packed_bytes(void);
int hnr_nbr_bwd_f16(const void* dz3, const void* h2, const void* h1, const void* h0, void* dz2, void* dz1, void* dz0, float* dX0,
                    int64_t ldx, int64_t nx0, const void* wpackT, int64_t rows, void* stream);
/* dE (rows,7) = dZ (image) . W[:, k0:k0+7]: gradient of block3's extra inputs */
int hnr_dz_extras_bwd(const void* dz, const float* W, int64_t ldw, int64_t k0, int64_t rows, float* dE, void* stream);
/* weight + bias gradients of up to 4 layers in ONE launch, operands bulk-copied from the images as MN-major UMMA tiles
 * (csrc/wgrad_img.cu).  Job i accumulates dZ_i^T [X_i | E_i] straight into the parameter-shaped dw[i] (n_rows, k_cols) through an
 * optional column map (kernel input-column order -> reference column, < 0 = padding) and the column sums of dZ_i into db[i];
 * ca[i] = dZ image width (the layer's padded output width, <= 256), rows_pad[i] = image rows. */
int hnr_wgrad_img_jobs(int njob, const void* const* a, const int64_t* ca, const void* const* b, const void* const* e, const int64_t* cb,
                       const int64_t* ce, float* const* dw, float* const* db, const int32_t* const* colmap, const int64_t* n_rows,
                       const int64_t* k_cols, const int64_t* rows_pad, void* stream);
/* Fused training path of the per-sample chains (color_feature_branch, aux_merge_weight_block, color_mixup_block;
 * point_aggregators.py:1028-1037, :1188-1217, :1285-1334).  hnr_chain_f16_forward_train = hnr_chain_f16_forward that also saves
 * the concatenated input (x0img, Kp[0] columns) and the inner outputs (himg[l], Np[l] columns) as split images;
 * hnr_chain_bwd_f16 (csrc/chain_bwd_f16.cu) = fused data-gradient chain: dZ_top = dY * act'(Ytop), dZ_{l-1} = (dZ_l W_l) *
 * act'(H_{l-1}), dX = dZ_0 W_0[:, :NX]; every dZ_l is also written as a split image for hnr_wgrad_img_jobs. */
int hnr_chain_f16_forward_train(const float* const* src, const int64_t* src_ld, const int64_t* src_k, const int64_t* src_mod,
                                float in_scale, int nlayer, const int64_t* Kp, const int64_t* N, const int64_t* Np, const int* act,
                                const void* wpack, const int64_t* w_off, const float* bias, const float* mul, const float* inv_next,
                                float* const* Y, const int64_t* ldy, const float* res, int64_t ldres, const float* head_w,
                                const float* head_b, int head_act, float* head_out, int64_t M, int32_t* status, void* x0img,
                                void* const* himg, void* stream);
/* hnr_chain_f16_forward(_train) with an addend of layer 0's pre-activation: y_0 = act(x_0 W_0^T + b_0 + add0[m % add0_mod, :]).  Used for
 * aux_merge_weight_block (:1199-1217): its first layer's input [g | aux_v | dview_v] shares g between the V views of a sample, so
 * W_0g g is computed once per sample (a one-layer chain) and this chain reads only the 48 view-dependent columns.  x0img / himg NULL =
 * inference.  hnr_img_sum_views: the addend's gradient, sum over the V views of the dZ_0 image rows (out (Nv, ldo) fp32). */
int hnr_chain_f16_forward_add0(const float* const* src, const int64_t* src_ld, const int64_t* src_k, const int64_t* src_mod, float in_scale,
                               int nlayer, const int64_t* Kp, const int64_t* N, const int64_t* Np, const int* act, const void* wpack,
                               const int64_t* w_off, const float* bias, const float* mul, const float* inv_next, float* const* Y,
                               const int64_t* ldy, const float* res, int64_t ldres, const float* head_w, const float* head_b, int head_act,
                               float* head_out, int64_t M, int32_t* status, void* x0img, void* const* himg, const float* add0,
                               int64_t add0_ld, int64_t add0_mod, float add0_scale, void* stream);
int hnr_img_sum_views(const void* img, int64_t C, int64_t Nv, int64_t V, float* out, int64_t ldo, void* stream);
int hnr_chain_bwd_f16(int nlayer, const int64_t* Np, const int64_t* N, int64_t NX, int act_top, const float* dY, int64_t lddy,
                      const float* Ytop, int64_t ldyt, const void* const* gimg, void* const* dzimg, const void* wpackT,
                      const int64_t* w_off, float* dX, int64_t ldx, int64_t M, void* stream);
/* Training loss (csrc/loss.cu): masked MSE (+1e-6) x frame_weight + zero-one regulariser on conf_coefficient
 * (models/base_rendering_model.py:1114-1118, :1205-1206, :1229-1240); value (written to loss) and both gradients.  The per-block
 * partial sums go through `partials` (HNR_TRAIN_LOSS_PARTIALS doubles of scratch) and are added in a fixed order: the value is the
 * same in every run. */
#define HNR_TRAIN_LOSS_PARTIALS 512
int hnr_train_loss(const float* color, const float* gt, const int32_t* ray_ids, int64_t n_rays, const float* confc, int64_t n_conf,
                   float frame_weight, float zero_one_weight, float* loss, double* partials, float* d_color, float* d_confc, void* stream);
/* Feature pyramid of the image branch (csrc/pyramid.cu): the six 3x3 convolutions + LeakyReLU of aux_block_s1/s2/s3
 * (models/aggregators/point_aggregators.py:598-630, :1047-1063), exact fp32, NHWC, forward and backward.  w/b: six torch-layout
 * (Cout,Cin,3,3) / (Cout) tensors; act: the six activated outputs (act[1], act[3], act[5] are the levels the lookup reads);
 * backward: dlev[3] level gradients (NULL = zero for the two finer ones), dw/db accumulate, scratch: 5 buffers shaped like
 * act[4], act[3], act[2], act[1], act[0]. */
int hnr_pyramid_fwd(const float* img, const float* const* w, const float* const* b, float* const* act, int64_t V, int64_t H, int64_t W,
                    void* stream);
int hnr_pyramid_bwd(const float* img, const float* const* w, const float* const* act, const float* const* dlev, float* const* dw,
                    float* const* db, float* const* scratch, int64_t V, int64_t H, int64_t W, void* stream);
/* One-launch re-packing of every weight image of the training step (csrc/pack.cu): device-resident job tables built by
 * hybridneuralrendering_b200/packer.py (struct layouts there and in pack.cu; sizes exported for the consistency check). */
int64_t hnr_pack_job_bytes(void);
int64_t hnr_bias_job_bytes(void);
int hnr_pack_weights(const void* jobs, int64_t njobs, int64_t total_pieces, const void* bias_jobs, int64_t nbias, int32_t* status,
                     void* stream);
int hnr_nbr_features_bwd_ld(const float* dX0, int64_t ldx, const float* dE, const float* emb, const int32_t* pidx, const uint8_t* mask,
                            const int32_t* vlist, const float* raydirs, const float* cam, int64_t Nv, int64_t K, float* d_emb,
                            float* d_color, float* d_dir, void* stream);

/* Fused chain of up to 4 dense layers (widths <= 128) on tcgen05, 3xFP16 split (csrc/chain_f16.cu): the per-sample MLPs
 * color_feature_branch, aux_merge_weight_block (+ sigmoid head), color_mixup_block (+ residual) of
 * point_aggregators.py:556-683 in one launch each, activations resident in shared memory between layers.
 * src/src_ld/src_k/src_mod: up to 3 concatenated fp32 sources (as hnr_linear_fwd).  Per-layer arrays have nlayer
 * entries: Kp (padded K), N, Np (N padded to 16), act, w_off (byte offset into wpack), mul, inv_next, Y (fp32 output of
 * the layer or NULL), ldy.  wpack/bias/mul/inv_next are built by hybridneuralrendering_b200/chain.py. */
int64_t hnr_chain_f16_chunk_bytes(int64_t Np);
/* profiling aid: CTA 0 of the following chain launches records (clock64, event, a, b) quadruples into buf
 * (int64[3][4096][2]: per role MMA / generator / epilogue, pairs (clock, id<<32 | a<<16 | b)); NULL switches it off */
void hnr_chain_f16_set_trace(void* buf);
int hnr_chain_f16_forward(const float* const* src, const int64_t* src_ld, const int64_t* src_k, const int64_t* src_mod, float in_scale,
                          int nlayer, const int64_t* Kp, const int64_t* N, const int64_t* Np, const int* act, const void* wpack,
                          const int64_t* w_off, const float* bias /* 4,128 */, const float* mul, const float* inv_next,
                          float* const* Y, const int64_t* ldy, const float* res, int64_t ldres, const float* head_w,
                          const float* head_b, int head_act, float* head_out /* M */, int64_t M,
                          int32_t* status /* optional device word: |= 2 when a value saturated fp16 */, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Compositing: neural_points_volumetric_model.py:331-339 + models/rendering/diff_ray_marching.py:508-557
 * ------------------------------------------------------------------------------------------- */
/* pass exactly one of z (camera depth per sample, element stride z_stride) or dist_in (ray_dist) */
int hnr_composite_fwd(const float* feats /* R,SR,4 */, const uint8_t* valid /* R,SR */, const float* z, int z_stride,
                      const float* dist_in, const float* bg /* 3 or NULL */, float vsize_z, int unit_mode, int64_t R, int64_t SR,
                      float* ray_color, float* opacity, float* acc_trans, float* blend_weight, float* bg_trans, float* dist_out,
                      void* stream);
int hnr_composite_bwd(const float* feats, const uint8_t* valid, const float* dist, const float* acc_trans, const float* bg_trans,
                      const float* bg, const float* g_color, const float* g_opacity, const float* g_bg_trans,
                      const float* g_blend_weight, const float* g_acc_trans, int64_t R, int64_t SR, float* g_feats, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Blur module: models/base_rendering_model.py:677-786
 * ------------------------------------------------------------------------------------------- */
int hnr_blur_select_fwd(const float* pred /* S*S,3 */, const float* gt, const float* kernels /* Nk,ks,ks */, int64_t patch_num,
                        int64_t patch_size, int64_t num_kernels, int64_t kernel_size, float* out, int32_t* select, void* stream);
int hnr_blur_select_bwd(const float* g_out, const float* kernels, const int32_t* select, int64_t patch_num, int64_t patch_size,
                        int64_t num_kernels, int64_t kernel_size, float* g_pred, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Learnable blur-kernel branch (SURVEY.md 8f N3): models/base_rendering_model.py:827-1020.
 *   hnr_blur_gray_*   predictor input rows feat (N, 2*ps*ps) = [mean_c gt | mean_c pred] per patch (:883-889)
 *   hnr_blur_learn_*  raw (N, ld_raw >= ks*ks [+1]) = the predictor's sigmoid outputs; kernel normalisation norm_mode 0 (/sum) or
 *                     1 (softmax) (:895-899); mix_mode 0, or 4 = predicted weight * kernel + (1-weight) * identity, renormalised
 *                     (:904-909); per-patch ks x ks zero-padded cross-correlation with boundary_mode 0 (/ (mask+1e-10)),
 *                     1 (+ (1-mask) * input) or 2 (as 1 with the mask detached from the kernel gradient) (:915-923)
 * ------------------------------------------------------------------------------------------- */
int hnr_blur_gray_fwd(const float* pred /* S*S,3 */, const float* gt, int64_t patch_num, int64_t patch_size, float* feat, void* stream);
int hnr_blur_gray_bwd(const float* g_feat, int64_t patch_num, int64_t patch_size, float* g_pred, void* stream);
int hnr_blur_learn_fwd(const float* pred, const float* raw, int64_t ld_raw, int64_t patch_num, int64_t patch_size, int64_t kernel_size,
                       int norm_mode, int mix_mode, int boundary_mode, float* out, void* stream);
int hnr_blur_learn_bwd(const float* pred, const float* raw, int64_t ld_raw, const float* g_out, int64_t patch_num, int64_t patch_size,
                       int64_t kernel_size, int norm_mode, int mix_mode, int boundary_mode, float* g_pred, float* g_raw, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused dense Adam step for the neural-point tables (SURVEY.md §8f N2; reference: one torch.optim.Adam over the point
 * parameters, models/mvs_points_volumetric_model.py:94-104).  Same arithmetic as torch.optim.Adam (amsgrad off);
 * step = 1-based count after this update.  One read of p,g,m,v and one write of p,m,v per element.
 * ------------------------------------------------------------------------------------------- */
int hnr_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int64_t step, void* stream);
/* the same step over nt <= 64 tensors in one launch (p/g/m/v/n: host arrays); guard: optional device word, the update is skipped
 * on the device when *guard != 0 (the saturation status of the split-fp16 kernels: a bad step is never applied). */
int hnr_adam_multi(int64_t nt, float* const* p, const float* const* g, float* const* m, float* const* v, const int64_t* n, float lr,
                   float beta1, float beta2, float eps, float weight_decay, int64_t step, const int32_t* guard, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Frame-dict producer on the device (SURVEY.md §8f N4): the per-item arithmetic of ScannetFtDataset.__getitem__
 * (data/scannet_ft_dataset.py:736-976) once the frames are decoded; the frames stay resident in HBM as uint8 (F,H,W,3).
 *   hnr_frame_rays   pixel grid + get_dtu_raydir (data/data_utils.py:57-71) + gt_image_full[py, px] lookup (:945-957).
 *                    patches = int32 (patch_num^2, 3) rows {x0, y0, dilation} in patch order (i, j) of the 'dilated' sampler
 *                    (:917-940; 'patch' mode = one patch with dilation 1, :887-892); NULL = full frame inside `margin`
 *                    (:941-944).  intrinsic = 9 floats row-major, c2w = 16 floats row-major, both DEVICE pointers.
 *                    Outputs: pixel_idx (n,2), raydir (n,3), gt_image (n,3) or NULL; n = (patch_num*patch_size)^2 or
 *                    (width-2*margin)*(height-2*margin).  frame_u8 = the item's own frame (H,W,3), only read for gt_image.
 *   hnr_frame_views  images_nearest (n_views, frame_bytes) fp32 = bank[view_ids[v]] / 255 (T.ToTensor, :743, :823-826);
 *                    frame_bytes = H*W*3.
 * ------------------------------------------------------------------------------------------- */
int hnr_frame_rays(const int32_t* patches, int64_t patch_num, int64_t patch_size, int64_t width, int64_t height, int64_t margin,
                   const float* intrinsic, const float* c2w, int dir_norm, const uint8_t* frame_u8, float* pixel_idx, float* raydir,
                   float* gt_image, void* stream);
int hnr_frame_views(const uint8_t* bank, const int32_t* view_ids, int64_t n_views, int64_t frame_bytes, float* out, void* stream);

/* ---- multi-GPU: one-shot SUM all-reduce of a small fp32 buffer over NVLink peer memory (csrc/peer.cu; SURVEY.md 8e).  No reference
 * counterpart (the reference is single-GPU, SURVEY.md 2.3); semantic = ncclAllReduce(ncclSum).  `peers`: device addresses of the
 * `world` copies of a symmetric buffer as mapped into this process, in rank order; result bit-identical on every rank. */
int hnr_peer_sum_f32(const void* const* peers, int world, int64_t n, float* out, void* stream);
/* the same with ONE multimem.ld_reduce per 16 bytes on the buffer's multicast address (reduction inside the NVSwitch) */
int hnr_multimem_sum_f32(const void* mc, int64_t n, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HNR_H */
