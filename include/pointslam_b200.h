/*
 * pointslam_b200.h -- C ABI of libpointslam_b200.so
 *
 * The B200-native (sm_100a) implementation of Point-SLAM's per-frame volumetric
 * rendering hot path.  The reference has NO native interface for this path: it is
 * a Python duck-typed API (src/neural_point.py, src/conv_onet/models/decoder.py,
 * src/utils/Renderer.py) whose GPU work is done by faiss-gpu 1.7.2 and ATen.  Each
 * entry point below names the reference call site it replaces; INTEGRATION.md shows
 * the ctypes binding a maintainer would add on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - all arithmetic tensors are contiguous float32, indices int32, radii float64
 *     (the reference's dynamic radii are float64 tensors, Tracker.py:247-250);
 *   - calls are asynchronous on `stream` (a cudaStream_t passed as void*), except
 *     psl_grid_sort which returns a host count and therefore synchronises;
 *   - the library allocates nothing the caller can see: scratch is passed in as
 *     (ws, ws_bytes), sized by the matching *_ws_bytes query;
 *   - return value 0 = success, negative = error (psl_last_error() gives the text);
 *   - no global mutable state except the per-thread last-error string: one process
 *     per GPU, any number of processes per box.
 */
#ifndef POINTSLAM_B200_H
#define POINTSLAM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSL_NN 8          /* pointcloud.nn_num   (configs/point_slam.yaml:107) */
#define PSL_CDIM 32       /* model.c_dim         (configs/point_slam.yaml:10)  */
#define PSL_GEO_EMB 93    /* decoder.py:101 */
#define PSL_COL_EMB 20    /* decoder.py:303 */
#define PSL_REL_EMB 10    /* decoder.py:313-314 */
#define PSL_GEO_HID 32    /* decoder.py:469 */
#define PSL_COL_HID 128   /* decoder.py:472 */

typedef void* psl_stream_t;

int psl_version(void);
const char* psl_last_error(void);
/* number of SMs of the current device (grid sizing is done inside the library) */
int psl_device_sm_count(void);
/* optional device timing: when enabled, every kernel launch made by the library is bracketed by CUDA events on the
 * launching stream; psl_timing_collect synchronises the device and returns summed milliseconds / launch counts per
 * kernel family: 0 knn, 1 decode_fwd, 2 decode_bwd, 3 composite/ray kernels, 4 feature scatter, 5 param pack,
 * 6 partial-gradient reduce, 7 colour forward (tcgen05), 8 colour backward data (tcgen05), 9 colour weight gradients
 * (tcgen05), 10 iteration-shell kernels (arrays of PSL_TIMING_SLOTS entries). */
#define PSL_TIMING_SLOTS 11
/* kernels launched by this process through the library so far (bench.py's gpu_launches) */
unsigned long long psl_launch_count(void);
int psl_timing_enable(int on);
int psl_timing_collect(float* ms_out_host, int* count_out_host);

/* ------------------------------------------------------------------------- *
 * K0  spatial hash of the neural point cloud
 * replaces: faiss GpuIndexIVFFlat train/add, src/neural_point.py:37-41,161-164
 * ------------------------------------------------------------------------- */
typedef struct psl_grid {
    const float* sorted_pts;      /* (n,4) float4: x,y,z,bitcast(original index); sorted by cell key */
    const uint64_t* table_keys;   /* (capacity) cell key or ~0 for empty                              */
    const uint32_t* table_vals;   /* (capacity,2) start,count into sorted_pts                         */
    uint32_t capacity;            /* power of two                                                     */
    int32_t n;                    /* number of points                                                 */
    float cell;                   /* cell edge length in metres                                       */
    float r_small;                /* first-pass search radius (0 = off): exact early exit when 8 points lie
                                     inside it, else the query radius is searched (see k_knn)            */
    const struct psl_grid_meta* meta; /* optional DEVICE copy of (capacity, n, r_small): when non-NULL the kernels read these
                                     three from device memory at run time instead of the launch arguments, so that
                                     a CUDA graph captured over fixed-capacity buffers stays valid after the cloud
                                     has grown and the hash has been rebuilt in place (add_neural_points,
                                     src/neural_point.py:147-164); the host fields must still describe a built grid */
} psl_grid;

typedef struct psl_grid_meta {    /* 16 bytes in device memory, written by the caller after each (re)build */
    uint32_t capacity;            /* power of two <= allocated table entries */
    int32_t n;
    float r_small;
    uint32_t reserved;
} psl_grid_meta;

size_t psl_grid_sort_ws_bytes(int64_t n);
/* step 1: keys, radix sort, gather.  Writes sorted_pts (n,4), sorted_keys (n) and returns the number
 * of occupied cells through *n_cells_host (synchronises `stream`). */
int psl_grid_sort(const float* cloud_pos, int64_t n, float cell, float* sorted_pts, uint64_t* sorted_keys,
                  void* ws, size_t ws_bytes, int64_t* n_cells_host, psl_stream_t stream);
/* step 1, incremental: after an append only the k_new new points (cloud_pos[n_old : n_old + k_new]) are keyed and sorted, then merged
 * (stable) into sorted_pts / sorted_keys IN PLACE (room for n_old + k_new entries) -- bit-identical to psl_grid_sort on the whole
 * cloud, without its 8 radix passes over every point.  This is the faiss `index.add(pts)` of neural_point.py:164. */
size_t psl_grid_append_ws_bytes(int64_t n_total, int64_t k_new);
int psl_grid_append(const float* cloud_pos, int64_t n_old, int64_t k_new, float cell, float* sorted_pts, uint64_t* sorted_keys,
                    void* ws, size_t ws_bytes, int64_t* n_cells_host, psl_stream_t stream);
/* step 2: fill the open-addressing table (capacity = power of two >= 2*n_cells, caller-allocated). */
int psl_grid_hash(const uint64_t* sorted_keys, int64_t n, uint64_t* table_keys, uint32_t* table_vals,
                  uint32_t capacity, psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * K1  ray-march + exact radius-kNN
 * replaces: Renderer.render_batch_ray sample placement (src/utils/Renderer.py:133-174) and
 *           NeuralPointCloud.find_neighbors_faiss (src/neural_point.py:169-215)
 *
 * Radius: r2 == NULL -> every query uses r2_scalar; else query m uses r2[m / r2_group].
 * Outputs per query: I (8) ascending by (D, index), -1 padded; D (8) squared L2 with the canonical
 * fp32 formula ((dx*dx+dy*dy)+dz*dz), FLT_MAX padded; nnum = #(D < r2) (strict, float64 compare).
 * Only neighbours with D <= r2 are reported (slots beyond the radius carry zero weight downstream).
 * ------------------------------------------------------------------------- */
int psl_knn_query(const psl_grid* grid_host, const float* pos, int64_t m, const double* r2, double r2_scalar,
                  int32_t r2_group, int32_t* I, float* D, int32_t* nnum, psl_stream_t stream);

/* rays: z = near*d*(1-t) + far*d*t for gt_depth>0 (operator order of Renderer.py:140-142), else the
 * row z_override[r] (may be NULL when all depths are > 0).  Writes z_vals (R,S), pos (R*S,3), I, D, nnum. */
int psl_raymarch_knn(const psl_grid* grid_host, const float* rays_o, const float* rays_d, const float* gt_depth,
                     int64_t n_rays, int32_t n_samples, const float* t_vals, float near_surface, float far_surface,
                     const float* z_override, const double* r2_ray, double r2_scalar,
                     float* z_vals, float* pos, int32_t* I, float* D, int32_t* nnum, psl_stream_t stream);
/* the same search with work counters for the bench's roofline line (SURVEY.md section 8d asks for the mean number of candidates
 * visited per query): stats (4 device uint64, zeroed by the caller) += [candidate points staged, warp search passes, queries,
 * hash cells probed] */
int psl_raymarch_knn_stats(const psl_grid* grid_host, const float* rays_o, const float* rays_d, const float* gt_depth,
                           int64_t n_rays, int32_t n_samples, const float* t_vals, float near_surface, float far_surface,
                           const float* z_override, const double* r2_ray, double r2_scalar,
                           float* z_vals, float* pos, int32_t* I, float* D, int32_t* nnum, uint64_t* stats, psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * K2+K3  IDW interpolation + per-neighbour colour MLP + geometry/colour MLP decode
 * replaces: POINT.forward (src/conv_onet/models/decoder.py:476-518) incl. get_feature_at_pos (:130-173,
 *           :341-390), GaussianFourierFeatureTransform (:30-37), MLP_geometry.forward (:175-222),
 *           MLP_color.forward (:392-449) and their autograd backward.
 * ------------------------------------------------------------------------- */
typedef struct psl_decoder_params {        /* row-major (out,in) exactly like the reference state_dict */
    const float* g_B;                      /* geo_decoder.embedder._B            (3,93)   */
    const float* g_W[5];                   /* geo_decoder.pts_linears.i.weight   (32,93|32|32|125|32) */
    const float* g_b[5];
    const float* g_Wc[5];                  /* geo_decoder.fc_c.i.weight          (32,32)  */
    const float* g_bc[5];
    const float* g_Wo;                     /* geo_decoder.output_linear.weight   (1,32)   */
    const float* g_bo;
    const float* c_B;                      /* color_decoder.embedder._B          (3,20)   */
    const float* c_Brel;                   /* color_decoder.embedder_rel_pos._B  (3,10)   */
    const float* c_N1;                     /* mlp_col_neighbor.linear1.weight    (128,52) */
    const float* c_n1b;
    const float* c_N2;                     /* mlp_col_neighbor.linear2.weight    (32,128) */
    const float* c_n2b;
    const float* c_W[5];                   /* color_decoder.pts_linears.i.weight (128,40|128|128|168|128) */
    const float* c_b[5];
    const float* c_Wc[5];                  /* color_decoder.fc_c.i.weight        (128,32) */
    const float* c_bc[5];
    const float* c_Wo;                     /* color_decoder.output_linear.weight (3,128)  */
    const float* c_bo;
} psl_decoder_params;

/* same field order, float* destinations; a NULL entry means "gradient not wanted" */
typedef struct psl_decoder_grads {
    float* g_B; float* g_W[5]; float* g_b[5]; float* g_Wc[5]; float* g_bc[5]; float* g_Wo; float* g_bo;
    float* c_B; float* c_Brel; float* c_N1; float* c_n1b; float* c_N2; float* c_n2b;
    float* c_W[5]; float* c_b[5]; float* c_Wc[5]; float* c_bc[5]; float* c_Wo; float* c_bo;
} psl_decoder_grads;

enum { PSL_STAGE_GEOMETRY = 0, PSL_STAGE_COLOR = 1 };
enum { PSL_RGB_SIGMOID = 0,      /* decoder.py:447                                     */
       PSL_RGB_AFFINE_SIGMOID = 1,/* sigmoid(out @ rot + trans), decoder.py:433-438     */
       PSL_RGB_RAW = 2 };        /* encode_exposure with exposure_feat None, :439-445  */
enum { PSL_WEIGHT_DISTANCE = 0, PSL_WEIGHT_EXPO = 1 };   /* pointcloud.nn_weighting, decoder.py:152-156 */

typedef struct psl_decode_cfg {
    int32_t stage;            /* PSL_STAGE_*                                                         */
    int32_t encode_rel_pos;   /* model.encode_rel_pos_in_col                                         */
    int32_t rgb_mode;         /* PSL_RGB_*                                                           */
    int32_t weighting;        /* PSL_WEIGHT_*                                                        */
    int32_t min_nn;           /* pointcloud.min_nn_num (2)                                           */
    int32_t r2_group;         /* r2[m / r2_group]; ignored when r2 == NULL                            */
    int32_t is_tracker;       /* backward only: propagate to pos through the recomputed D (:143-148) */
    int32_t reserved;         /* bit 0 (psl_decode_fwd, geometry stage): write only raw[:,3] (the colour kernel owns raw[:,0:3]) */
    double r2_scalar;
} psl_decode_cfg;

size_t psl_packed_params_floats(void);
/* floats of activations kept per sample for the backward (0 when save == NULL is passed to forward) */
size_t psl_decode_save_floats_per_sample(const psl_decode_cfg* cfg);
size_t psl_decode_bwd_ws_bytes(int64_t m);

/* repack the reference-layout parameters into the transposed/padded blob the kernels stage in shared memory */
int psl_pack_params(const psl_decoder_params* params_host, float* packed, psl_stream_t stream);

/* forward.  raw (m,4) = [rgb, occ]; has_nb (m) uint8.  exposure_affine: 12 floats (rot row-major 3x3, trans 3)
 * or NULL.  rand_geo / rand_col: the N(0,0.01^2) vectors given to samples without neighbours (decoder.py:170,387).
 * save: NULL (inference) or m * psl_decode_save_floats_per_sample floats. */
int psl_decode_fwd(const psl_decode_cfg* cfg, const float* packed, const float* pos, int64_t m,
                   const int32_t* I, const float* D, const int32_t* nnum, const double* r2,
                   const float* cloud_pos, const float* geo_feats, const float* col_feats,
                   const float* rand_geo, const float* rand_col, const float* exposure_affine,
                   float* raw, uint8_t* has_nb, float* save, psl_stream_t stream);

/* backward.  d_raw (m,4).  Outputs (any may be NULL): d_pos (m,3); pair gradients for the deterministic
 * feature scatter: d_cg (m,32) (geometry feature grad before IDW), wn (m,8) normalised weights,
 * d_colpair (m,8,32) (gradient w.r.t. col_feats[I[m,k]]); parameter grads via psl_decoder_grads;
 * d_exposure_affine (12).  ws: psl_decode_bwd_ws_bytes(m). */
int psl_decode_bwd(const psl_decode_cfg* cfg, const psl_decoder_params* params_host, const float* packed,
                   const float* pos, int64_t m, const int32_t* I, const float* D, const int32_t* nnum,
                   const double* r2, const float* cloud_pos, const float* geo_feats, const float* col_feats,
                   const float* exposure_affine, const float* raw, const float* save, const float* d_raw,
                   float* d_pos, float* d_cg, float* wn, float* d_colpair,
                   const psl_decoder_grads* grads_host, float* d_exposure_affine,
                   const float* dwn_extra /* (m,8) or NULL: added to dL/d(weights) */,
                   const float* dpos_extra /* (m,3) or NULL: added to d_pos */,
                   void* ws, size_t ws_bytes, psl_stream_t stream);

/* d_pos (m,3) += dpos_add (m,3 or NULL) + the IDW-weight chain rule (d wn -> d D -> d pos, tracker path of decoder.py:143-163)
 * applied to dwn (m,8).  The chain is linear in d wn: psl_decode_bwd applies it to the geometry branch's own share while the
 * colour backward runs on another stream, and this pass adds the colour branch's share (its dwn / dpos outputs) afterwards. */
int psl_idw_chain(const psl_decode_cfg* cfg, const float* pos, int64_t m, const int32_t* I, const float* D, const double* r2,
                  const float* cloud_pos, const float* dwn, const float* dpos_add, float* d_pos, psl_stream_t stream);

/* deterministic scatter of per-(sample,neighbour) feature gradients into dense (n_points,32) tensors
 * (replaces ATen's sort-based index_put_(accumulate=True) backward of feats[I], decoder.py:164,372).
 * d_geo / d_col must be zero-filled by the caller; either may be NULL. */
size_t psl_feat_scatter_ws_bytes(int64_t m);
int psl_feat_scatter(const int32_t* I, int64_t m, int64_t n_points, const float* wn, const float* d_cg,
                     const float* d_colpair, const float* d_cc, float* d_geo, float* d_col,
                     void* ws, size_t ws_bytes, psl_stream_t stream);

/* same, into a compact (n_rows,32) gradient of a SUBSET of the points: row_map (n_points) gives the output row of a point or
 * -1 (its pairs are dropped) -- the frustum-selected slices Mapper.optimize_map optimises (Mapper.py:345-414) without the
 * dense index_put / gather round trip.  n_rows replaces n_points as the row count of d_geo / d_col. */
int psl_feat_scatter_mapped(const int32_t* I, int64_t m, const int32_t* row_map, int64_t n_rows, const float* wn,
                            const float* d_cg, const float* d_colpair, const float* d_cc, float* d_geo, float* d_col,
                            void* ws, size_t ws_bytes, psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * alpha composite      replaces: raw2outputs_nerf_color (src/common.py:298-336) + the -100 masking of
 *                      Renderer.py:189-190 (mask applied to the VALUE only, gradient passes through)
 * ------------------------------------------------------------------------- */
int psl_composite_fwd(const float* raw, const uint8_t* has_nb, const float* z_vals, int64_t n_rays, int32_t n_samples,
                      float coef, float* depth, float* var, float* rgb, float* weights, psl_stream_t stream);
int psl_composite_bwd(const float* raw, const uint8_t* has_nb, const float* z_vals, int64_t n_rays, int32_t n_samples,
                      float coef, const float* d_depth, const float* d_var, const float* d_rgb,
                      float* d_raw, psl_stream_t stream);

/* d_rays_o = sum_s d_pos, d_rays_d = sum_s z * d_pos   (backward of Renderer.py:172-174) */
int psl_rays_bwd(const float* d_pos, const float* z_vals, int64_t n_rays, int32_t n_samples,
                 float* d_rays_o, float* d_rays_d, psl_stream_t stream);

/* ray validity: >= int(S/2+1) samples with neighbours (decoder.py:200-201) */
int psl_ray_mask(const uint8_t* has_nb, int64_t n_rays, int32_t n_samples, int32_t min_count, uint8_t* ray_mask,
                 psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * tensor-core (tcgen05, 3xTF32, TMEM-resident activations, 16 worker warps) colour branch: the A/B baseline of the f16-plane
 * kernels below (PSL_H2=0 / PSL_H2_BWD=0) and the producer of FFMA-layout activations.
 * psl_tc_pack_params folds fc_c into the next layer and lays the weights out as canonical K-major tf32 hi/lo chunk
 * images (blob: psl_tc_blob_floats() floats).  psl_color_fwd_tc writes raw[:, 0:3]; raw[:, 3] and has_nb come from
 * psl_decode_fwd(stage = PSL_STAGE_GEOMETRY) on the same kNN result.  Same reference lines as psl_decode_fwd.
 * ------------------------------------------------------------------------- */
size_t psl_tc_blob_floats(void);
int psl_tc_pack_params(const psl_decoder_params* params_host, float* tc_blob, psl_stream_t stream);
/* only the folded fp32 rows + small vectors of the above (what psl_h2_pack_params / psl_h2_bwd_pack_params read), no tf32 images */
int psl_tc_fold_params(const psl_decoder_params* params_host, float* tc_blob, psl_stream_t stream);
int psl_color_fwd_tc(const psl_decode_cfg* cfg, const float* tc_blob, const float* pos, int64_t m, const int32_t* I,
                     const float* D, const int32_t* nnum, const double* r2, const float* cloud_pos,
                     const float* col_feats, const float* rand_col, const float* exposure_affine, float* raw,
                     float* save /* NULL, or the psl_decode_fwd save buffer (FFMA backward) */,
                     float* tsave /* NULL, or psl_tc_save_floats() floats (tensor-core backward) */, psl_stream_t stream);

/* Round-2 forward of the colour branch: operands as f16 hi/lo planes (kind::f16, three MMAs per K = 16 step, same accuracy as
 * 3xTF32 at twice the MMA rate and half the TMEM / weight bytes) and TWO tiles in flight per CTA (csrc/psl_color_h2.cu).
 * psl_h2_pack_params builds its operand image (psl_h2_blob_bytes() bytes) from the folded matrices psl_tc_pack_params left in
 * `tc_blob`; psl_color_fwd_h2 has the contract of psl_color_fwd_tc without the FFMA-layout `save` (tsave or inference only). */
size_t psl_h2_blob_bytes(void);
int psl_h2_pack_params(const psl_decoder_params* params_host, const float* tc_blob, void* h2_blob, psl_stream_t stream);
int psl_color_fwd_h2(const psl_decode_cfg* cfg, const void* h2_blob, const float* pos, int64_t m, const int32_t* I,
                     const float* D, const int32_t* nnum, const double* r2, const float* cloud_pos, const float* col_feats,
                     const float* rand_col, const float* exposure_affine, float* raw, float* tsave, psl_stream_t stream);

/* Round-2 backward (data gradients) of the colour branch on f16 hi/lo planes with a per-row power-of-two gradient scale
 * (csrc/psl_color_bwd_h2.cu): contract of psl_color_bwd_tc, operand image from psl_h2_bwd_pack_params (psl_h2_bwd_blob_bytes()). */
size_t psl_h2_bwd_blob_bytes(void);
int psl_h2_bwd_pack_params(const psl_decoder_params* params_host, const float* tc_blob, void* h2_bwd_blob, psl_stream_t stream);
int psl_color_bwd_h2(const psl_decode_cfg* cfg, const void* h2_bwd_blob, const float* pos, int64_t m, const int32_t* I,
                     const float* D, const int32_t* nnum, const double* r2, const float* cloud_pos, const float* col_feats,
                     const float* exposure_affine, const float* raw, const float* d_raw, const float* tsave, float* tbwd,
                     float* d_colpair, float* wn_out, float* dwn_col, float* dpos_col, int32_t want_wgrad, int32_t* grid_out,
                     psl_stream_t stream);

/* tensor-core training path of the colour branch: psl_color_fwd_tc(tsave) -> psl_color_bwd_tc (data gradients; the
 * geometry branch, the IDW-weight gradient and d_pos are finished by psl_decode_bwd(stage = GEOMETRY, dwn_extra, dpos_extra)). */
size_t psl_tc_fold_offset_floats(void);
size_t psl_tc_bwd_blob_floats(void);
size_t psl_tc_save_floats(int64_t m, int32_t encode_rel_pos);
size_t psl_tc_bwd_tmp_floats(int64_t m, int32_t encode_rel_pos);
int psl_tc_bwd_pack_params(const psl_decoder_params* params_host, const float* tc_blob, size_t tc_fold_offset_floats,
                           float* bwd_blob, psl_stream_t stream);
int psl_color_bwd_tc(const psl_decode_cfg* cfg, const float* bwd_blob, const float* pos, int64_t m, const int32_t* I,
                     const float* D, const int32_t* nnum, const double* r2, const float* cloud_pos, const float* col_feats,
                     const float* exposure_affine, const float* raw, const float* d_raw, const float* tsave, float* tbwd,
                     float* d_colpair, float* wn_out, float* dwn_col, float* dpos_col, int32_t want_wgrad, int32_t* grid_out,
                     psl_stream_t stream);


/* weight gradients of the colour branch (GEMMs over the sample index) from the buffers left by psl_color_fwd_tc(tsave) and
 * psl_color_bwd_tc(want_wgrad = 1); only the c_* entries of `grads_host` are written.  ws: psl_wgrad_tc_ws_floats(m). */
size_t psl_wgrad_tc_ws_floats(int64_t m);
int psl_wgrad_tc(const psl_decode_cfg* cfg, const psl_decoder_params* params_host, const float* pos, int64_t m, const int32_t* I,
                 const float* cloud_pos, const float* col_feats, const float* tsave, const float* tbwd, int32_t n_cta_bwd,
                 const psl_decoder_grads* grads_host, float* d_exposure_affine, float* ws, size_t ws_floats, psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * iteration shell       the per-iteration glue of the two callers as single kernels (no data-dependent shapes, no host
 *                       synchronisation, fixed-order reductions), so that one optimisation iteration is ~20 launches
 *                       and can be replayed as a CUDA graph.
 * ------------------------------------------------------------------------- */
/* pixel sampling -> rays.  pix (n_frames*per_frame) int64: index into the (H - 2*H0... ) window, row = pix / win_w + H0,
 * column = pix % win_w + W0 (common.get_sample_uv, common.py:77-89); pix < 0 = no pixel: sampled depth 0 (zero loss weight).  Pose: `cam` (7) = [quaternion w,x,y,z (not normalised), T]
 * (common.get_camera_from_tensor, common.py:225-267) for ONE frame, or `c2w` (n_frames,3,4).  Outputs: rays_o/rays_d
 * (common.get_rays_from_uv, common.py:40-56), the sampled depth / colour and r2 = dyn_radius^2 (float64, may be NULL). */
int psl_sample_rays(const int64_t* pix, int32_t n_frames, int32_t per_frame, int32_t H, int32_t W, int32_t H0, int32_t W0,
                    int32_t win_w, const float* cam, const float* c2w, const float* color /* (n_frames,H,W,3) */,
                    const float* depth /* (n_frames,H,W) */, const double* dyn_radius /* (n_frames,H,W) or NULL */,
                    float fx, float fy, float cx, float cy, float* rays_o, float* rays_d, float* b_depth, float* b_color,
                    double* r2, psl_stream_t stream);
/* inside = depth > 0 and depth <= min(10 * median(depth > 0), 1.2 * max(depth))  (Tracker.py:142-148, Mapper.py:507-513);
 * depth_in = depth where inside else 0 (rays that the reference compacts away stay in the batch with zero weight). n <= 8192 */
int psl_depth_gate(const float* b_depth, int32_t n, float* depth_in, uint8_t* inside, psl_stream_t stream);
/* loss AND its gradient w.r.t. the rendered depth / colour.  mode 0 = tracking (Tracker.py:158-180, uncertainty-normalised,
 * 10x-mean outlier mask, clamp 1e3), mode 1 = mapping (Mapper.py:524-552).  d_rgb NULL: depth term only (geometry stage). */
int psl_shell_loss(int32_t mode, int32_t n, const float* depth_in, const uint8_t* inside, const uint8_t* ray_mask,
                   const float* depth, const float* var, const float* rgb, const float* b_color, float w_color,
                   float* loss, float* d_depth, float* d_rgb, psl_stream_t stream);
/* render tail of one optimisation iteration in ONE launch: composite (common.py:298-336, Renderer.py:189-190 masking), ray validity
 * (decoder.py:200-201, min_count = int(S / 2 + 1)), the loss of psl_shell_loss (mode 0 tracking, 1 mapping; b_color NULL = depth term
 * only) and the composite backward.  Writes depth / var / rgb / ray_mask (n), loss (1) and d_raw (n * n_samples, 4).
 * mode 1 runs one thread per ray over many CTAs and reduces the loss in a fixed order through `ws` (psl_render_tail_ws_bytes(n)
 * bytes, zero-initialised ONCE by the caller: the kernel re-arms its ticket); mode 0 (batch statistic) is a single-CTA launch. */
size_t psl_render_tail_ws_bytes(int32_t n);
int psl_render_tail(int32_t mode, int32_t n, int32_t n_samples, float coef, int32_t min_count, const float* raw,
                    const uint8_t* has_nb, const float* z_vals, const float* depth_in, const uint8_t* inside,
                    const float* b_color, float w_color, float* depth, float* var, float* rgb, uint8_t* ray_mask,
                    float* loss, float* d_raw, void* ws, size_t ws_bytes, psl_stream_t stream);

/* chain rule of psl_sample_rays(cam): (d_rays_o, d_rays_d) (n,3) -> d_cam (7) */
int psl_pose_bwd(const int64_t* pix, int32_t n, int32_t H0, int32_t W0, int32_t win_w, float fx, float fy, float cx, float cy,
                 const float* cam, const float* d_rays_o, const float* d_rays_d, float* d_cam, psl_stream_t stream);
/* torch.optim.Adam step (no weight decay / amsgrad) on `n_slots` rows of width `width`: slot u updates row rows[u] of `param`
 * (rows NULL: row u; rows[u] < 0: skipped) from grad/exp_avg/exp_avg_sq (n_slots,width); `step` (device int) is incremented
 * first.  zero_grad != 0 clears the consumed gradient (so that psl_feat_scatter_mapped finds a zeroed buffer). */
int psl_adam_rows(float* param, float* grad, float* exp_avg, float* exp_avg_sq, const int64_t* rows, int64_t n_slots,
                  int32_t width, int32_t* step, float lr, float beta1, float beta2, float eps, int32_t zero_grad,
                  psl_stream_t stream);
/* Tracker pose step (Tracker.py:289-349): torch.optim.Adam on cam = [quat(4), T(3)] with lr_quat / lr_trans (tracking.separate_LR:
 * lr/5 and lr; one shared step count) and, when best_loss != NULL, the candidate bookkeeping of the tracking loop: if *loss <
 * *best_loss the pose is copied to best_cam -- the pose this iteration rendered with (candidate_pre_step != 0, the separate_LR
 * branch) or the stepped pose (candidate_pre_step == 0) -- and *best_loss updated.  One launch. */
int psl_pose_adam(float* cam, const float* d_cam, float* exp_avg, float* exp_avg_sq, int32_t* step, float lr_quat, float lr_trans,
                  float beta1, float beta2, float eps, const float* loss, float* best_loss, float* best_cam,
                  int32_t candidate_pre_step, psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * map maintenance between renders (SURVEY.md section 8f rank 1)
 * ------------------------------------------------------------------------- */
/* NeuralPointCloud.add_neural_points (src/neural_point.py:91-167) without host round trips.  For ray i with
 * gt_depth[i] > 0 the surface point p = o + d*depth is tested against the indexed cloud: kept iff NO point has
 * D < r^2 (canonical fp32 D, float64 compare; r^2 = r2_valid[rank of i among the depth > 0 rays] or r2_scalar;
 * an empty grid keeps every valid ray, :116).  Kept rays are compacted IN ORDER: ray with keep-rank j writes
 * input_pos[j] = p, input_rgb[j] = 255*gt_color[i] (both optional) and its n_add points o + d*z_s to
 * new_pos[j*n_add + s], z_s = near*depth*(1-steps[s]) + far*depth*steps[s]  (:135-137, steps = linspace(0,1,n_add)) or
 * depth + steps[s] when fixed_interval (:131-133, steps = linspace(-0.04,0.04,n_add)).  counts (device, 2 x int32) =
 * {number of depth > 0 rays, number of kept rays}.  new_pos needs room for n*n_add points.  ws: psl_add_points_ws_bytes(n). */
size_t psl_add_points_ws_bytes(int64_t n);
int psl_add_points(const psl_grid* grid_host, const float* rays_o, const float* rays_d, const float* gt_depth,
                   const float* gt_color /* (n,3) or NULL */, int64_t n, const double* r2_valid, double r2_scalar,
                   int32_t n_add, int32_t fixed_interval, float near_surface, float far_surface, const float* steps,
                   float* new_pos, float* input_pos, float* input_rgb, int32_t* counts, void* ws, size_t ws_bytes,
                   psl_stream_t stream);
/* Mapper.get_mask_from_c2w (src/Mapper.py:120-168): frustum feature selection.  w2c_host: 12 doubles on the HOST = rows
 * 0..2 of numpy.linalg.inv(c2w float32) promoted to float64 (the reference inverts in float32 and projects a float64
 * copy of the cloud).  depth (H,W) float32 sensor depth; the bilinear lookup reproduces cv2.remap(INTER_LINEAR, border 0)
 * bit for bit; depth must be NaN-free.  mask (n) uint8; indices (optional, room for n) receives np.where(mask)[0] in
 * ascending order and *count (device int32) its length.  ws: psl_frustum_select_ws_bytes(n). */
size_t psl_frustum_select_ws_bytes(int64_t n);
int psl_frustum_select(const float* cloud_pos, int64_t n, const double* w2c_host, double fx, double fy, double cx, double cy,
                       const float* depth, int32_t H, int32_t W, int32_t edge, uint8_t* mask, int64_t* indices,
                       int32_t* count, void* ws, size_t ws_bytes, psl_stream_t stream);

/* ------------------------------------------------------------------------- *
 * per-frame colour gradient: dynamic-radius maps and gradient-based pixel selection
 * ------------------------------------------------------------------------- */
/* color (H,W,3) float32 -> float64 (H,W) maps, exactly as synth.sobel_radius_map computes them (Tracker.py:237-248):
 * grey = 0.2125 R + 0.7154 G + 0.0721 B, 3x3 Sobel with [1,2,1]/4 smoothing and a zeroed 1-pixel border,
 * mag = sqrt(gx^2 + gy^2) (not clipped), r_add = np.interp(clip(mag, 0, thr), [0, 0.01, thr], [r_add_max, r_add_max, r_add_min]),
 * r_query = radius_query_ratio * r_add.  Any output may be NULL.  color_grad_threshold must exceed 0.01. */
int psl_frame_grad(const float* color, int32_t H, int32_t W, double r_add_max, double r_add_min, double radius_query_ratio,
                   double color_grad_threshold, double* mag, double* r_add, double* r_query, psl_stream_t stream);
/* Candidate pixels of get_selected_index_with_grad (common.py:92-159): the k pixels of largest mag (H,W) over the whole image
 * (ties: the smaller flat index first), of those the ones with H0 <= row < H1, W0 <= column < W1 and 0 < depth <= depth_max
 * (+inf: no upper bound).  cand (room for k) receives their flat indices row * W + column in ascending order, *count (device
 * int32) their number.  No host synchronisation.  ws: psl_grad_candidates_ws_bytes(H * W). */
size_t psl_grad_candidates_ws_bytes(int32_t n_pixels);
int psl_grad_candidates(const double* mag, const float* depth, int32_t H, int32_t W, int32_t H0, int32_t H1, int32_t W0, int32_t W1,
                        float depth_max, int32_t k, int64_t* cand, int32_t* count, void* ws, size_t ws_bytes, psl_stream_t stream);
/* n distinct entries of cand[0 .. *count) drawn uniformly without replacement: keys (capacity) uint32 are the caller's random
 * keys, one per candidate slot; the n slots of smallest key (ties: smaller slot) are taken.  pix (n) int64 receives them as
 * window-relative indices (row - H0) * win_w + (column - W0), the form psl_sample_rays / psl_pose_bwd take; when *count < n
 * the slots beyond it are -1 ("no pixel": psl_sample_rays gives such a sample depth 0, so it carries no loss).  Shapes depend
 * on capacity and n only.  ws: psl_pick_candidates_ws_bytes(capacity). */
size_t psl_pick_candidates_ws_bytes(int32_t capacity);
int psl_pick_candidates(const int64_t* cand, const int32_t* count, int32_t capacity, const uint32_t* keys, int32_t n, int32_t W,
                        int32_t H0, int32_t W0, int32_t win_w, int64_t* pix, void* ws, size_t ws_bytes, psl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* POINTSLAM_B200_H */
