/*
 * neuradar_b200.h - C ABI of libneuradar_b200.so: the NeuRadar per-ray neural-field hot path on B200 (sm_100a).
 *
 * Conventions (SURVEY.md 8b):
 *   - every pointer is a DEVICE pointer to a contiguous row-major fp32 array unless stated otherwise;
 *   - the caller owns and pre-allocates every buffer; no entry point allocates or synchronises;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); distinct streams may be used concurrently;
 *   - return value: 0 on success, a negative NRB_ERR_* code for argument errors (nothing is launched), or the
 *     positive cudaError_t of the failed launch.  nrb_last_error_string() describes the last failure of the
 *     calling thread.
 *   - there is no CPU fallback: on a machine without an sm_100 device every launch fails with a CUDA error.
 *
 * The reference (mrafidashti/neuradar, a nerfstudio fork) has no native code; each entry point below replaces a
 * call site of its torch / tiny-cuda-nn / nerfacc path.  Citations are file:line in the reference checkout.
 */
#ifndef NEURADAR_B200_H
#define NEURADAR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRB_VERSION 100 /* major*10000 + minor*100 + patch */

#define NRB_OK 0
#define NRB_ERR_BAD_ARG (-1)     /* null pointer, non-positive or out-of-range dimension */
#define NRB_ERR_ALIGNMENT (-2)   /* a vector-accessed pointer is not 16-byte aligned */
#define NRB_ERR_UNSUPPORTED (-3) /* configuration outside what the kernels were built for */

#define NRB_MAX_LEVELS 16
#define NRB_MAX_MLP_LAYERS 4
#define NRB_MAX_MLP_WIDTH 64
#define NRB_MAX_SAMPLES 256 /* samples per ray handled by the warp-per-ray kernels */
#define NRB_MAX_ACTORS 256  /* per-actor hash grids handled by the fused kernels */

typedef void* nrb_stream_t; /* cudaStream_t */

/* One multiresolution hash grid = HashEncoding (nerfstudio/field_components/encodings.py:311-384).
 * `table` is the `hash_table` parameter [num_levels * 2^log2_hashmap_size, features_per_level];
 * `scalings` are the per-level resolutions of the `scalings` buffer (encodings.py:350), by value. */
typedef struct {
  const float* table;
  float scalings[NRB_MAX_LEVELS];
  int32_t num_levels;
  int32_t features_per_level; /* 1, 2 or 4 */
  int32_t log2_hashmap_size;  /* <= 24 */
} nrb_grid_t;

/* Per-ray inputs = the RayBundle fields the path reads (nerfstudio/cameras/rays.py:251-271), un-broadcast. */
typedef struct {
  const float* origins;    /* [N,3] */
  const float* directions; /* [N,3] */
  const float* pixel_area; /* [N]   */
  const float* nears;      /* [N]   */
  const float* fars;       /* [N]   */
  int64_t num_rays;
} nrb_rays_t;

/* Sample intervals along rays = Frustums.starts / Frustums.ends (nerfstudio/cameras/rays.py:41-44), [N, S] each
 * with a common row stride.  Samples cut from S+1 shared bin edges (what every sampler on the path produces,
 * ray_samplers.py:122-129,368-374) are passed as starts = bins, ends = bins + 1, row_stride = S + 1. */
typedef struct {
  const float* starts;
  const float* ends;
  int64_t row_stride;
  int32_t num_samples;
} nrb_intervals_t;

/* Linear+ReLU chain = MLP.pytorch_fwd (nerfstudio/field_components/mlp.py:142-178).
 * weights[i] is layers.i.weight [dims[i+1], dims[i]], biases[i] is layers.i.bias [dims[i+1]] or NULL. */
typedef struct {
  const float* weights[NRB_MAX_MLP_LAYERS];
  const float* biases[NRB_MAX_MLP_LAYERS];
  int32_t dims[NRB_MAX_MLP_LAYERS + 1];
  int32_t num_layers;
} nrb_mlp_t;

/* Gradient sinks matching nrb_mlp_t; every buffer is ACCUMULATED into (caller zeroes). */
typedef struct {
  float* weights[NRB_MAX_MLP_LAYERS];
  float* biases[NRB_MAX_MLP_LAYERS];
} nrb_mlp_grad_t;

/* Power-transform spacing of PowerSampler (nerfstudio/model_components/ray_samplers.py:838-852,
 * nerfstudio/utils/math.py:541-580): spacing_fn(x) = power_fn(x*scaling, lambda). */
typedef struct {
  float lambda;
  float scaling;
} nrb_spacing_t;

int nrb_version(void);
/* NRB_MAX_ACTORS of this build: the length of nrb_actor_grids_t::tables, so that a binding can check its mirror. */
int32_t nrb_max_actors(void);
const char* nrb_last_error_string(void);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
int64_t nrb_launch_count(void);

/* ---- hash grid: HashEncoding.pytorch_fwd, encodings.py:425-466 (replaces the tcnn.Encoding call, :468-470) ----
 * x [M,3] in grid units [0,1]; out [M, L*F].  When `std` [M] is non-NULL each level is additionally multiplied by
 * 1/max(1, 2*scalings[l]*std) = NeuRADHashEncoding._rescale_grid_features (neurad_encoding.py:309-316). */
int nrb_hash_fwd(const nrb_grid_t* grid, const float* x, const float* std, float* out, int64_t M, nrb_stream_t stream);
/* Table rows of the 8 cell corners, idx [M, L, 8] int64 in the corner order of encodings.py:436-443
 * (HashEncoding.hash_fn, encodings.py:406-423).  Parity/debug entry: bit-exact with the reference. */
int nrb_hash_indices(const nrb_grid_t* grid, const float* x, int64_t* idx, int64_t M, nrb_stream_t stream);
/* Backward of nrb_hash_fwd: dtable [L*T, F] += scatter(dy [M, L*F]);  dx [M,3] (optional, may be NULL) is
 * OVERWRITTEN with the gradient through the in-cell offsets (floor/ceil have zero gradient).
 * `workspace` (optional, 16-byte aligned, nrb_hash_bwd_workspace_bytes(grid, M) bytes, contents ignored) lets the
 * kernel spread the reductions of the coarse levels over replicated lattices; without it the result is the same,
 * only slower. */
int64_t nrb_hash_bwd_workspace_bytes(const nrb_grid_t* grid, int64_t M);
int nrb_hash_bwd(const nrb_grid_t* grid, const float* x, const float* std, const float* dy, float* dtable, float* dx,
                 int64_t M, void* workspace, int64_t workspace_bytes, nrb_stream_t stream);

/* ---- sample gaussians + contraction: Frustums.get_fast_isotropic_gaussian(1) (cameras/rays.py:109-124) followed by
 * ScaledSceneContraction(order=inf, scale) on GaussiansStd (field_components/spatial_distortions.py:103-113,132-136).
 * x [N*S, 3] contracted means in [0,1]^3, std [N*S] contracted standard deviations. */
int nrb_frustum_gaussians(const nrb_rays_t* rays, const nrb_intervals_t* iv, float scale, float* x, float* std,
                          nrb_stream_t stream);

/* ---- tiny MLP: MLP.pytorch_fwd (mlp.py:159-178; replaces tcnn.Network, mlp.py:109-113) ----
 * x [M, dims[0]] -> y [M, dims[L]].  `hidden` (optional) receives the post-ReLU activations of the L-1 hidden
 * layers, feature-major: layer i at hidden + M * sum(dims[1..i]) laid out [dims[i+1], M]; needed by nrb_mlp_bwd. */
int nrb_mlp_fwd(const nrb_mlp_t* mlp, const float* x, float* y, float* hidden, int64_t M, nrb_stream_t stream);
int nrb_mlp_bwd(const nrb_mlp_t* mlp, const float* x, const float* hidden, const float* dy, float* dx,
                const nrb_mlp_grad_t* grads, int64_t M, nrb_stream_t stream);

/* ---- the NeuRAD field's two MLPs (fields/neurad_field.py:132-152; they replace the two tcnn FullyFusedMLP networks,
 * mlp.py:109-127), as the fused field kernels below evaluate them:
 *   geo = mlp_geo(x) [32 -> 32 ReLU -> 33]; sdf, emb = split(geo, [1, 32]);
 *   feature = emb + mlp_feature([emb, sh]) [48 -> 32 ReLU -> 32 ReLU -> 32]; alpha = sigmoid(-sdf (|beta| + beta_min)).
 * weights[0..1] = mlp_geo.layers.{0,1}.weight, weights[2..4] = mlp_feature.layers.{0,1,2}.weight ([out,in] row-major),
 * biases likewise (may be NULL). */
typedef struct {
  const float* weights[5];
  const float* biases[5];
  const float* beta;
  float beta_min;
} nrb_field_mlp_t;
/* Leading dimension of the per-sample buffers the fused kernels keep: M rounded up to the 128-sample tile. */
int64_t nrb_field_saved_ld(int64_t M);
/* ---- fused field: hash-grid gather + geometry MLP + feature MLP in one kernel, backward with recomputed activations
 * (NeuRADHashEncoding.forward + NeuRADField.forward in one launch, neurad_encoding.py:152-189, neurad_field.py:128-152).
 * Forward: pass EITHER `grid` with the contracted sample means xyz [M,3] and stds std [M] (or NULL) from
 * nrb_frustum_gaussians - the 32 hash features (num_levels * features_per_level == 32, 2 or 4 features per level) are
 * gathered inside the kernel and never written - OR the hash features x [M,32] (grid == NULL; scenes with actors).
 * x and sh [N_rays,16] (the SH basis of each ray's direction; row m belongs to ray m / samples_per_ray) are fp32, as are
 * the outputs feature [M,32], sdf [M], alpha [M]; products are evaluated as 3xTF32 with fp32 accumulation.  For training pass `saved`: ximg receives the bf16 hi / mid operand image of the hash
 * features (nrb_field_fused_image_bytes(M) bytes: 16 KB per 128-sample tile) and masks [3][ld] one bit per ReLU unit of
 * the three hidden layers, ld = nrb_field_saved_ld(M).  Nothing else is kept: the backward recomputes the activations. */
typedef struct {
  void* ximg;
  uint32_t* masks;
  int64_t ld;
} nrb_field_fused_saved_t;
/* Dynamic actors (NeuRADHashEncoding's actor branch on the torch path: one 3-D grid per actor,
 * neurad_encoding.py:112-119,295-307).  tables[i] = actor_grids.i.hash_table [4 * 2^log2_hashmap_size, 4]; scalings = the
 * four level resolutions.  The per-sample assignment comes from nrb_actor_assign: grid_id [M] (-1 = static world), pos
 * [M,3] in the grid's unit cube, std [M], dirs [M,3] (view direction in the actor frame).  Samples with grid_id >= 0 take
 * their 16 features from that grid (zero-padded to 32, neurad_encoding.py:181-187) and the SH basis of dirs.
 * num_grids is 1..NRB_MAX_ACTORS (256); only tables[0 .. num_grids-1] are read.  Every entry point that takes actor grids
 * returns NRB_ERR_UNSUPPORTED for more, before any launch.  The struct is passed to the kernels by value as part of their
 * parameters (two such pointer arrays, 4 KB, in the proposal backward), which CUDA >= 12.1 allows on sm_100. */
typedef struct {
  const float* tables[NRB_MAX_ACTORS];
  float scalings[NRB_MAX_LEVELS];
  int32_t num_levels;         /* 4 */
  int32_t features_per_level; /* 4 */
  int32_t log2_hashmap_size;
  int32_t num_grids;
} nrb_actor_grids_t;
typedef struct {
  const int32_t* grid_id;
  const float* pos;
  const float* std;
  const float* dirs;
} nrb_actor_samples_t;
int64_t nrb_field_fused_image_bytes(int64_t M);
int nrb_field_fused_fwd(const nrb_field_mlp_t* mlp, const nrb_grid_t* grid, const float* xyz, const float* std,
                        const float* x, const float* sh, int32_t samples_per_ray, int64_t M, float* feature, float* sdf,
                        float* alpha, const nrb_field_fused_saved_t* saved, const nrb_actor_grids_t* actor_grids,
                        const nrb_actor_samples_t* actor_samples, nrb_stream_t stream);
/* Backward.  The gradient of the feature output is EITHER dfeature [M,32] OR - with the compositor folded in
 * (sum_s w f, models/neuradar.py:509) - its factors dfeat_ray [rays,32] and weights [M]: dfeature[m] = weights[m] *
 * dfeat_ray[m / samples_per_ray].  dsdf / dalpha [M] are optional.  dximg (optional) receives the gradient with
 * respect to the hash features as a tile image: float4 element (tile, chunk c of 4 features, sample r of the tile) at
 * [(tile * 8 + c) * 128 + r] (nrb_field_fused_image_bytes(M) * 1 bytes); nrb_hash_bwd_image scatters it into the table.
 * Parameter gradients (dweights[i] / dbiases[i] shaped like the parameters, each optional) are ACCUMULATED; dbeta [1] is the gradient with respect to
 * beta itself (the sign of beta is applied inside). */
typedef struct {
  nrb_field_fused_saved_t saved;
  const float* sh;
  const float* sdf;
  const float* alpha;
  const float* dfeature;
  const float* dfeat_ray;
  const float* weights;
  const float* dsdf;
  const float* dalpha;
  const int32_t* actor_grid_id; /* optional, with actor_dirs: the per-sample assignment of the forward */
  const float* actor_dirs;
} nrb_field_fused_bwd_in_t;
typedef struct {
  float* dximg;
  float* dweights[5];
  float* dbiases[5];
  float* dbeta;
} nrb_field_fused_bwd_out_t;
int nrb_field_fused_bwd(const nrb_field_mlp_t* mlp, const nrb_field_fused_bwd_in_t* in,
                        const nrb_field_fused_bwd_out_t* out, int32_t samples_per_ray, int64_t M, nrb_stream_t stream);
/* nrb_hash_bwd for a data gradient in the tile-image layout above (32 features per sample); samples whose
 * actor_grid_id (optional) is >= 0 are skipped: their features came from an actor grid. */
int nrb_hash_bwd_image(const nrb_grid_t* grid, const float* x, const float* std, const float* dyimg, float* dtable,
                       const int32_t* actor_grid_id, int64_t M, void* workspace, int64_t workspace_bytes,
                       nrb_stream_t stream);
/* ---- dynamic actors as kernels (SURVEY.md 8a H8, 8f next-3; neurad_encoding.py:176-275) ----
 * Per sample of (rays, iv): exact box test against every valid actor of the ray - world2boxes [N,A,3,4] row-major (the
 * inverse of DynamicActors.get_boxes2world, dynamic_actors.py:183-197), valid [N,A] uint8, bounds [A,3] half extents -
 * then the box-frame gaussian contracted with actor_scale, the rotated and normalised view direction, and the optional
 * per-ray mirror flip [N] (+1 / -1, training).  Outputs as nrb_actor_samples_t plus the optional actor_index [M] (index
 * into the ray's actor list).  No compaction, no host synchronisation. */
int nrb_actor_assign(const nrb_rays_t* rays, const nrb_intervals_t* iv, const float* world2boxes, const uint8_t* valid,
                     const float* bounds, const int32_t* actor_to_id, int32_t num_actors, const float* flip,
                     float actor_scale, int32_t* grid_id, float* pos, float* std, float* dirs, int32_t* actor_index,
                     nrb_stream_t stream);
/* Scatter of the actor samples' feature gradient (tile image, features 0..15) into dtables[grid] (accumulated); dpos
 * [M,3] (optional) receives the gradient with respect to pos. */
int nrb_actor_scatter(const nrb_actor_grids_t* grids, float* const* dtables, const nrb_actor_samples_t* samples,
                      const float* dyimg, float* dpos, int64_t M, nrb_stream_t stream);
/* Gradient of the actor samples' features with respect to the world-to-box poses, for trained actor trajectories
 * (NeuRADHashEncoding keeps grad mode for them, neurad_encoding.py:176-229; the box-frame point is
 * transform_points_pairwise, cameras/lidars.py:507-519).  Inputs are those of the nrb_actor_assign call that produced
 * `samples` - rays, iv, world2boxes [N,A,3,4], num_actors, flip [N] or NULL, actor_scale - plus its actor_index [M]
 * output (M = N * iv->num_samples), the actor grids and dyimg, the tile image of d loss / d feature that
 * nrb_actor_scatter reads.  dworld2boxes [N,A,3,4] += d loss / d world2boxes through the box-frame position, the flip,
 * the contraction (mean and, outside its linear region, std) and the level weights.  No allocation, no synchronisation. */
int nrb_actor_pose_grad(const nrb_rays_t* rays, const nrb_intervals_t* iv, const float* world2boxes, int32_t num_actors,
                        const int32_t* actor_index, const float* flip, float actor_scale, const nrb_actor_grids_t* grids,
                        const nrb_actor_samples_t* samples, const float* dyimg, float* dworld2boxes, nrb_stream_t stream);

/* One linear layer y = x W^T + b (optional ReLU) through the same tcgen05 building blocks (K = 32 or 48,
 * n_out <= 48): the unit test of the descriptor / layout conventions. */
int nrb_tc_linear(const float* x, const float* w, const float* b, int32_t K, int32_t n_out, int32_t relu, int64_t M,
                  float* y, nrb_stream_t stream);

/* ---- all-reduce of the gradient arena over NVLink peer memory (SURVEY.md 8e): DistributedDataParallel's gradient
 * average (pipelines/base_pipeline.py:305-307) as one kernel per rank.  buffer_ptrs[p] / signal_flag_ptrs[p] (host arrays
 * of `world` device addresses): rank p's arena and a 1 KB zero-initialised flag area, both mapped into this process
 * (symmetric memory).  In place over floats [offset, offset + n) of every arena: sum over ranks, times `scale`.  Two-shot:
 * each rank reduces its 1/world slice from all arenas and writes the result to all arenas; epoch-stamped flags at system
 * scope order the phases, so the call can be captured in a CUDA graph.  `slot` (0..3) selects an independent flag set
 * (collectives that may be in flight together need different slots); `max_ctas` bounds the SMs the kernel occupies
 * (0: no bound).  multicast_ptr (0: none): the arenas bound to one NVLS multicast object - the reduction then happens in
 * the switch (multimem.ld_reduce / multimem.st), which moves half the bytes.  All ranks must call with the same arguments
 * but `rank`. */
int nrb_peer_all_reduce(const uint64_t* buffer_ptrs, const uint64_t* signal_flag_ptrs, uint64_t multicast_ptr,
                        int32_t rank, int32_t world, int32_t slot, int64_t offset, int64_t n, float scale, int32_t max_ctas, nrb_stream_t stream);

/* ---- radar ray generation (SURVEY.md 8f next-4): Radars._generate_rays_from_fov (cameras/radars.py:268-357) for a list
 * of scans in one launch.  Per radar pose r: radar_to_worlds [R,3,4] and the field-of-view grid min_azimuth / azimuth_step
 * / min_elevation / elevation_step [R] (the reference's `min_*` and `radar_*_ray_divergence` buffers).  scan_indices
 * [n_scans] selects poses; ray_offsets [n_scans + 1] are the prefix sums of the rays per scan, n_azimuths x n_elevations
 * with n = len(torch.arange(min, max, step)) (host arithmetic on the static sensor description), rays azimuth-major.
 * Outputs, one row per ray: origins / directions [N,3], pixel_area [N] = (azimuth_step / 5)(elevation_step / 5),
 * directions_spher [N,2] = (azimuth, elevation), directions_norm [N], ray_scan [N] = the pose index of the ray
 * (camera_indices / the index the reference gathers times and metadata with). */
int nrb_radar_rays(const float* radar_to_worlds, const float* min_azimuth, const float* azimuth_step,
                   const float* min_elevation, const float* elevation_step, const int64_t* scan_indices,
                   const int64_t* ray_offsets, const int32_t* n_elevations, int32_t n_scans, int64_t total_rays,
                   float* origins, float* directions, float* pixel_area, float* directions_spher,
                   float* directions_norm, int64_t* ray_scan, nrb_stream_t stream);

/* ---- degree-4 real spherical harmonics of (d+1)/2: SHEncoding.pytorch_fwd on get_normalized_directions
 * (encodings.py:797-805, utils/math.py:31-94, fields/base_field.py:136-142).  dirs [M,3] -> out [M,16]. */
int nrb_sh16(const float* dirs, float* out, int64_t M, int32_t normalize_to_unit_cube, nrb_stream_t stream);

/* ---- samplers ----
 * SpacedSampler/PowerSampler.generate_ray_samples (ray_samplers.py:80-132).  base_bins [S+1] = linspace(0,1,S+1);
 * jitter is the torch.rand draw: [N] (jitter_per_bin=0, single_jitter) or [N, S+1] (jitter_per_bin=1), or NULL in
 * eval mode.  Outputs: spacing bins sbins [N, S+1] and euclidean bins ebins [N, S+1]. */
int nrb_spaced_bins(const nrb_rays_t* rays, nrb_spacing_t spacing, const float* base_bins, const float* jitter,
                    int32_t jitter_per_bin, int32_t S, float* sbins, float* ebins, nrb_stream_t stream);
/* PDFSampler.generate_ray_samples with include_original=False (ray_samplers.py:280-376): inverse-CDF importance
 * sampling of S_out+1 new bin edges from S_in weighted bins.  weights [N, S_in]; sbins_in [N, S_in+1];
 * u_base [S_out+1] = linspace(0, 1-1/nb, nb); jitter [N] (training, single_jitter) or NULL (eval: +1/(2nb)).
 * Outputs sbins_out / ebins_out [N, S_out+1]; optional inds [N, S_out+1] int64 (= torch.searchsorted(cdf, u,
 * side="right"), ray_samplers.py:349) and cdf [N, S_in+1] for stage-level parity checks. */
int nrb_pdf_sample(const nrb_rays_t* rays, nrb_spacing_t spacing, const float* weights, const float* sbins_in,
                   int32_t S_in, const float* u_base, const float* jitter, int32_t S_out, float histogram_padding,
                   float eps, float* sbins_out, float* ebins_out, int64_t* inds, float* cdf, nrb_stream_t stream);

/* ---- compositing ----
 * RaySamples.get_weights (cameras/rays.py:188-210): weights [N,S] from densities [N,S], deltas = ends - starts. */
int nrb_density_weights_fwd(const float* densities, const nrb_intervals_t* iv, int64_t N, float* weights,
                            nrb_stream_t stream);
int nrb_density_weights_bwd(const float* densities, const nrb_intervals_t* iv, const float* dweights, int64_t N,
                            float* ddensities, nrb_stream_t stream);
/* Alpha compositing tail of NeuRadarModel.get_nff_outputs (models/neuradar.py:504-517): replaces
 * nerfacc.render_weight_from_alpha (:1016), AccumulationRenderer, FeatureRenderer (renderers.py:59-90,322-350)
 * and render_depth_simple (models/neurad.py:721-728).
 *   T_i = prod_{j<i}(1 - alpha_j + trans_eps); w_i = alpha_i T_i; acc = sum w;
 *   sky_sample != 0: w_{S-1} += 1 - acc before the feature sum, and depth excludes sample S-1;
 *   features[N,C] = sum_s w f; depth[N] = sum_s w (start+end)/2.
 * alphas [N,S], feats [N,S,C] (C multiple of 4, <= 64), iv the sample intervals; outputs weights [N,S] (after the sky
 * fix-up), features [N,C], depth [N], accumulation [N], transmittance [N,S] (T_i); each output may be NULL.
 * trans_eps = 0 (nerfacc) or 1e-7 (cameras/rays.py:242). */
int nrb_alpha_composite_fwd(const float* alphas, const float* feats, const nrb_intervals_t* iv, int64_t N, int32_t C,
                            float trans_eps, int32_t sky_sample, float* weights, float* features, float* depth,
                            float* accumulation, float* transmittance, nrb_stream_t stream);
/* Backward: upstream dweights [N,S] (may be NULL), dfeatures [N,C], ddepth [N], daccumulation [N] (each may be
 * NULL) -> dalphas [N,S], dfeats [N,S,C]. */
int nrb_alpha_composite_bwd(const float* alphas, const float* feats, const nrb_intervals_t* iv, int64_t N, int32_t C,
                            float trans_eps, int32_t sky_sample, const float* dweights, const float* dfeatures,
                            const float* ddepth, const float* daccumulation, float* dalphas, float* dfeats,
                            nrb_stream_t stream);

/* render_depth_simple for given weights (models/neurad.py:721-728; `renderer_depth(prop_w, prop_rs)` of the proposal rounds,
 * models/neuradar.py:528): depth [N] = sum_s weights[n,s] (start + end) / 2, and d depth / d weights. */
int nrb_weighted_depth_fwd(const float* weights, const nrb_intervals_t* iv, int64_t N, float* depth, nrb_stream_t stream);
int nrb_weighted_depth_bwd(const nrb_intervals_t* iv, const float* ddepth, int64_t N, float* dweights, nrb_stream_t stream);
/* nerfacc.accumulate_along_rays on dense samples (call sites models/neurad.py:728, renderers.py:85,349,412):
 * out [N,C] = sum_s weights[N,S] * values[N,S,C]; values == NULL gives out [N] = sum_s weights. */
int nrb_accumulate_fwd(const float* weights, const float* values, int64_t N, int32_t S, int32_t C, float* out,
                       nrb_stream_t stream);
int nrb_accumulate_bwd(const float* weights, const float* values, const float* dout, int64_t N, int32_t S, int32_t C,
                       float* dweights, float* dvalues, nrb_stream_t stream);

/* ---- per-ray tail: point heads and lidar carving terms (SURVEY.md 8a C6, appendix A7) ----
 * Point heads: rendered depth [N] -> one 3-D point per ray.  Rays flagged in is_radar (uint8 [N], may be NULL) use
 * the spherical direction directions_spher [N,2] = (phi, theta): p = depth (cos phi cos theta, sin phi cos theta,
 * sin theta) (models/neuradar.py:463-473,1025-1029); all others p = o + d depth (models/ad_model.py:105), optionally
 * mapped by world2sensor [3,4] row-major (the lidar frame, ad_model.py:103-108).  Backward: ddepth [N] from dpoints. */
int nrb_point_heads_fwd(const float* origins, const float* directions, const float* depth, const uint8_t* is_radar,
                        const float* directions_spher, const float* world2sensor, float* points, int64_t N,
                        nrb_stream_t stream);
int nrb_point_heads_bwd(const float* directions, const uint8_t* is_radar, const float* directions_spher,
                        const float* world2sensor, const float* dpoints, float* ddepth, int64_t N, nrb_stream_t stream);
/* NeuRadarModel._compute_is_close_to_lidar (models/neuradar.py:971-994) and the proposal carving loss (:527-531):
 * is_close [N,S] (uint8, optional) = for lidar rays |directions_norm - (start+end)/2| < carving_epsilon, or with
 * did_return (uint8 [N], optional): (did_return & close) | (~did_return & mid < non_return_lidar_distance); false for
 * other rays.  With weights [N,S] and dloss == NULL: out [N,S] = (w * (is_lidar & ~is_close))^2 (sum it for the loss);
 * with dloss [1]: out = d loss / d weights = 2 w mask dloss. */
int nrb_lidar_carving(const nrb_intervals_t* iv, int64_t N, const uint8_t* is_lidar, const float* directions_norm,
                      const uint8_t* did_return, float carving_epsilon, float non_return_lidar_distance,
                      const float* weights, const float* dloss, uint8_t* is_close, float* out, nrb_stream_t stream);

/* ---- per-ray training losses on the path's outputs (SURVEY.md 8f next-1) ----
 * MipNeRF-360 distortion loss (nerfstudio/model_components/losses.py:137-156, called on the final level at
 * models/neurad.py via ray_samples.spacing bins): sbins [N,S+1] (row stride bin_stride floats), weights [N,S] ->
 * loss_per_ray [N]; grad_factor [N,S] (may be NULL) = d loss_per_ray / d weights. */
int nrb_distortion_loss(const float* sbins, int64_t bin_stride, const float* weights, int64_t N, int32_t S,
                        float* loss_per_ray, float* grad_factor, nrb_stream_t stream);
/* ZipNeRF anti-aliased interlevel loss of ONE proposal round (losses.py:620-705): the final level's spacing bins
 * c [N,Sc+1] and weights w [N,Sc] (constants; the remaining accumulation is added to the last sample inside) are
 * blurred with a box of half-width pulse_width and resampled at the proposal's bins cp [N,Sp+1]; wp [N,Sp] are the
 * proposal's weights.  loss_per_ray [N]; grad_factor [N,Sp] (may be NULL) = d loss_per_ray / d wp. */
int nrb_interlevel_loss(const float* c_bins, int64_t c_stride, const float* w, int32_t Sc, const float* cp_bins,
                        int64_t cp_stride, const float* wp, int32_t Sp, float pulse_width, int64_t N,
                        float* loss_per_ray, float* grad_factor, nrb_stream_t stream);

/* ---- optimiser step (SURVEY.md 8f next-2) ----
 * torch.optim.Adam / AdamW exactly as the reference configures them for the "hashgrids" (Adam, lr 1e-2, eps 1e-15) and
 * "fields" (AdamW, weight_decay 1e-7) parameter groups (nerfstudio/configs/method_configs.py:393-400) and steps them
 * through GradScaler (nerfstudio/engine/optimizers.py:159-181): one pass over a flat fp32 segment that reads p, g, m, v
 * and writes p, m, v.  The gradient is first multiplied by grad_mult (e.g. 1 / world_size for the data-parallel
 * average) and divided by *loss_scale when that device scalar is given (GradScaler.unscale_); when *found_inf != 0
 * the update is skipped (GradScaler.step), zero_grad still applies; torch does not count a skipped step, so when
 * `skipped_steps` (device float, starts at 0) is given it is incremented on a skip and the bias corrections use
 * cfg->step - *skipped_steps: the caller keeps counting every call and never synchronises. */
typedef struct {
  double lr, beta1, beta2, eps, weight_decay; /* the Python floats torch.optim receives; constants such as 1 - beta2
                                                 and lr / (1 - beta1^step) are formed in double and rounded once */
  int32_t decoupled_weight_decay; /* 0: Adam (L2 term added to the gradient), 1: AdamW (p *= 1 - lr * wd) */
  int32_t step;                   /* 1-based count of this update (bias corrections 1 - beta^step) */
  float grad_mult;
  int32_t zero_grad;              /* also write zeros to g (optimizer.zero_grad fused) */
} nrb_adam_t;
int nrb_adam_step(float* p, float* g, float* m, float* v, int64_t n, const nrb_adam_t* cfg, const float* loss_scale,
                  const float* found_inf, float* skipped_steps, nrb_stream_t stream);
/* found_inf[0] = 1.0f if any of the n gradients is inf or nan (GradScaler._unscale_grads_'s check); never cleared. */
int nrb_grad_check(const float* g, int64_t n, float* found_inf, nrb_stream_t stream);

/* ---- fused proposal round: NeuRADProposalField.get_density + RaySamples.get_weights
 * (fields/neurad_field.py:208-213, cameras/rays.py:188-210) in one kernel, one warp per ray:
 * gaussians -> contraction -> hash encode -> level weights -> Linear(L*F, 1, bias=False) -> trunc_exp -> weights.
 * decoder_w [L*F].  Outputs: density [N,S], weights [N,S]; when `saved_feats` [N,S,L*F] and `saved_pre` [N,S]
 * are non-NULL the rescaled features and the pre-activation are kept for the backward pass.  Dynamic actors (optional,
 * both NULL otherwise): samples with actor_samples->grid_id >= 0 read the 4-level grid of their actor (same features per
 * level as the static grid; features beyond the actor grid's are zero), see nrb_actor_assign. */
int nrb_proposal_fwd(const nrb_rays_t* rays, const nrb_grid_t* grid, const float* decoder_w, float static_scale,
                     const nrb_intervals_t* iv, float* density, float* weights, float* saved_feats, float* saved_pre,
                     const nrb_actor_grids_t* actor_grids, const nrb_actor_samples_t* actor_samples, nrb_stream_t stream);
/* Backward of the fused round given dweights [N,S] and/or ddensity [N,S] (either may be NULL):
 * dtable += ..., ddecoder_w [L*F] += ...; workspace as for nrb_hash_bwd (nrb_hash_bwd_workspace_bytes(grid, N*S)). */
int nrb_proposal_bwd(const nrb_rays_t* rays, const nrb_grid_t* grid, const float* decoder_w, float static_scale,
                     const nrb_intervals_t* iv, const float* saved_feats, const float* saved_pre,
                     const float* dweights, const float* ddensity, float* dtable, float* ddecoder_w,
                     void* workspace, int64_t workspace_bytes, const nrb_actor_grids_t* actor_grids,
                     const nrb_actor_samples_t* actor_samples, float* const* actor_dtables, nrb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NEURADAR_B200_H */
