// Fused proposal round: sample gaussians -> contraction -> hash encode -> anti-alias level weights -> linear decoder
// -> trunc_exp -> density-to-weights scan, one warp per ray, nothing but the per-sample results leaves the SM.
// Semantics: NeuRADProposalField.get_density (nerfstudio/fields/neurad_field.py:208-213) followed by
// RaySamples.get_weights (nerfstudio/cameras/rays.py:188-210); trunc_exp backward clamps the exponent to +-15
// (nerfstudio/field_components/activations.py:28-41).
#include "actor_grid.cuh"
#include "common.cuh"
#include "hash_bwd_plan.cuh"

namespace nrb {

constexpr int kPropWarps = 4;
constexpr int kMaxChunks = NRB_MAX_SAMPLES / 32;

struct PropGrid {
  const float* table;
  float scalings[NRB_MAX_LEVELS];
  const float* decoder;  // [L*F] device pointer (density_decoder.weight)
  int num_levels;
  int log2_size;
  // dynamic actors (optional): samples with agid >= 0 read the 4-level grid of their actor instead, features beyond
  // 4 * F are zero (neurad_encoding.py:181-187); apos / astd come from nrb_actor_assign
  const int32_t* agid;
  const float* apos;
  const float* astd;
  ActorGridsDev ag;
  float* adtables[NRB_MAX_ACTORS];  // backward: gradient tables of the actor grids
};

template <int F, bool kSave>
__global__ void __launch_bounds__(kPropWarps * 32) proposal_fwd_kernel(
    const __grid_constant__ PropGrid g, const float* __restrict__ origins, const float* __restrict__ directions,
    const float* __restrict__ pixel_area, float scale, nrb_intervals_t iv, int64_t N,
    float* __restrict__ density, float* __restrict__ weights, float* __restrict__ saved_feats,
    float* __restrict__ saved_pre) {
  __shared__ float s_dec[NRB_MAX_LEVELS * 4];
  const int lane = threadIdx.x & 31;
  const int S = iv.num_samples;
  const int LF = g.num_levels * F;
  if (threadIdx.x < NRB_MAX_LEVELS * 4) s_dec[threadIdx.x] = threadIdx.x < LF ? g.decoder[threadIdx.x] : 0.0f;
  __syncthreads();
  const int64_t n = static_cast<int64_t>(blockIdx.x) * kPropWarps + (threadIdx.x >> 5);
  if (n >= N) return;
  const float ox = origins[3 * n], oy = origins[3 * n + 1], oz = origins[3 * n + 2];
  const float dx = directions[3 * n], dy = directions[3 * n + 1], dz = directions[3 * n + 2];
  const float pa = pixel_area[n];
  const float* st = iv.starts + n * iv.row_stride;
  const float* en = iv.ends + n * iv.row_stride;
  const uint32_t mask = (1u << g.log2_size) - 1u;
  float carry = 0.0f;
  for (int base = 0; base < S; base += 32) {
    const int i = base + lane;
    const bool ok = i < S;
    float dd = 0.0f, dens = 0.0f;
    if (ok) {
      const float start = st[i], end = en[i];
      const Gaussian q = sample_gaussian(ox, oy, oz, dx, dy, dz, pa, start, end, scale);
      float pre = 0.0f;
      const int agid = g.agid != nullptr ? g.agid[n * S + i] : -1;
      if (agid >= 0) {  // inside an actor box: that actor's grid, zero-padded
        const float ax = g.apos[3 * (n * S + i)], ay = g.apos[3 * (n * S + i) + 1], az = g.apos[3 * (n * S + i) + 2];
        const float asd = g.astd[n * S + i];
        const uint32_t amask = (1u << g.ag.log2_size) - 1u;
        for (int l = 0; l < g.num_levels; ++l) {
          float v[F];
#pragma unroll
          for (int j = 0; j < F; ++j) v[j] = 0.0f;
          float lw = 0.0f;
          if (l < kActorLevels) {
            const float scal = g.ag.scalings[l];
            const Cell c = locate_cell(ax, ay, az, scal, amask);
            interpolate<F>(g.ag.tables[agid] + (static_cast<size_t>(l) << g.ag.log2_size) * F, c, v);
            lw = level_weight(scal, asd);
          }
#pragma unroll
          for (int j = 0; j < F; ++j) {
            const float f = v[j] * lw;
            pre = fmaf(f, s_dec[l * F + j], pre);
            if constexpr (kSave) saved_feats[(n * S + i) * LF + l * F + j] = f;
          }
        }
      } else {
        for (int l = 0; l < g.num_levels; ++l) {
          const float scal = g.scalings[l];
          const Cell c = locate_cell(q.x, q.y, q.z, scal, mask);
          float v[F];
          interpolate<F>(g.table + (static_cast<size_t>(l) << g.log2_size) * F, c, v);
          const float lw = level_weight(scal, q.std);
#pragma unroll
          for (int j = 0; j < F; ++j) {
            const float f = v[j] * lw;
            pre = fmaf(f, s_dec[l * F + j], pre);
            if constexpr (kSave) saved_feats[(n * S + i) * LF + l * F + j] = f;
          }
        }
      }
      dens = expf(pre);
      if constexpr (kSave) saved_pre[n * S + i] = pre;
      if (density != nullptr) density[n * S + i] = dens;
      dd = mul(sub(end, start), dens);
    }
    const float incl = warp_inclusive_sum(dd, lane);
    float excl = __shfl_up_sync(kFull, incl, 1);
    if (lane == 0) excl = 0.0f;
    const float alpha = 1.0f - expf(-dd);
    const float trans = expf(-(carry + excl));
    if (ok) weights[n * S + i] = nan_to_num(alpha * trans);
    carry += __shfl_sync(kFull, incl, 31);
  }
}

// Two phases.  (1) Warp per ray: the forward weight scan is recomputed from the saved pre-activations and the reverse
// scan turns d weights into d density; kChunks = ceil(S / 32) rounded up to 2 / 4 / 8, because the per-chunk state of
// the two scans lives in registers and a kernel instantiated for 8 chunks carries 40 of them for nothing at S <= 64.
// Each sample's d pre (after trunc_exp) goes to shared memory.  (2) The block's rays_per_block * S samples, ray-major,
// are cut into consecutive chunks of 32 and every warp scatters a contiguous range of them: a chunk may cross a ray
// boundary, so S = 48 runs no idle lanes (one warp per ray would run a second chunk of 16).  Run merging stays exact
// across the boundary: runs are formed on cell coordinates only, and two samples in one cell update the same rows
// whichever ray they belong to.
template <int F, int kChunks>
__global__ void __launch_bounds__(kPropWarps * 32) proposal_bwd_kernel(
    const __grid_constant__ PropGrid g, const __grid_constant__ BwdPlan plan, const float* __restrict__ origins, const float* __restrict__ directions,
    const float* __restrict__ pixel_area, float scale, nrb_intervals_t iv, int64_t N, int rays_per_block,
    const float* __restrict__ saved_feats, const float* __restrict__ saved_pre, const float* __restrict__ dweights,
    const float* __restrict__ ddensity, float* __restrict__ dtable, float* __restrict__ ddecoder) {
  extern __shared__ float s_gpre[];  // [rays_per_block * S]
  __shared__ float s_ddec[NRB_MAX_LEVELS * 4];
  __shared__ float s_dec[NRB_MAX_LEVELS * 4];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int S = iv.num_samples;
  const int LF = g.num_levels * F;
  if (threadIdx.x < NRB_MAX_LEVELS * 4) {
    s_ddec[threadIdx.x] = 0.0f;
    s_dec[threadIdx.x] = threadIdx.x < LF ? g.decoder[threadIdx.x] : 0.0f;
  }
  const int64_t n0 = static_cast<int64_t>(blockIdx.x) * rays_per_block;
  const int rays = static_cast<int>(min(static_cast<int64_t>(rays_per_block), N - n0));
#pragma unroll 1
  for (int r = warp; r < rays; r += kPropWarps) {
    const int64_t n = n0 + r;
    const float* st = iv.starts + n * iv.row_stride;
    const float* en = iv.ends + n * iv.row_stride;
    // forward recompute of the weight scan from the saved pre-activations
    float delta[kChunks], dd[kChunks], trans[kChunks], pre[kChunks];
    float carry = 0.0f;
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
      if (c * 32 < S) {
        const int i = c * 32 + lane;
        const bool ok = i < S;
        pre[c] = ok ? saved_pre[n * S + i] : 0.0f;
        delta[c] = ok ? sub(en[i], st[i]) : 0.0f;
        dd[c] = ok ? mul(delta[c], expf(pre[c])) : 0.0f;
        const float incl = warp_inclusive_sum(dd[c], lane);
        float excl = __shfl_up_sync(kFull, incl, 1);
        if (lane == 0) excl = 0.0f;
        trans[c] = expf(-(carry + excl));
        carry += __shfl_sync(kFull, incl, 31);
      }
    }
    // d weights -> d density (reverse exclusive scan), see density_weights_bwd_kernel, -> d pre (trunc_exp)
    float suffix = 0.0f;
#pragma unroll
    for (int c = kChunks - 1; c >= 0; --c) {
      if (c * 32 < S) {
        const int i = c * 32 + lane;
        const bool ok = i < S;
        const float e = expf(-dd[c]);
        const float w = (1.0f - e) * trans[c];
        float gwt = (ok && dweights != nullptr) ? dweights[n * S + i] : 0.0f;
        if (isnan(w) || isinf(w)) gwt = 0.0f;
        const float gw = ok ? gwt * w : 0.0f;
        float incl = gw;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float v = __shfl_down_sync(kFull, incl, o);
          if (lane + o < 32) incl += v;
        }
        float excl = __shfl_down_sync(kFull, incl, 1);
        if (lane == 31) excl = 0.0f;
        const float later = suffix + excl;
        if (ok) {
          float gdens = (gwt * trans[c] * e - later) * delta[c];
          if (ddensity != nullptr) gdens += ddensity[n * S + i];
          s_gpre[r * S + i] = gdens * expf(fminf(fmaxf(pre[c], -15.0f), 15.0f));
        }
        suffix += __shfl_sync(kFull, incl, 0);
      }
    }
  }
  __syncthreads();
  // d pre -> decoder and table gradients, over the block's samples in chunks of 32
  const int total = rays * S;
  const int chunks = (total + 31) >> 5;
  const int per_warp = (chunks + kPropWarps - 1) / kPropWarps;
  const int c_end = min(chunks, (warp + 1) * per_warp);
  const unsigned spread = static_cast<unsigned>(blockIdx.x * kPropWarps + warp);
  const uint32_t mask = (1u << g.log2_size) - 1u;
#pragma unroll 1
  for (int c = warp * per_warp; c < c_end; ++c) {  // warp-uniform: all lanes take part in the run merging below
    const int k = c * 32 + lane;
    const bool act = k < total;
    const int kc = act ? k : total - 1;
    const int r = kc / S;
    const int i = kc - r * S;
    const int64_t n = n0 + r;
    const int64_t m = n0 * S + kc;  // == n * S + i
    const float gpre = act ? s_gpre[kc] : 0.0f;
    const Gaussian q = sample_gaussian(origins[3 * n], origins[3 * n + 1], origins[3 * n + 2], directions[3 * n],
                                       directions[3 * n + 1], directions[3 * n + 2], pixel_area[n],
                                       iv.starts[n * iv.row_stride + i], iv.ends[n * iv.row_stride + i], scale);
    const float* sf = saved_feats + m * LF;
    const int agid = g.agid != nullptr ? g.agid[m] : -1;
    if (act && agid >= 0) {  // the sample's gradient goes to its actor's table (plain reductions: ~10 % of the samples)
      const float ax = g.apos[3 * m], ay = g.apos[3 * m + 1], az = g.apos[3 * m + 2];
      const float asd = g.astd[m];
      const uint32_t amask = (1u << g.ag.log2_size) - 1u;
#pragma unroll
      for (int l = 0; l < kActorLevels; ++l) {
        const float scal = g.ag.scalings[l];
        const Cell cell = locate_cell(ax, ay, az, scal, amask);
        const float lw = level_weight(scal, asd);
        float gr[F];
#pragma unroll
        for (int j = 0; j < F; ++j) gr[j] = gpre * s_dec[l * F + j] * lw;
        float w8[8];
        corner_weights(cell, w8);
        float* dt = g.adtables[agid] + (static_cast<size_t>(l) << g.ag.log2_size) * F;
#pragma unroll
        for (int k8 = 0; k8 < 8; ++k8) {
          float v[F];
#pragma unroll
          for (int j = 0; j < F; ++j) v[j] = gr[j] * w8[k8];
          scatter_row<F>(dt, cell.row[k8], v);
        }
      }
    }
    const bool act_static = act && agid < 0;
    // A real loop over the levels: unrolled 16 x (with the chunks: up to 128 copies of the merge-and-scatter body)
    // the kernel was 150 K instructions, far beyond the instruction cache.
#pragma unroll 1
    for (int l = 0; l < g.num_levels; ++l) {
      const float scal = g.scalings[l];
      const Cell cell = locate_cell(q.x, q.y, q.z, scal, mask);
      const float lw = level_weight(scal, q.std);
      float gr[F];
#pragma unroll
      for (int j = 0; j < F; ++j) {
        const float dd_lj = warp_sum(gpre * sf[l * F + j]);  // decoder gradient of this chunk's 32 samples
        if (lane == 0) atomicAdd(&s_ddec[l * F + j], dd_lj);
        gr[j] = gpre * s_dec[l * F + j] * lw;
      }
      float w8[8];
      corner_weights(cell, w8);
      // runs of adjacent samples that share a cell are summed before scattering (hash_bwd_plan.cuh)
      float v[8][F];
#pragma unroll
      for (int k8 = 0; k8 < 8; ++k8)
#pragma unroll
        for (int j = 0; j < F; ++j) v[k8][j] = w8[k8] * gr[j];
      merge_runs_and_scatter<F>(plan, l, g.log2_size, q.x, q.y, q.z, scal, cell, v, act_static, lane, dtable, spread);
    }
  }
  __syncthreads();
  if (threadIdx.x < LF && ddecoder != nullptr) atomicAdd(ddecoder + threadIdx.x, s_ddec[threadIdx.x]);
}

static PropGrid make_prop_grid(const nrb_grid_t* grid, const float* decoder, const nrb_actor_grids_t* agrids = nullptr,
                               const nrb_actor_samples_t* asamples = nullptr, float* const* adtables = nullptr) {
  PropGrid out{};
  if (agrids != nullptr) {
    out.ag = to_dev(agrids);
    out.agid = asamples->grid_id, out.apos = asamples->pos, out.astd = asamples->std;
    for (int i = 0; i < agrids->num_grids; ++i) out.adtables[i] = adtables != nullptr ? adtables[i] : nullptr;
  }
  out.table = grid->table;
  for (int i = 0; i < NRB_MAX_LEVELS; ++i) out.scalings[i] = grid->scalings[i];
  out.decoder = decoder;
  out.num_levels = grid->num_levels;
  out.log2_size = grid->log2_hashmap_size;
  return out;
}

static int check_proposal(const char* who, const nrb_rays_t* rays, const nrb_grid_t* grid, const float* decoder_w,
                          float scale, const nrb_intervals_t* iv) {
  if (int rc = check_rays(rays)) return rc;
  if (int rc = check_grid(grid)) return rc;
  if (int rc = check_intervals(who, iv)) return rc;
  NRB_REQUIRE(decoder_w != nullptr, NRB_ERR_BAD_ARG, "%s: null pointer", who);
  NRB_REQUIRE(scale > 0.f, NRB_ERR_BAD_ARG, "%s: static_scale must be positive", who);
  return NRB_OK;
}

}  // namespace nrb

using namespace nrb;

static int check_prop_actors(const char* who, const nrb_grid_t* grid, const nrb_actor_grids_t* agrids,
                             const nrb_actor_samples_t* asamples) {
  if (agrids == nullptr) return NRB_OK;
  NRB_REQUIRE(agrids->num_grids >= 1 && agrids->num_grids <= NRB_MAX_ACTORS && agrids->num_levels == kActorLevels &&
                  agrids->features_per_level == grid->features_per_level && grid->num_levels >= kActorLevels,
              NRB_ERR_UNSUPPORTED, "%s: actor grids must have 4 levels and the static grid's features per level", who);
  NRB_REQUIRE(asamples && asamples->grid_id && asamples->pos && asamples->std, NRB_ERR_BAD_ARG, "%s: actor samples missing", who);
  for (int i = 0; i < agrids->num_grids; ++i) NRB_REQUIRE(agrids->tables[i] != nullptr, NRB_ERR_BAD_ARG, "%s: actor table %d", who, i);
  return NRB_OK;
}

extern "C" int nrb_proposal_fwd(const nrb_rays_t* rays, const nrb_grid_t* grid, const float* decoder_w,
                                float static_scale, const nrb_intervals_t* iv, float* density, float* weights,
                                float* saved_feats, float* saved_pre, const nrb_actor_grids_t* actor_grids,
                                const nrb_actor_samples_t* actor_samples, nrb_stream_t stream) {
  if (int rc = check_proposal("nrb_proposal_fwd", rays, grid, decoder_w, static_scale, iv)) return rc;
  if (int rc = check_prop_actors("nrb_proposal_fwd", grid, actor_grids, actor_samples)) return rc;
  NRB_REQUIRE(weights != nullptr, NRB_ERR_BAD_ARG, "nrb_proposal_fwd: weights is null");
  NRB_REQUIRE((saved_feats == nullptr) == (saved_pre == nullptr), NRB_ERR_BAD_ARG,
              "nrb_proposal_fwd: saved_feats and saved_pre must be given together");
  const int64_t N = rays->num_rays;
  if (N == 0) return NRB_OK;
  const PropGrid g = make_prop_grid(grid, decoder_w, actor_grids, actor_samples);
  const unsigned blocks = blocks_for(N, kPropWarps);
  auto s = static_cast<cudaStream_t>(stream);
  const bool save = saved_feats != nullptr;
#define NRB_LAUNCH(F, SAVE)                                                                                          \
  proposal_fwd_kernel<F, SAVE><<<blocks, kPropWarps * 32, 0, s>>>(g, rays->origins, rays->directions,               \
                                                                  rays->pixel_area, static_scale, *iv, N,           \
                                                                  density, weights, saved_feats, saved_pre)
  switch (grid->features_per_level) {
    case 1: if (save) NRB_LAUNCH(1, true); else NRB_LAUNCH(1, false); break;
    case 2: if (save) NRB_LAUNCH(2, true); else NRB_LAUNCH(2, false); break;
    default: if (save) NRB_LAUNCH(4, true); else NRB_LAUNCH(4, false); break;
  }
#undef NRB_LAUNCH
  return finish_launch("nrb_proposal_fwd");
}

extern "C" int nrb_proposal_bwd(const nrb_rays_t* rays, const nrb_grid_t* grid, const float* decoder_w,
                                float static_scale, const nrb_intervals_t* iv, const float* saved_feats,
                                const float* saved_pre, const float* dweights, const float* ddensity, float* dtable,
                                float* ddecoder_w, void* workspace, int64_t workspace_bytes,
                                const nrb_actor_grids_t* actor_grids, const nrb_actor_samples_t* actor_samples,
                                float* const* actor_dtables, nrb_stream_t stream) {
  if (int rc = check_proposal("nrb_proposal_bwd", rays, grid, decoder_w, static_scale, iv)) return rc;
  if (int rc = check_prop_actors("nrb_proposal_bwd", grid, actor_grids, actor_samples)) return rc;
  NRB_REQUIRE(actor_grids == nullptr || actor_dtables != nullptr, NRB_ERR_BAD_ARG, "nrb_proposal_bwd: actor gradient tables missing");
  NRB_REQUIRE(saved_feats && saved_pre && dtable, NRB_ERR_BAD_ARG, "nrb_proposal_bwd: null pointer");
  NRB_REQUIRE(dweights || ddensity, NRB_ERR_BAD_ARG, "nrb_proposal_bwd: no upstream gradient");
  NRB_REQUIRE(aligned16(dtable), NRB_ERR_ALIGNMENT, "nrb_proposal_bwd: dtable must be 16-byte aligned");
  const int64_t N = rays->num_rays;
  if (N == 0) return NRB_OK;
  const PropGrid g = make_prop_grid(grid, decoder_w, actor_grids, actor_samples, actor_dtables);
  // Rays per block: the scatter phase deals the block's rays * S samples to its warps as chunks of 32, so they are
  // taken as the smallest of 4, 8 and 16 rays for which that is a multiple of 4 x 32 (whole chunks, the same number for
  // every warp): 4 when S % 32 == 0, 8 when S % 16 == 0 (S = 48: 3 chunks per warp), 16 when S % 8 == 0.  Any other S
  // keeps 4 rays and a partly filled last chunk.
  int rays_per_block = kPropWarps;
  while (rays_per_block < 4 * kPropWarps && (rays_per_block * iv->num_samples) % (kPropWarps * 32) != 0) rays_per_block *= 2;
  if ((rays_per_block * iv->num_samples) % (kPropWarps * 32) != 0) rays_per_block = kPropWarps;
  const unsigned blocks = blocks_for(N, rays_per_block);
  const size_t smem = static_cast<size_t>(rays_per_block) * iv->num_samples * sizeof(float);  // at most 16 KB
  auto s = static_cast<cudaStream_t>(stream);
  BwdPlan plan;
  int64_t vertices = 0;
  if (int rc = prepare_bwd_plan(grid, N * iv->num_samples, workspace, workspace_bytes, s, &plan, &vertices)) return rc;
#define NRB_LAUNCH_C(F, CH)                                                                                          \
  proposal_bwd_kernel<F, CH><<<blocks, kPropWarps * 32, smem, s>>>(g, plan, rays->origins, rays->directions,         \
                                                                   rays->pixel_area, static_scale, *iv, N,           \
                                                                   rays_per_block, saved_feats, saved_pre, dweights, \
                                                                   ddensity, dtable, ddecoder_w)
#define NRB_LAUNCH(F)                                   \
  if (iv->num_samples <= 64) {                          \
    NRB_LAUNCH_C(F, 2);                                 \
  } else if (iv->num_samples <= 128) {                  \
    NRB_LAUNCH_C(F, 4);                                 \
  } else {                                              \
    NRB_LAUNCH_C(F, kMaxChunks);                        \
  }
  switch (grid->features_per_level) {
    case 1: NRB_LAUNCH(1); break;
    case 2: NRB_LAUNCH(2); break;
    default: NRB_LAUNCH(4); break;
  }
#undef NRB_LAUNCH
#undef NRB_LAUNCH_C
  launch_fold(grid, plan, dtable, vertices, s);
  return finish_launch("nrb_proposal_bwd");
}
