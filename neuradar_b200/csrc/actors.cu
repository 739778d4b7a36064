// Dynamic actors as kernels (SURVEY.md 8a row H8, 8f next-3): which samples fall into which actor box, their box-frame
// gaussians and view directions, and the scatter of their gradient into the per-actor hash tables.
// Semantics: NeuRADHashEncoding._split_static_vs_actors / _get_actor_indices / actor contraction
// (nerfstudio/field_components/neurad_encoding.py:176-275) with DynamicActors.get_boxes2world
// (nerfstudio/model_components/dynamic_actors.py:183-197) supplying the per-ray poses.
//
// The reference finds the samples in three steps - ray line vs bounding sphere, sample vs sphere, exact box test - with
// three nonzero() round trips; the first two are prefilters of the third (inside the box => inside the sphere => the ray
// line passes the sphere), so one thread per sample simply runs the exact test against every valid actor: 16 actors x
// ~20 flops, no compaction, no host synchronisation.  A sample inside several boxes goes to the highest actor index
// (the reference overwrites in an unspecified order, neurad_encoding.py:187,274; scenes have disjoint boxes).
#include "actor_grid.cuh"
#include "hash_bwd_plan.cuh"

namespace nrb {

__global__ void __launch_bounds__(256) actor_assign_kernel(const float* __restrict__ origins,
                                                           const float* __restrict__ directions,
                                                           const float* __restrict__ pixel_area, nrb_intervals_t iv,
                                                           const float* __restrict__ world2boxes,  // [N,A,3,4]
                                                           const uint8_t* __restrict__ valid,      // [N,A]
                                                           const float* __restrict__ bounds,       // [A,3]
                                                           const int32_t* __restrict__ actor_to_id, int A,
                                                           const float* __restrict__ flip,         // [N] (+1 / -1) or null
                                                           float actor_scale, int32_t* __restrict__ grid_id,
                                                           float* __restrict__ pos, float* __restrict__ std,
                                                           float* __restrict__ dirs, int32_t* __restrict__ actor_index,
                                                           int64_t total) {
  // Per-ray pre-cull (the reference's own first filter, neurad_encoding.py:231-247): an actor can only claim samples of
  // a ray whose line passes its bounding sphere.  The block's 256 consecutive samples belong to a handful of rays; the
  // block first tests every (ray, actor) pair once and leaves a bit set of ceil(A / 32) words per ray in shared memory
  // (sized by the launch from S and A, actor_cull_bytes), and the per-sample loop below runs the exact box test only for
  // the flagged actors (typically none or one).  The sphere contains the box, and the test is evaluated with a margin,
  // so the result is the plain loop's.  Above NRB_MAX_ACTORS the launch passes no shared memory and every sample runs
  // the plain loop.
  extern __shared__ uint32_t s_mask[];  // [rays of the block][words]
  const int S = iv.num_samples;
  const int64_t first = static_cast<int64_t>(blockIdx.x) * blockDim.x;
  const int64_t last = min(first + blockDim.x, total) - 1;
  const int64_t n0 = first / S;
  const int nrays = static_cast<int>(last / S - n0) + 1;
  const bool cull = A <= NRB_MAX_ACTORS;
  const int words = (A + 31) / 32;
  if (cull) {
    for (int i = threadIdx.x; i < nrays * words; i += blockDim.x) s_mask[i] = 0u;
    __syncthreads();
    for (int p = threadIdx.x; p < nrays * A; p += blockDim.x) {
      const int64_t n = n0 + p / A;
      const int a = p % A;
      if (!valid[n * A + a]) continue;
      const float* m = world2boxes + (n * A + a) * 12;
      const float ox = origins[3 * n], oy = origins[3 * n + 1], oz = origins[3 * n + 2];
      const float dx = directions[3 * n], dy = directions[3 * n + 1], dz = directions[3 * n + 2];
      const float px = m[0] * ox + m[1] * oy + m[2] * oz + m[3], py = m[4] * ox + m[5] * oy + m[6] * oz + m[7],
                  pz = m[8] * ox + m[9] * oy + m[10] * oz + m[11];
      const float qx = m[0] * dx + m[1] * dy + m[2] * dz, qy = m[4] * dx + m[5] * dy + m[6] * dz,
                  qz = m[8] * dx + m[9] * dy + m[10] * dz;
      const float cx = py * qz - pz * qy, cy = pz * qx - px * qz, cz = px * qy - py * qx;  // |p x q| = distance * |q|
      const float r2 = bounds[3 * a] * bounds[3 * a] + bounds[3 * a + 1] * bounds[3 * a + 1] + bounds[3 * a + 2] * bounds[3 * a + 2];
      if (cx * cx + cy * cy + cz * cz <= (r2 * 1.01f + 1.0e-6f) * (qx * qx + qy * qy + qz * qz))
        atomicOr(&s_mask[(p / A) * words + a / 32], 1u << (a % 32));
    }
    __syncthreads();
  }
  const int64_t gid = first + threadIdx.x;
  if (gid >= total) return;
  const int64_t n = gid / S;
  const int s = static_cast<int>(gid - n * S);
  const float dx = directions[3 * n], dy = directions[3 * n + 1], dz = directions[3 * n + 2];
  const Gaussian w = world_gaussian(origins[3 * n], origins[3 * n + 1], origins[3 * n + 2], dx, dy, dz, pixel_area[n],
                                    iv.starts[n * iv.row_stride + s], iv.ends[n * iv.row_stride + s]);
  int hit = -1;
  float bx = 0.f, by = 0.f, bz = 0.f;
  auto box_test = [&](int a) {  // ascending a: the highest actor index wins
    if (!valid[n * A + a]) return;
    const float3 b = to_box_frame(world2boxes + (n * A + a) * 12, w);
    if (fabsf(b.x) < bounds[3 * a] && fabsf(b.y) < bounds[3 * a + 1] && fabsf(b.z) < bounds[3 * a + 2]) {
      hit = a;
      bx = b.x, by = b.y, bz = b.z;
    }
  };
  if (cull) {
    const uint32_t* flagged = s_mask + (n - n0) * words;
    for (int k = 0; k < words; ++k) {
      for (uint32_t bits = flagged[k]; bits != 0u; bits &= bits - 1u) box_test(32 * k + __ffs(bits) - 1);
    }
  } else {
    for (int a = 0; a < A; ++a) box_test(a);
  }
  grid_id[gid] = hit >= 0 ? actor_to_id[hit] : -1;
  if (actor_index != nullptr) actor_index[gid] = hit;
  if (hit < 0) return;
  const float* m = world2boxes + (n * A + hit) * 12;
  float rx = m[0] * dx + m[1] * dy + m[2] * dz, ry = m[4] * dx + m[5] * dy + m[6] * dz, rz = m[8] * dx + m[9] * dy + m[10] * dz;
  const float inv = 1.0f / (sqrtf(rx * rx + ry * ry + rz * rz) + 1.0e-7f);
  rx *= inv, ry *= inv, rz *= inv;
  if (flip != nullptr) {  // random mirror of the actor's x axis, one draw per ray (neurad_encoding.py:218-225)
    bx *= flip[n];
    rx *= flip[n];
  }
  const Gaussian c = contract_gaussian(bx, by, bz, w.std, actor_scale);
  pos[3 * gid] = c.x, pos[3 * gid + 1] = c.y, pos[3 * gid + 2] = c.z;
  std[gid] = c.std;
  dirs[3 * gid] = rx, dirs[3 * gid + 1] = ry, dirs[3 * gid + 2] = rz;
}

// Shared memory of actor_assign_kernel's pre-cull: the rays a block of 256 consecutive samples can touch (at most
// ceil(255 / S) + 1, 256 for S = 1) times ceil(A / 32) mask words; at most 8 KB.  None above NRB_MAX_ACTORS.
static size_t actor_cull_bytes(int S, int A) {
  if (A > NRB_MAX_ACTORS) return 0;
  return sizeof(uint32_t) * static_cast<size_t>((255 + S - 1) / S + 1) * ((A + 31) / 32);
}

struct ActorGradDev {
  float* tables[NRB_MAX_ACTORS];
};

// Scatter of the 16 actor features' gradient (tile image of the fused field backward, tile_image_chunk) into the
// sample's actor table; optionally the gradient with respect to the sample's position in the grid's unit cube.  One
// thread per (sample, level); ~10 % of the samples belong to actors.
template <bool kNeedDx>
__global__ void __launch_bounds__(256) actor_scatter_kernel(const __grid_constant__ ActorGridsDev ag,
                                                            const __grid_constant__ ActorGradDev grads,
                                                            const __grid_constant__ ActorSamplesDev as,
                                                            const float* __restrict__ dyimg, float* __restrict__ dpos,
                                                            int64_t total) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int64_t m = gid / kActorLevels;
  const int l = static_cast<int>(gid - m * kActorLevels);
  const int grid = as.grid_id[m];
  if (grid < 0) return;
  const float scal = ag.scalings[l];
  const float px = as.pos[3 * m], py = as.pos[3 * m + 1], pz = as.pos[3 * m + 2];
  const Cell c = locate_cell(px, py, pz, scal, (1u << ag.log2_size) - 1u);
  float gr[4];
  load_row<4>(tile_image_chunk(dyimg, m, l), 0, gr);  // features 4l .. 4l+3
  const float lw = level_weight(scal, as.std[m]);
#pragma unroll
  for (int j = 0; j < 4; ++j) gr[j] *= lw;
  float w[8];
  corner_weights(c, w);
  const size_t level_off = (static_cast<size_t>(l) << ag.log2_size) * 4;
  float* dt = grads.tables[grid] + level_off;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = gr[j] * w[k];
    scatter_row<4>(dt, c.row[k], v);
  }
  if constexpr (kNeedDx) {
    const float3 d = position_grad<4>(ag.tables[grid] + level_off, c, gr);
    atomicAdd(dpos + 3 * m + 0, d.x * scal);
    atomicAdd(dpos + 3 * m + 1, d.y * scal);
    atomicAdd(dpos + 3 * m + 2, d.z * scal);
  }
}

// Gradient with respect to world2boxes [N,A,3,4] of the actor samples' features, for trained actor trajectories
// (NeuRADHashEncoding keeps grad mode for the poses, neurad_encoding.py:176-229).  One thread per sample.  The sample's
// box-frame point p = R x + t is recomputed with actor_assign_kernel's helper; its grid position and std are the
// forward's own (`as`), so cells and level weights are the ones the forward used.  With g = d loss / d feat[0..15] (tile
// image, as actor_scatter_kernel reads it):
//   d pos = sum_l lw_l scal_l grad_o interp_l . g_l,   d std = sum_l lw_l'(std) interp_l . g_l,
// lw_l' = -2 scal_l / (2 scal_l std)^2 where 2 scal_l std >= 1 (torch's clamp_min passes the gradient at equality), else
// 0; then back through pos = (c + 2) / 4, std = sc / 4, the L-inf contraction of u = q / actor_scale (its full Jacobian
// for the mean, and the sc(max|u|) path outside the linear region), the flip q = (f p_x, p_y, p_z) and p = R x + t:
// dR += dp x^T, dt += dp.  The view direction takes no gradient (the SH encoding is no-grad).  The samples of one
// (ray, actor) are consecutive, so a warp adds its lanes per key n * A + a (segmented scan) before the 12 atomics.
__global__ void __launch_bounds__(256) actor_pose_grad_kernel(const float* __restrict__ origins,
                                                              const float* __restrict__ directions,
                                                              const float* __restrict__ pixel_area, nrb_intervals_t iv,
                                                              const float* __restrict__ world2boxes, int A,
                                                              const int32_t* __restrict__ actor_index,
                                                              const float* __restrict__ flip, float actor_scale,
                                                              const __grid_constant__ ActorGridsDev ag,
                                                              const __grid_constant__ ActorSamplesDev as,
                                                              const float* __restrict__ dyimg, float* __restrict__ dw2b,
                                                              int64_t total) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int lane = static_cast<int>(threadIdx.x) & (kWarp - 1);
  const int hit = gid < total ? actor_index[gid] : -1;
  if (__ballot_sync(kFull, hit >= 0) == 0u) return;  // (whole warps: the block size is a multiple of 32)
  const int S = iv.num_samples;
  const int64_t n = gid / S;
  float g[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) g[i] = 0.f;
  if (hit >= 0) {
    const int s = static_cast<int>(gid - n * S);
    const Gaussian w = world_gaussian(origins[3 * n], origins[3 * n + 1], origins[3 * n + 2], directions[3 * n],
                                      directions[3 * n + 1], directions[3 * n + 2], pixel_area[n],
                                      iv.starts[n * iv.row_stride + s], iv.ends[n * iv.row_stride + s]);
    const float3 p = to_box_frame(world2boxes + (n * A + hit) * 12, w);
    const float f = flip != nullptr ? flip[n] : 1.0f;
    // d loss / d (pos, std) of the 4-level lookup
    const int grid = as.grid_id[gid];
    const float px = as.pos[3 * gid], py = as.pos[3 * gid + 1], pz = as.pos[3 * gid + 2], sd = as.std[gid];
    const uint32_t mask = (1u << ag.log2_size) - 1u;
    float dpx = 0.f, dpy = 0.f, dpz = 0.f, dsd = 0.f;
#pragma unroll
    for (int l = 0; l < kActorLevels; ++l) {
      const float scal = ag.scalings[l];
      const Cell c = locate_cell(px, py, pz, scal, mask);
      const float* base = ag.tables[grid] + (static_cast<size_t>(l) << ag.log2_size) * 4;
      float gr[4], v[4];
      load_row<4>(tile_image_chunk(dyimg, gid, l), 0, gr);
      interpolate<4>(base, c, v);
      const float t = mul(mul(scal, 2.0f), sd);
      if (t >= 1.0f) dsd -= (gr[0] * v[0] + gr[1] * v[1] + gr[2] * v[2] + gr[3] * v[3]) * (2.0f * scal) / (t * t);
      const float lw = level_weight(scal, sd);
#pragma unroll
      for (int j = 0; j < 4; ++j) gr[j] *= lw;
      const float3 d = position_grad<4>(base, c, gr);
      dpx += d.x * scal, dpy += d.y * scal, dpz += d.z * scal;
    }
    // ... through pos = (c + 2) / 4, std = sc / 4 and contract_gaussian (the branch is the forward's: same fp32 u)
    float dcx = 0.25f * dpx, dcy = 0.25f * dpy, dcz = 0.25f * dpz;
    const float dsc = 0.25f * dsd;
    const float ux = div(p.x * f, actor_scale), uy = div(p.y, actor_scale), uz = div(p.z, actor_scale);
    const float ax = fabsf(ux), ay = fabsf(uy), az = fabsf(uz);
    const float mag = fmaxf(fmaxf(ax, ay), az);
    if (!(mag < 1.0f)) {
      // c = h(m) u with h = 2/m - 1/m^2; sc = (std / scale) (2m - 1)^(2/3) / m^2; m = max |u_i| (torch's amax shares
      // the gradient among tied maxima)
      const float im = 1.0f / mag, h = (2.0f - im) * im, dh = 2.0f * im * im * (im - 1.0f);
      const float q = cbrtf(2.0f * mag - 1.0f);
      const float dr2 = (4.0f / 3.0f) / q * im * im - 2.0f * q * q * im * im * im;
      const float dm = dh * (dcx * ux + dcy * uy + dcz * uz) + dsc * (w.std / actor_scale) * dr2;
      const float ties = static_cast<float>((ax == mag) + (ay == mag) + (az == mag));
      const float dmt = dm / ties;
      dcx = h * dcx + (ax == mag ? (ux < 0.f ? -dmt : dmt) : 0.f);
      dcy = h * dcy + (ay == mag ? (uy < 0.f ? -dmt : dmt) : 0.f);
      dcz = h * dcz + (az == mag ? (uz < 0.f ? -dmt : dmt) : 0.f);
    }
    // ... through u = q / scale and the flip: d p
    const float is = 1.0f / actor_scale;
    const float dp[3] = {dcx * is * f, dcy * is, dcz * is};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      g[4 * r + 0] = dp[r] * w.x;
      g[4 * r + 1] = dp[r] * w.y;
      g[4 * r + 2] = dp[r] * w.z;
      g[4 * r + 3] = dp[r];
    }
  }
  // segmented inclusive sum over the warp's runs of equal (ray, actor); the last lane of a run adds it
  const int64_t key = hit >= 0 ? n * A + hit : -1;
  const int64_t prev = __shfl_up_sync(kFull, key, 1);
  const int64_t next = __shfl_down_sync(kFull, key, 1);
  const uint32_t heads = __ballot_sync(kFull, lane == 0 || prev != key);
  const int head = 31 - __clz(heads & (0xFFFFFFFFu >> (31 - lane)));
#pragma unroll
  for (int o = 1; o < kWarp; o <<= 1) {
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const float v = __shfl_up_sync(kFull, g[i], o);
      if (lane - o >= head) g[i] += v;
    }
  }
  if (hit >= 0 && (lane == kWarp - 1 || next != key)) {
#pragma unroll
    for (int i = 0; i < 12; ++i) atomicAdd(dw2b + key * 12 + i, g[i]);
  }
}

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_actor_assign(const nrb_rays_t* rays, const nrb_intervals_t* iv, const float* world2boxes,
                                const uint8_t* valid, const float* bounds, const int32_t* actor_to_id, int32_t num_actors,
                                const float* flip, float actor_scale, int32_t* grid_id, float* pos, float* std, float* dirs,
                                int32_t* actor_index, nrb_stream_t stream) {
  if (int rc = check_rays(rays)) return rc;
  if (int rc = check_intervals("nrb_actor_assign", iv)) return rc;
  NRB_REQUIRE(world2boxes && valid && bounds && actor_to_id && grid_id && pos && std && dirs, NRB_ERR_BAD_ARG,
              "nrb_actor_assign: null pointer");
  NRB_REQUIRE(num_actors >= 1 && actor_scale > 0.f, NRB_ERR_BAD_ARG, "nrb_actor_assign: bad num_actors / actor_scale");
  if (rays->num_rays == 0) return NRB_OK;
  const int64_t total = rays->num_rays * iv->num_samples;
  actor_assign_kernel<<<blocks_for(total, 256), 256, actor_cull_bytes(iv->num_samples, num_actors),
                        static_cast<cudaStream_t>(stream)>>>(
      rays->origins, rays->directions, rays->pixel_area, *iv, world2boxes, valid, bounds, actor_to_id, num_actors, flip,
      actor_scale, grid_id, pos, std, dirs, actor_index, total);
  return finish_launch("nrb_actor_assign");
}

extern "C" int nrb_actor_scatter(const nrb_actor_grids_t* grids, float* const* dtables, const nrb_actor_samples_t* samples,
                                 const float* dyimg, float* dpos, int64_t M, nrb_stream_t stream) {
  if (int rc = check_actor_grids("nrb_actor_scatter", grids)) return rc;
  NRB_REQUIRE(dtables && samples && samples->grid_id && samples->pos && samples->std && dyimg && M >= 0, NRB_ERR_BAD_ARG,
              "nrb_actor_scatter: null pointer");
  NRB_REQUIRE(aligned16(dyimg), NRB_ERR_ALIGNMENT, "nrb_actor_scatter: dyimg must be 16-byte aligned");
  if (M == 0) return NRB_OK;
  ActorGradDev gd{};
  for (int i = 0; i < grids->num_grids; ++i) {
    NRB_REQUIRE(dtables[i] != nullptr && aligned16(dtables[i]), NRB_ERR_BAD_ARG, "nrb_actor_scatter: gradient table %d", i);
    gd.tables[i] = dtables[i];
  }
  const ActorSamplesDev as{samples->grid_id, samples->pos, samples->std, samples->dirs};
  const int64_t total = M * kActorLevels;
  auto s = static_cast<cudaStream_t>(stream);
  if (dpos != nullptr) {
    cudaError_t e = cudaMemsetAsync(dpos, 0, sizeof(float) * 3 * M, s);
    NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "nrb_actor_scatter: memset failed: %s", cudaGetErrorString(e));
    actor_scatter_kernel<true><<<blocks_for(total, 256), 256, 0, s>>>(to_dev(grids), gd, as, dyimg, dpos, total);
  } else {
    actor_scatter_kernel<false><<<blocks_for(total, 256), 256, 0, s>>>(to_dev(grids), gd, as, dyimg, dpos, total);
  }
  return finish_launch("nrb_actor_scatter");
}

extern "C" int nrb_actor_pose_grad(const nrb_rays_t* rays, const nrb_intervals_t* iv, const float* world2boxes,
                                   int32_t num_actors, const int32_t* actor_index, const float* flip, float actor_scale,
                                   const nrb_actor_grids_t* grids, const nrb_actor_samples_t* samples, const float* dyimg,
                                   float* dworld2boxes, nrb_stream_t stream) {
  if (int rc = check_rays(rays)) return rc;
  if (int rc = check_intervals("nrb_actor_pose_grad", iv)) return rc;
  if (int rc = check_actor_grids("nrb_actor_pose_grad", grids)) return rc;
  NRB_REQUIRE(world2boxes && actor_index && samples && samples->grid_id && samples->pos && samples->std && dyimg &&
                  dworld2boxes,
              NRB_ERR_BAD_ARG, "nrb_actor_pose_grad: null pointer");
  NRB_REQUIRE(num_actors >= 1 && actor_scale > 0.f, NRB_ERR_BAD_ARG, "nrb_actor_pose_grad: bad num_actors / actor_scale");
  NRB_REQUIRE(aligned16(dyimg), NRB_ERR_ALIGNMENT, "nrb_actor_pose_grad: dyimg must be 16-byte aligned");
  if (rays->num_rays == 0) return NRB_OK;
  const int64_t total = rays->num_rays * iv->num_samples;
  const ActorSamplesDev as{samples->grid_id, samples->pos, samples->std, samples->dirs};
  actor_pose_grad_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      rays->origins, rays->directions, rays->pixel_area, *iv, world2boxes, num_actors, actor_index, flip, actor_scale,
      to_dev(grids), as, dyimg, dworld2boxes, total);
  return finish_launch("nrb_actor_pose_grad");
}
