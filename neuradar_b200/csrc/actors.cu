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
  // first threads test every (ray, actor) pair once and leave a bit mask per ray, the per-sample loop below then runs
  // the exact box test only for the flagged actors (typically none or one of 16).  The sphere contains the box, and the
  // test is evaluated with a margin, so the result is the plain loop's.
  constexpr int kCullRays = 8;
  __shared__ uint32_t s_mask[kCullRays];
  const int S = iv.num_samples;
  const int64_t first = static_cast<int64_t>(blockIdx.x) * blockDim.x;
  const int64_t last = min(first + blockDim.x, total) - 1;
  const int64_t n0 = first / S;
  const int nrays = static_cast<int>(last / S - n0) + 1;
  const bool cull = nrays <= kCullRays && A <= 32;
  if (cull) {
    if (threadIdx.x < kCullRays) s_mask[threadIdx.x] = 0u;
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
        atomicOr(&s_mask[p / A], 1u << a);
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
  uint32_t todo = cull ? s_mask[n - n0] : (A >= 32 ? 0xFFFFFFFFu : (1u << A) - 1u);
  for (int a0 = 0; a0 < A; a0 += 32) {  // (more than 32 actors: plain loop in chunks of 32)
    uint32_t bits = a0 == 0 ? todo : 0xFFFFFFFFu;
    while (bits != 0u) {
      const int a = a0 + __ffs(bits) - 1;
      bits &= bits - 1u;
      if (a >= A) break;
      if (!valid[n * A + a]) continue;
      const float* m = world2boxes + (n * A + a) * 12;
      // rotation as a dot product, then the translation (transform_points_pairwise, cameras/lidars.py:507-519)
      const float x = add(fmaf(m[2], w.z, fmaf(m[1], w.y, mul(m[0], w.x))), m[3]);
      const float y = add(fmaf(m[6], w.z, fmaf(m[5], w.y, mul(m[4], w.x))), m[7]);
      const float z = add(fmaf(m[10], w.z, fmaf(m[9], w.y, mul(m[8], w.x))), m[11]);
      if (fabsf(x) < bounds[3 * a] && fabsf(y) < bounds[3 * a + 1] && fabsf(z) < bounds[3 * a + 2]) {
        hit = a;
        bx = x, by = y, bz = z;
      }
    }
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
  actor_assign_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
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
