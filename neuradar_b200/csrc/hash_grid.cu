// Multiresolution hash grid: forward gather, index dump, backward scatter, and the sample-gaussian producer.
// Semantics: HashEncoding.pytorch_fwd / hash_fn (nerfstudio/field_components/encodings.py:406-466) and
// NeuRADHashEncoding._rescale_grid_features (nerfstudio/field_components/neurad_encoding.py:309-316).
//
// Work decomposition: one thread per (point, level) pair with the level index fastest.  The 2^19..2^22-row tables
// are hit at random, so there is nothing to coalesce on the gather side; what can be coalesced is the [M, L*F]
// feature matrix, and with the level fastest a warp writes (reads, in the backward pass) one contiguous
// 32*F*4-byte span of it.  Each thread issues its 8 independent F-wide vector gathers before touching any of them.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "hash_bwd_plan.cuh"

namespace nrb {

template <int F>
__global__ void __launch_bounds__(256) hash_fwd_kernel(const __grid_constant__ GridDev g, const float* __restrict__ x,
                                                       const float* __restrict__ std, float* __restrict__ out,
                                                       int64_t total) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int64_t m = gid / g.num_levels;
  const int l = static_cast<int>(gid - m * g.num_levels);
  const float scal = g.scalings[l];
  const Cell c = locate_cell(__ldg(x + 3 * m), __ldg(x + 3 * m + 1), __ldg(x + 3 * m + 2), scal,
                             (1u << g.log2_size) - 1u);
  const float* base = g.table + (static_cast<size_t>(l) << g.log2_size) * F;
  float v[F];
  interpolate<F>(base, c, v);
  if (std != nullptr) {
    const float w = level_weight(scal, __ldg(std + m));
#pragma unroll
    for (int j = 0; j < F; ++j) v[j] *= w;
  }
  using V = typename Feat<F>::type;
  V o;
  if constexpr (F == 1) {
    o = v[0];
  } else if constexpr (F == 2) {
    o = make_float2(v[0], v[1]);
  } else {
    o = make_float4(v[0], v[1], v[2], v[3]);
  }
  reinterpret_cast<V*>(out)[gid] = o;
}

// Sample-major forward: one warp = 32 consecutive samples (lane = sample), looping over the levels.  Consecutive
// samples of a ray mostly fall into the same cell (see hash_bwd_merge_kernel), so the 32 gathers of one corner hit a
// handful of distinct rows and coalesce in L1/TEX, which is the unit that bounds the level-major kernel above (ncu:
// 95 % busy, one line per lane).  The 32 output rows are assembled in a swizzled shared-memory tile and written with
// coalesced 16-byte stores.
constexpr int kFwdWarps = 8;

template <int F>
__global__ void __launch_bounds__(kFwdWarps * 32) hash_fwd_rows_kernel(const __grid_constant__ GridDev g,
                                                                      const float* __restrict__ x,
                                                                      const float* __restrict__ std,
                                                                      float* __restrict__ out, int64_t M) {
  extern __shared__ __align__(16) char fwd_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = g.num_levels, RW = L * F, CPR = RW / 4;
  char* tile = fwd_smem + warp * (32 * RW * 4);
  const int64_t base = (static_cast<int64_t>(blockIdx.x) * kFwdWarps + warp) * 32;
  if (base >= M) return;
  const int64_t mc = min(base + lane, M - 1);
  const float px = __ldg(x + 3 * mc), py = __ldg(x + 3 * mc + 1), pz = __ldg(x + 3 * mc + 2);
  const float sd = std != nullptr ? __ldg(std + mc) : 0.0f;
  const uint32_t mask = (1u << g.log2_size) - 1u;
  char* rowp = tile + lane * (RW * 4);
  for (int l = 0; l < L; ++l) {
    const float scal = g.scalings[l];
    const Cell c = locate_cell(px, py, pz, scal, mask);
    float v[F];
    interpolate<F>(g.table + (static_cast<size_t>(l) << g.log2_size) * F, c, v);
    if (std != nullptr) {
      const float w = level_weight(scal, sd);
#pragma unroll
      for (int j = 0; j < F; ++j) v[j] *= w;
    }
    const int f0 = l * F;
    char* dst = rowp + (((f0 >> 2) ^ (lane % CPR)) << 4) + (f0 & 3) * 4;
    if constexpr (F == 4) {
      *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    } else if constexpr (F == 2) {
      *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
    } else {
      *reinterpret_cast<float*>(dst) = v[0];
    }
  }
  __syncwarp();
  for (int e = lane; e < 32 * CPR; e += 32) {
    const int r = e / CPR, cc = e - r * CPR;
    if (base + r < M)
      reinterpret_cast<float4*>(out + (base + r) * RW)[cc] =
          *reinterpret_cast<const float4*>(tile + r * (RW * 4) + ((cc ^ (r % CPR)) << 4));
  }
}

__global__ void __launch_bounds__(256) hash_indices_kernel(const __grid_constant__ GridDev g, const float* __restrict__ x,
                                                           int64_t* __restrict__ idx, int64_t total) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int64_t m = gid / g.num_levels;
  const int l = static_cast<int>(gid - m * g.num_levels);
  const Cell c = locate_cell(x[3 * m], x[3 * m + 1], x[3 * m + 2], g.scalings[l], (1u << g.log2_size) - 1u);
  const int64_t off = static_cast<int64_t>(l) << g.log2_size;
#pragma unroll
  for (int k = 0; k < 8; ++k) idx[gid * 8 + k] = off + c.row[k];
}

template <int F, bool kNeedDx>
__global__ void __launch_bounds__(256) hash_bwd_kernel(const __grid_constant__ GridDev g,
                                                       const __grid_constant__ BwdPlan plan,
                                                       const float* __restrict__ x, const float* __restrict__ std,
                                                       const float* __restrict__ dy, float* __restrict__ dtable,
                                                       float* __restrict__ dx, int64_t total) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int64_t m = gid / g.num_levels;
  const int l = static_cast<int>(gid - m * g.num_levels);
  const float scal = g.scalings[l];
  const float px = __ldg(x + 3 * m), py = __ldg(x + 3 * m + 1), pz = __ldg(x + 3 * m + 2);
  const Cell c = locate_cell(px, py, pz, scal, (1u << g.log2_size) - 1u);
  float gr[F];
  load_row<F>(dy + gid * F, 0, gr);
  if (std != nullptr) {
    const float lw = level_weight(scal, __ldg(std + m));
#pragma unroll
    for (int j = 0; j < F; ++j) gr[j] *= lw;
  }
  if constexpr (kNeedDx) {  // d out / d offset needs the corner features themselves
    const float3 d = position_grad<F>(g.table + (static_cast<size_t>(l) << g.log2_size) * F, c, gr);
    atomicAdd(dx + 3 * m + 0, d.x * scal);
    atomicAdd(dx + 3 * m + 1, d.y * scal);
    atomicAdd(dx + 3 * m + 2, d.z * scal);
  }
  float w[8];
  corner_weights(c, w);
  float v[8][F];
#pragma unroll
  for (int k = 0; k < 8; ++k)
#pragma unroll
    for (int j = 0; j < F; ++j) v[k][j] = w[k] * gr[j];
  const float sx = mul(px, scal), sy = mul(py, scal), sz = mul(pz, scal);
  const int xf = static_cast<int>(floorf(sx)), yf = static_cast<int>(floorf(sy)), zf = static_cast<int>(floorf(sz));
  const int xc = static_cast<int>(ceilf(sx)), yc = static_cast<int>(ceilf(sy)), zc = static_cast<int>(ceilf(sz));
  scatter_corners<F>(plan, l, g.log2_size, xf, yf, zf, xc, yc, zc, c.row, v, dtable, static_cast<unsigned>(gid >> 5));
}

// Backward scatter with run merging.  One warp = 32 consecutive samples (lane = sample), looping over the levels.
// Samples come ray by ray, and after two importance-sampling rounds neighbours along a ray are close: on the benchmark
// rays 67 % (finest level) to 95 % (coarsest) of adjacent samples fall into the SAME cell, i.e. update the same 8 rows.
// The scatter kernels are bound by the number of reductions they issue (RED issue rate, DESIGN.md section 4), so each
// run of adjacent lanes with identical (floor, ceil) cell coordinates first adds up its 8 x F corner contributions with
// a segmented shuffle reduction, and only the head lane of the run issues reductions (merge_runs_and_scatter,
// hash_bwd_plan.cuh).
//   kImage = false: dy is row-major [M, L*F] (nrb_hash_bwd).  Its rows are staged through shared memory (coalesced
//                   loads, XOR-swizzled 16-byte chunks) because a lane reading its own row touches 32 lines per load.
//   kImage = true:  dy is the fused field backward's tile image (nrb_hash_bwd_image, tile_image_chunk), which a lane
//                   reads coalesced without staging.  actor_grid_id (may be null) marks the samples claimed by an actor
//                   grid: they took none of their features from this table.
constexpr int kMergeWarps = 8;

template <int F, bool kImage>
__global__ void __launch_bounds__(kMergeWarps * 32) hash_bwd_merge_kernel(const __grid_constant__ GridDev g,
                                                                          const __grid_constant__ BwdPlan plan,
                                                                          const float* __restrict__ x,
                                                                          const float* __restrict__ std,
                                                                          const float* __restrict__ dy,
                                                                          const int32_t* __restrict__ actor_grid_id,
                                                                          float* __restrict__ dtable, int64_t M) {
  extern __shared__ __align__(16) char dy_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = g.num_levels, RW = L * F;  // floats per dy row (4, 8, ..., 64: checked by the launcher)
  const int CPR = RW / 4;                  // 16-byte chunks per row
  char* tile = dy_smem + warp * (32 * RW * 4);
  const int64_t base = (static_cast<int64_t>(blockIdx.x) * kMergeWarps + warp) * 32;
  if (base >= M) return;
  const int64_t m = base + lane;
  const int64_t mc = m < M ? m : (M - 1);
  const bool valid = m < M && (!kImage || actor_grid_id == nullptr || __ldg(actor_grid_id + mc) < 0);
  if constexpr (!kImage) {  // coalesced copy of the 32 dy rows into the swizzled tile
    for (int e = lane; e < 32 * CPR; e += 32) {
      const int r = e / CPR, cc = e - r * CPR;
      const int64_t rr = min(base + r, M - 1);
      const float4 t = __ldg(reinterpret_cast<const float4*>(dy + rr * RW) + cc);
      *reinterpret_cast<float4*>(tile + r * (RW * 4) + ((cc ^ (r % CPR)) << 4)) = t;
    }
  }
  const float px = __ldg(x + 3 * mc), py = __ldg(x + 3 * mc + 1), pz = __ldg(x + 3 * mc + 2);
  const float sd = std != nullptr ? __ldg(std + mc) : 0.0f;
  if constexpr (!kImage) __syncwarp();
  const uint32_t mask = (1u << g.log2_size) - 1u;
  const unsigned spread = static_cast<unsigned>(base >> 5);
  for (int l = 0; l < L; ++l) {
    const float scal = g.scalings[l];
    const Cell c = locate_cell(px, py, pz, scal, mask);
    const int f0 = l * F;  // first float of this level in the row
    float gr[F];
    if constexpr (kImage) {
      load_row<F>(tile_image_chunk(dy, m, f0 >> 2) + (f0 & 3), 0, gr);
    } else {
      const char* p = tile + lane * (RW * 4) + (((f0 >> 2) ^ (lane % CPR)) << 4) + (f0 & 3) * 4;
      if constexpr (F == 4) {
        const float4 t = *reinterpret_cast<const float4*>(p);
        gr[0] = t.x, gr[1] = t.y, gr[2] = t.z, gr[3] = t.w;
      } else if constexpr (F == 2) {
        const float2 t = *reinterpret_cast<const float2*>(p);
        gr[0] = t.x, gr[1] = t.y;
      } else {
        gr[0] = *reinterpret_cast<const float*>(p);
      }
    }
    const float lw = (std != nullptr ? level_weight(scal, sd) : 1.0f) * (valid ? 1.0f : 0.0f);
    float w[8];
    corner_weights(c, w);
    float v[8][F];
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
      for (int j = 0; j < F; ++j) v[k][j] = w[k] * (gr[j] * lw);
    merge_runs_and_scatter<F>(plan, l, g.log2_size, px, py, pz, scal, c, v, valid, lane, dtable, spread);
  }
}

// Adds the replicas of every replicated level into the table: one thread per lattice vertex.
template <int F>
__global__ void __launch_bounds__(256) hash_bwd_fold_kernel(const __grid_constant__ GridDev g,
                                                            const __grid_constant__ BwdPlan plan,
                                                            float* __restrict__ dtable, int64_t total_vertices) {
  int64_t v = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= total_vertices) return;
  int l = 0;
  for (; l < g.num_levels; ++l) {
    if (plan.copies[l] <= 1) continue;
    const int64_t nvl = static_cast<int64_t>(plan.r1[l]) * plan.r1[l] * plan.r1[l];
    if (v < nvl) break;
    v -= nvl;
  }
  if (l >= g.num_levels) return;
  const float* rep = plan.scratch + plan.offset[l] + v * F;
  float sum[F];
#pragma unroll
  for (int j = 0; j < F; ++j) sum[j] = 0.0f;
  for (int cpy = 0; cpy < plan.copies[l]; ++cpy) {
    float t[F];
    load_row<F>(rep + static_cast<size_t>(cpy) * plan.stride[l], 0, t);
#pragma unroll
    for (int j = 0; j < F; ++j) sum[j] += t[j];
  }
  bool any = false;
#pragma unroll
  for (int j = 0; j < F; ++j) any |= (sum[j] != 0.0f);
  if (!any) return;
  const int R1 = plan.r1[l];
  const int ix = static_cast<int>(v % R1), iy = static_cast<int>((v / R1) % R1), iz = static_cast<int>(v / (R1 * R1));
  const uint32_t row = (static_cast<uint32_t>(ix) ^ (static_cast<uint32_t>(iy) * kPrimeY) ^
                        (static_cast<uint32_t>(iz) * kPrimeZ)) & ((1u << g.log2_size) - 1u);
  scatter_row<F>(dtable + (static_cast<size_t>(l) << g.log2_size) * F, row, sum);
}

void launch_fold(const nrb_grid_t* grid, const BwdPlan& plan, float* dtable, int64_t vertices, cudaStream_t s) {
  if (vertices <= 0) return;
  count_launch();
  const unsigned blocks = blocks_for(vertices, 256);
  switch (grid->features_per_level) {
    case 1: hash_bwd_fold_kernel<1><<<blocks, 256, 0, s>>>(to_dev(grid), plan, dtable, vertices); break;
    case 2: hash_bwd_fold_kernel<2><<<blocks, 256, 0, s>>>(to_dev(grid), plan, dtable, vertices); break;
    default: hash_bwd_fold_kernel<4><<<blocks, 256, 0, s>>>(to_dev(grid), plan, dtable, vertices); break;
  }
}

__global__ void __launch_bounds__(256) frustum_gaussians_kernel(const float* __restrict__ origins,
                                                                const float* __restrict__ directions,
                                                                const float* __restrict__ pixel_area,
                                                                nrb_intervals_t iv, float scale,
                                                                float* __restrict__ x, float* __restrict__ std,
                                                                int64_t total) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int S = iv.num_samples;
  const int64_t n = gid / S;
  const int s = static_cast<int>(gid - n * S);
  const Gaussian g = sample_gaussian(origins[3 * n], origins[3 * n + 1], origins[3 * n + 2], directions[3 * n],
                                     directions[3 * n + 1], directions[3 * n + 2], pixel_area[n],
                                     iv.starts[n * iv.row_stride + s], iv.ends[n * iv.row_stride + s], scale);
  x[3 * gid + 0] = g.x;
  x[3 * gid + 1] = g.y;
  x[3 * gid + 2] = g.z;
  std[gid] = g.std;
}

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_hash_fwd(const nrb_grid_t* grid, const float* x, const float* std, float* out, int64_t M,
                            nrb_stream_t stream) {
  if (int rc = check_grid(grid)) return rc;
  NRB_REQUIRE(x && out && M >= 0, NRB_ERR_BAD_ARG, "nrb_hash_fwd: null pointer or negative M");
  NRB_REQUIRE(aligned16(out), NRB_ERR_ALIGNMENT, "nrb_hash_fwd: out must be 16-byte aligned");
  if (M == 0) return NRB_OK;
  const int64_t total = M * grid->num_levels;
  const GridDev g = to_dev(grid);
  auto s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = blocks_for(total, 256);
  const int row_floats = grid->num_levels * grid->features_per_level;
  // power-of-two row widths (the field grids): warp-transposed rows kernel; other shapes (L6/F1 proposals, tiny M): generic
  if (row_floats >= 4 && row_floats <= 64 && (row_floats & (row_floats - 1)) == 0 && M >= 32) {
    const size_t smem = static_cast<size_t>(kFwdWarps) * 32 * row_floats * 4;
    const unsigned nb = blocks_for(M, kFwdWarps * 32);
#define NRB_ROWS(F)                                                                                                    \
  {                                                                                                                    \
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(hash_fwd_rows_kernel<F>), 64 * 1024); \
    NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "nrb_hash_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); \
    hash_fwd_rows_kernel<F><<<nb, kFwdWarps * 32, smem, s>>>(g, x, std, out, M);                                        \
  }
    switch (grid->features_per_level) {
      case 1: NRB_ROWS(1) break;
      case 2: NRB_ROWS(2) break;
      default: NRB_ROWS(4) break;
    }
#undef NRB_ROWS
    return finish_launch("nrb_hash_fwd");
  }
  switch (grid->features_per_level) {
    case 1: hash_fwd_kernel<1><<<blocks, 256, 0, s>>>(g, x, std, out, total); break;
    case 2: hash_fwd_kernel<2><<<blocks, 256, 0, s>>>(g, x, std, out, total); break;
    default: hash_fwd_kernel<4><<<blocks, 256, 0, s>>>(g, x, std, out, total); break;
  }
  return finish_launch("nrb_hash_fwd");
}

extern "C" int nrb_hash_indices(const nrb_grid_t* grid, const float* x, int64_t* idx, int64_t M,
                                nrb_stream_t stream) {
  if (int rc = check_grid(grid)) return rc;
  NRB_REQUIRE(x && idx && M >= 0, NRB_ERR_BAD_ARG, "nrb_hash_indices: null pointer or negative M");
  if (M == 0) return NRB_OK;
  const int64_t total = M * grid->num_levels;
  hash_indices_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(to_dev(grid), x, idx,
                                                                                             total);
  return finish_launch("nrb_hash_indices");
}

// Replica plan: as many copies of a coarse level's lattice as it takes to bring its reductions per address down to
// those of a level that fills the whole table, within the caller's workspace.
extern "C" int64_t nrb_hash_bwd_workspace_bytes(const nrb_grid_t* grid, int64_t M) {
  if (grid == nullptr || check_grid(grid) != NRB_OK) return -1;
  BwdPlan plan;
  return plan_hash_bwd(grid, M, &plan);
}

template <int F>
static int launch_hash_bwd(const nrb_grid_t* grid, const GridDev& g, const float* x, const float* std, const float* dy,
                           float* dtable, float* dx, int64_t M, void* workspace, int64_t workspace_bytes,
                           cudaStream_t s) {
  BwdPlan plan;
  int64_t vertices = 0;
  if (int rc = prepare_bwd_plan(grid, M, workspace, workspace_bytes, s, &plan, &vertices)) return rc;
  const int64_t total = M * grid->num_levels;
  const unsigned blocks = blocks_for(total, 256);
  const int row_floats = grid->num_levels * F;
  if (dx == nullptr && row_floats >= 4 && row_floats <= 64 && (row_floats & (row_floats - 1)) == 0 && M >= 32) {
    const size_t smem = static_cast<size_t>(kMergeWarps) * 32 * row_floats * 4;
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(hash_bwd_merge_kernel<F, false>), 64 * 1024);
    NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "nrb_hash_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    hash_bwd_merge_kernel<F, false><<<blocks_for(M, kMergeWarps * 32), kMergeWarps * 32, smem, s>>>(g, plan, x, std, dy,
                                                                                                    nullptr, dtable, M);
  } else if (dx != nullptr) {
    hash_bwd_kernel<F, true><<<blocks, 256, 0, s>>>(g, plan, x, std, dy, dtable, dx, total);
  } else {
    hash_bwd_kernel<F, false><<<blocks, 256, 0, s>>>(g, plan, x, std, dy, dtable, dx, total);
  }
  launch_fold(grid, plan, dtable, vertices, s);
  return finish_launch("nrb_hash_bwd");
}

extern "C" int nrb_hash_bwd(const nrb_grid_t* grid, const float* x, const float* std, const float* dy, float* dtable,
                            float* dx, int64_t M, void* workspace, int64_t workspace_bytes, nrb_stream_t stream) {
  if (int rc = check_grid(grid)) return rc;
  NRB_REQUIRE(x && dy && dtable && M >= 0, NRB_ERR_BAD_ARG, "nrb_hash_bwd: null pointer or negative M");
  NRB_REQUIRE(aligned16(dy) && aligned16(dtable), NRB_ERR_ALIGNMENT, "nrb_hash_bwd: dy/dtable must be 16-byte aligned");
  if (M == 0) return NRB_OK;
  const GridDev g = to_dev(grid);
  auto s = static_cast<cudaStream_t>(stream);
  if (dx != nullptr) {
    cudaError_t e = cudaMemsetAsync(dx, 0, sizeof(float) * 3 * M, s);
    NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "nrb_hash_bwd: memset failed: %s", cudaGetErrorString(e));
  }
  switch (grid->features_per_level) {
    case 1: return launch_hash_bwd<1>(grid, g, x, std, dy, dtable, dx, M, workspace, workspace_bytes, s);
    case 2: return launch_hash_bwd<2>(grid, g, x, std, dy, dtable, dx, M, workspace, workspace_bytes, s);
    default: return launch_hash_bwd<4>(grid, g, x, std, dy, dtable, dx, M, workspace, workspace_bytes, s);
  }
}

extern "C" int nrb_hash_bwd_image(const nrb_grid_t* grid, const float* x, const float* std, const float* dyimg,
                                  float* dtable, const int32_t* actor_grid_id, int64_t M, void* workspace,
                                  int64_t workspace_bytes, nrb_stream_t stream) {
  if (int rc = check_grid(grid)) return rc;
  NRB_REQUIRE(x && dyimg && dtable && M >= 0, NRB_ERR_BAD_ARG, "nrb_hash_bwd_image: null pointer or negative M");
  NRB_REQUIRE(aligned16(dyimg) && aligned16(dtable), NRB_ERR_ALIGNMENT, "nrb_hash_bwd_image: dyimg/dtable must be 16-byte aligned");
  NRB_REQUIRE(grid->num_levels * grid->features_per_level == 32, NRB_ERR_UNSUPPORTED,
              "nrb_hash_bwd_image: the tile image holds 32 features per sample");
  if (M == 0) return NRB_OK;
  auto s = static_cast<cudaStream_t>(stream);
  BwdPlan plan;
  int64_t vertices = 0;
  if (int rc = prepare_bwd_plan(grid, M, workspace, workspace_bytes, s, &plan, &vertices)) return rc;
  const GridDev g = to_dev(grid);
  const unsigned nblk = blocks_for(M, kMergeWarps * 32);
  switch (grid->features_per_level) {
    case 2:
      hash_bwd_merge_kernel<2, true><<<nblk, kMergeWarps * 32, 0, s>>>(g, plan, x, std, dyimg, actor_grid_id, dtable, M);
      break;
    case 4:
      hash_bwd_merge_kernel<4, true><<<nblk, kMergeWarps * 32, 0, s>>>(g, plan, x, std, dyimg, actor_grid_id, dtable, M);
      break;
    default:
      NRB_REQUIRE(false, NRB_ERR_UNSUPPORTED, "nrb_hash_bwd_image: features_per_level must be 2 or 4");
  }
  launch_fold(grid, plan, dtable, vertices, s);
  return finish_launch("nrb_hash_bwd_image");
}

extern "C" int nrb_frustum_gaussians(const nrb_rays_t* rays, const nrb_intervals_t* iv, float scale, float* x,
                                     float* std, nrb_stream_t stream) {
  if (int rc = check_rays(rays)) return rc;
  if (int rc = check_intervals("nrb_frustum_gaussians", iv)) return rc;
  NRB_REQUIRE(x && std, NRB_ERR_BAD_ARG, "nrb_frustum_gaussians: null output pointer");
  NRB_REQUIRE(scale > 0.f, NRB_ERR_BAD_ARG, "nrb_frustum_gaussians: scale must be positive");
  if (rays->num_rays == 0) return NRB_OK;
  const int64_t total = rays->num_rays * iv->num_samples;
  frustum_gaussians_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      rays->origins, rays->directions, rays->pixel_area, *iv, scale, x, std, total);
  return finish_launch("nrb_frustum_gaussians");
}
