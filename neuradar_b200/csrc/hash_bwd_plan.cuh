// Shared by the hash-grid and the fused proposal backward kernels: the device view of a grid, the vector reduction
// into one table row, and the replica plan that spreads the reductions of spatially coherent levels (see below).
#pragma once

#include <algorithm>

#include "common.cuh"

namespace nrb {

struct GridDev {
  const float* table;
  float scalings[NRB_MAX_LEVELS];
  int num_levels;
  int log2_size;
};

inline GridDev to_dev(const nrb_grid_t* g) {
  GridDev d;
  d.table = g->table;
  for (int i = 0; i < NRB_MAX_LEVELS; ++i) d.scalings[i] = g->scalings[i];
  d.num_levels = g->num_levels;
  d.log2_size = g->log2_hashmap_size;
  return d;
}

// Backward scatter.  Same-row float reductions serialise in L2: 25 M reductions take 0.16 ms when they spread over
// the 2^19 rows of a res-1024 level and 7 ms when they pile onto the 4913 rows of a res-16 level (measured, B200).
// Coarse levels are therefore accumulated into `copies[l]` replicas of the level's dense vertex lattice
// ((res+1)^3 x F floats, a few MB in total, L2 resident); warps are dealt round-robin over the replicas, which
// divides the per-address contention by the replica count, and a small fold kernel adds the replicas into the
// hashed rows.  Levels that already fill the table scatter straight into it (DESIGN.md section 4 has the measurements
// behind the plan).  Shared-memory privatisation was measured and rejected: fp32 shared atomics are CAS loops
// (ATOMS.CAST.SPIN) on sm_100 and cost ~1 ms per level.
struct BwdPlan {
  float* scratch;                   // replicated lattices, zeroed by the launcher
  int64_t offset[NRB_MAX_LEVELS];   // float offset of level l's first replica
  int64_t stride[NRB_MAX_LEVELS];   // floats between replicas (multiple of 4: keeps vector reductions 16-byte aligned)
  int copies[NRB_MAX_LEVELS];       // 0/1: scatter straight into the table
  int r1[NRB_MAX_LEVELS];           // res + 1
};

// The scatter works on per-corner VALUES: contributions already multiplied by their corner weights (and, in the
// run-merging kernels, summed over a run of samples that share a cell).
template <int F>
__device__ __forceinline__ void scatter_row(float* __restrict__ base, uint32_t row, const float (&v)[F]) {
  float* p = base + static_cast<size_t>(row) * F;
  if constexpr (F == 1) {
    atomicAdd(p, v[0]);
  } else if constexpr (F == 2) {
    atomicAdd(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
  } else {
    atomicAdd(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
  }
}

// Two rows that differ only in the x corner (floor / ceil).  The x prime of the hash is 1, so the rows are
// floor(x) ^ H and (floor(x) + 1) ^ H with the same H: they differ only in the low bits that the increment carries
// into.  The L2 reduction rate is per operation, not per byte, so the pair is updated with ONE reduction whenever both
// rows lie in one aligned 16-byte group:
//   F = 1: rows r and r' with r >> 2 == r' >> 2 (floor(x) mod 4 != 3: 3 pairs in 4), one F32x4 whose other two slots
//          add +0;
//   F = 2: rows r and r ^ 1 (floor(x) even: 1 pair in 2), one F32x4.
// That is 5 instead of 8 reductions per (point, level) on average for F = 1, 6 for F = 2.  The same holds for the dense
// lattice replicas (x neighbours are adjacent; replicas are 16-byte aligned and padded to whole groups).  `quad`: the
// level holds at least 4 rows, so a 16-byte group of F = 1 rows lies inside it and is aligned (only a 2-row table is
// smaller).
template <int F>
__device__ __forceinline__ void scatter_x_pair(float* __restrict__ base, uint32_t row_f, uint32_t row_c,
                                               const float (&vf)[F], const float (&vc)[F], bool quad) {
  if (row_c == row_f) {  // integral x (ceil == floor; the ceil weight is 0) or a hash collision: one reduction
    float t[F];
#pragma unroll
    for (int j = 0; j < F; ++j) t[j] = vf[j] + vc[j];
    scatter_row<F>(base, row_f, t);
    return;
  }
  if constexpr (F == 1) {
    if (quad && (row_f ^ row_c) < 4u) {
      const uint32_t sf = row_f & 3u, sc = row_c & 3u;
      const float4 t = make_float4(sf == 0 ? vf[0] : (sc == 0 ? vc[0] : 0.0f), sf == 1 ? vf[0] : (sc == 1 ? vc[0] : 0.0f),
                                   sf == 2 ? vf[0] : (sc == 2 ? vc[0] : 0.0f), sf == 3 ? vf[0] : (sc == 3 ? vc[0] : 0.0f));
      atomicAdd(reinterpret_cast<float4*>(base) + (row_f >> 2), t);
      return;
    }
  } else if constexpr (F == 2) {
    if (row_c == (row_f ^ 1u)) {
      const bool f_low = (row_f & 1u) == 0;
      atomicAdd(reinterpret_cast<float4*>(base) + (row_f >> 1), f_low ? make_float4(vf[0], vf[1], vc[0], vc[1])
                                                                     : make_float4(vc[0], vc[1], vf[0], vf[1]));
      return;
    }
  }
  scatter_row<F>(base, row_f, vf);
  scatter_row<F>(base, row_c, vc);
}

// corner order (common.cuh): 0:(c,c,c) 1:(c,f,c) 2:(f,f,c) 3:(f,c,c) 4:(c,c,f) 5:(c,f,f) 6:(f,f,f) 7:(f,c,f);
// x pairs (floor, ceil): (3,0) (2,1) (7,4) (6,5)
template <int F>
__device__ __forceinline__ void scatter_rows8(float* __restrict__ base, const uint32_t (&row)[8], const float (&v)[8][F],
                                              bool quad) {
  scatter_x_pair<F>(base, row[3], row[0], v[3], v[0], quad);
  scatter_x_pair<F>(base, row[2], row[1], v[2], v[1], quad);
  scatter_x_pair<F>(base, row[7], row[4], v[7], v[4], quad);
  scatter_x_pair<F>(base, row[6], row[5], v[6], v[5], quad);
}

// Scatter the 8 corner values of one (point, level): into a replica when the level is replicated and the point lies
// inside the lattice, otherwise straight into the table.  (xf, yf, zf) / (xc, yc, zc): integer floor / ceil
// coordinates of the cell; `spread` picks the replica (warp index).
template <int F>
__device__ __forceinline__ void scatter_corners(const BwdPlan& plan, int l, int log2_size, int xf, int yf, int zf, int xc,
                                                int yc, int zc, const uint32_t (&hashed_rows)[8], const float (&v)[8][F],
                                                float* __restrict__ dtable, unsigned spread) {
  const int copies = plan.copies[l];
  if (copies > 1) {
    const int R1 = plan.r1[l];
    if (xf >= 0 && yf >= 0 && zf >= 0 && xc < R1 && yc < R1 && zc < R1) {
      float* rep = plan.scratch + plan.offset[l] + static_cast<size_t>(spread % static_cast<unsigned>(copies)) * plan.stride[l];
      const int cx[8] = {xc, xc, xf, xf, xc, xc, xf, xf};
      const int cy[8] = {yc, yf, yf, yc, yc, yf, yf, yc};
      const int cz[8] = {zc, zc, zc, zc, zf, zf, zf, zf};
      uint32_t rows[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) rows[k] = static_cast<uint32_t>((cz[k] * R1 + cy[k]) * R1 + cx[k]);
      scatter_rows8<F>(rep, rows, v, true);
      return;
    }
  }
  scatter_rows8<F>(dtable + (static_cast<size_t>(l) << log2_size) * F, hashed_rows, v, log2_size >= 2);
}

// Run merging (called by all 32 lanes of a converged warp whose lanes hold CONSECUTIVE samples of a ray): lanes whose
// points fall into the same cell of level l (identical floor / ceil coordinates) update the same 8 rows, so each run of
// adjacent such lanes adds up its 8 x F corner contributions v (already weighted) with a segmented shuffle reduction
// and only the head lane of the run issues reductions.  Warps whose samples are spread out (more than kMergeMaxRuns
// runs) skip the shuffles.  The scatter kernels are bound by the NUMBER of reductions they issue.
constexpr int kMergeMaxRuns = 26;

template <int F>
__device__ __forceinline__ void merge_runs_and_scatter(const BwdPlan& plan, int l, int log2_size, float px, float py,
                                                       float pz, float scal, const Cell& c, float (&v)[8][F], bool valid,
                                                       int lane, float* __restrict__ dtable, unsigned spread) {
  const float sx = mul(px, scal), sy = mul(py, scal), sz = mul(pz, scal);
  const int xf = static_cast<int>(floorf(sx)), yf = static_cast<int>(floorf(sy)), zf = static_cast<int>(floorf(sz));
  const int xc = static_cast<int>(ceilf(sx)), yc = static_cast<int>(ceilf(sy)), zc = static_cast<int>(ceilf(sz));
  const int ceq = (xc == xf ? 1 : 0) | (yc == yf ? 2 : 0) | (zc == zf ? 4 : 0) | (valid ? 8 : 0);
  const int pxf = __shfl_up_sync(kFull, xf, 1), pyf = __shfl_up_sync(kFull, yf, 1), pzf = __shfl_up_sync(kFull, zf, 1);
  const int pce = __shfl_up_sync(kFull, ceq, 1);
  const bool head = lane == 0 || pxf != xf || pyf != yf || pzf != zf || pce != ceq;
  const unsigned heads = __ballot_sync(kFull, head);
  bool issue = valid;
  if (__popc(heads) <= kMergeMaxRuns) {
    const unsigned above = heads & ~((2u << lane) - 1u);       // heads strictly above this lane
    const int next_head = above != 0 ? __ffs(above) - 1 : 32;  // first lane of the next run
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const bool take = lane + d < next_head;
      if (!__any_sync(kFull, take)) break;
#pragma unroll
      for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int j = 0; j < F; ++j) {
          const float t = __shfl_down_sync(kFull, v[k][j], d);
          if (take) v[k][j] += t;  // one predicated FADD
        }
    }
    issue = valid && head;
  }
  if (issue) scatter_corners<F>(plan, l, log2_size, xf, yf, zf, xc, yc, zc, c.row, v, dtable, spread);
}

// Dense-lattice replicas for the coarse levels: copies ~ table rows / lattice vertices, at most 32 MiB per level
// (DESIGN.md section 4).  Levels whose lattice is not much smaller than the table get none.
inline int64_t plan_hash_bwd(const nrb_grid_t* grid, int64_t M, BwdPlan* plan) {
  constexpr double kMaxBytesPerLevel = 32.0 * 1024 * 1024;
  const int F = grid->features_per_level;
  const double table_rows = static_cast<double>(int64_t{1} << grid->log2_hashmap_size);
  int64_t floats = 0;
  for (int l = 0; l < NRB_MAX_LEVELS; ++l) {
    plan->copies[l] = 0;
    plan->offset[l] = 0;
    plan->stride[l] = 0;
    plan->r1[l] = 0;
    if (l >= grid->num_levels || M < (int64_t{1} << 16)) continue;
    const int64_t r1 = static_cast<int64_t>(grid->scalings[l]) + 1;
    const double verts = static_cast<double>(r1) * r1 * r1;
    if (verts * 1.5 > table_rows || r1 > 1024) continue;  // the level already spreads over (most of) the table
    const int64_t per_copy = (r1 * r1 * r1 * F + 3) & ~int64_t{3};
    int copies = std::min(static_cast<int>(table_rows / verts + 0.5), 1024);
    while (copies > 1 && static_cast<double>(copies) * per_copy * 4 > kMaxBytesPerLevel) --copies;
    if (copies <= 1) continue;
    plan->copies[l] = copies;
    plan->stride[l] = per_copy;
    plan->offset[l] = floats;
    plan->r1[l] = static_cast<int>(r1);
    floats += static_cast<int64_t>(copies) * per_copy;
    floats = (floats + 3) & ~int64_t{3};
  }
  return floats * 4;
}

// Host side of a backward launch: plan, zero the workspace, return the number of lattice vertices to fold (0: none).
inline int prepare_bwd_plan(const nrb_grid_t* grid, int64_t M, void* workspace, int64_t workspace_bytes, cudaStream_t s,
                            BwdPlan* plan, int64_t* vertices) {
  const int64_t need = plan_hash_bwd(grid, M, plan);
  *vertices = 0;
  if (need > 0 && workspace != nullptr && workspace_bytes >= need && aligned16(workspace)) {
    plan->scratch = static_cast<float*>(workspace);
    cudaError_t e = cudaMemsetAsync(workspace, 0, static_cast<size_t>(need), s);
    NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "backward workspace memset failed: %s", cudaGetErrorString(e));
    for (int l = 0; l < grid->num_levels; ++l)
      if (plan->copies[l] > 1) *vertices += static_cast<int64_t>(plan->r1[l]) * plan->r1[l] * plan->r1[l];
  } else {  // no (or too small a) workspace: every level scatters straight into the table
    plan->scratch = nullptr;
    for (int l = 0; l < NRB_MAX_LEVELS; ++l) plan->copies[l] = 0;
  }
  return NRB_OK;
}

// Adds the replicas of every replicated level into the table (hash_grid.cu); nothing to do when `vertices` is 0.
void launch_fold(const nrb_grid_t* grid, const BwdPlan& plan, float* dtable, int64_t vertices, cudaStream_t s);

}  // namespace nrb
