// Dynamic-actor hash grids: device-side description and the per-sample gather shared by the fused field kernels.
// Semantics: NeuRADHashEncoding's actor branch on the reference's torch path - one 3-D HashEncoding per actor
// (nerfstudio/field_components/neurad_encoding.py:112-119,295-307), features zero-padded to the scene width and written
// over the static ones (:186-187).
#pragma once

#include "common.cuh"

namespace nrb {

constexpr int kActorLevels = 4;    // ActorSettings defaults (neurad_encoding.py:50-68): 4 levels x 4 features
constexpr int kActorFeatures = 4;

struct ActorGridsDev {
  const float* tables[NRB_MAX_ACTORS];  // actor_grids.{i}.hash_table, [4 * 2^log2_size, 4] each
  float scalings[kActorLevels];
  int log2_size;
  int num_grids;
};

struct ActorSamplesDev {
  const int32_t* grid_id;  // [M] actor grid of the sample, -1 = static world
  const float* pos;        // [M,3] position in the actor grid's unit cube (box frame, flipped, contracted)
  const float* std;        // [M] contracted standard deviation
  const float* dirs;       // [M,3] view direction in the box frame, normalised
};

inline ActorGridsDev to_dev(const nrb_actor_grids_t* g) {
  ActorGridsDev d{};
  for (int i = 0; i < NRB_MAX_ACTORS; ++i) d.tables[i] = i < g->num_grids ? g->tables[i] : nullptr;
  for (int l = 0; l < kActorLevels; ++l) d.scalings[l] = g->scalings[l];
  d.log2_size = g->log2_hashmap_size;
  d.num_grids = g->num_grids;
  return d;
}

inline int check_actor_grids(const char* who, const nrb_actor_grids_t* g) {
  NRB_REQUIRE(g != nullptr, NRB_ERR_BAD_ARG, "%s: null actor grids", who);
  NRB_REQUIRE(g->num_grids >= 1 && g->num_grids <= NRB_MAX_ACTORS, NRB_ERR_UNSUPPORTED, "%s: %d actor grids (1..%d supported)",
              who, g->num_grids, NRB_MAX_ACTORS);
  NRB_REQUIRE(g->num_levels == kActorLevels && g->features_per_level == kActorFeatures, NRB_ERR_UNSUPPORTED,
              "%s: actor grids must have %d levels x %d features", who, kActorLevels, kActorFeatures);
  NRB_REQUIRE(g->log2_hashmap_size >= 1 && g->log2_hashmap_size <= 24, NRB_ERR_BAD_ARG, "%s: bad log2_hashmap_size", who);
  for (int i = 0; i < g->num_grids; ++i)
    NRB_REQUIRE(g->tables[i] != nullptr && aligned16(g->tables[i]), NRB_ERR_BAD_ARG, "%s: actor table %d null or unaligned", who, i);
  return NRB_OK;
}

// A world-space point in the frame of one actor box, m = world2boxes[n,a] [3,4] row-major: the rotation as a dot product,
// then the translation (transform_points_pairwise, cameras/lidars.py:507-519).  Shared by the assignment and its
// derivative, so that the pose gradient is taken at exactly the point the forward classified and contracted.
__device__ __forceinline__ float3 to_box_frame(const float* m, const Gaussian& w) {
  const float x = add(fmaf(m[2], w.z, fmaf(m[1], w.y, mul(m[0], w.x))), m[3]);
  const float y = add(fmaf(m[6], w.z, fmaf(m[5], w.y, mul(m[4], w.x))), m[7]);
  const float z = add(fmaf(m[10], w.z, fmaf(m[9], w.y, mul(m[8], w.x))), m[11]);
  return make_float3(x, y, z);
}

// The 16 features of one actor sample (4 levels x 4 features, anti-alias weighted); the caller zero-pads to 32.
__device__ __forceinline__ void actor_gather16(const ActorGridsDev& ag, int gid, float px, float py, float pz, float sd,
                                               float (&out)[16]) {
  const float* table = ag.tables[gid];
  const uint32_t mask = (1u << ag.log2_size) - 1u;
#pragma unroll
  for (int l0 = 0; l0 < kActorLevels; l0 += 2) {  // two levels' 16 corner rows in flight at a time
    Cell c[2];
    float f[2][8][4];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      c[i] = locate_cell(px, py, pz, ag.scalings[l0 + i], mask);
      const float* base = table + (static_cast<size_t>(l0 + i) << ag.log2_size) * 4;
#pragma unroll
      for (int k = 0; k < 8; ++k) load_row<4>(base, c[i].row[k], f[i][k]);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float ax = c[i].ox, bx = 1.0f - c[i].ox, ay = c[i].oy, by = 1.0f - c[i].oy, az = c[i].oz, bz = 1.0f - c[i].oz;
      const float w = level_weight(ag.scalings[l0 + i], sd);
#pragma unroll
      for (int j = 0; j < 4; ++j) {  // lerp order of encodings.py:454-464, as common.cuh:interpolate
        const float f03 = f[i][0][j] * ax + f[i][3][j] * bx;
        const float f12 = f[i][1][j] * ax + f[i][2][j] * bx;
        const float f56 = f[i][5][j] * ax + f[i][6][j] * bx;
        const float f47 = f[i][4][j] * ax + f[i][7][j] * bx;
        const float f0312 = f03 * ay + f12 * by;
        const float f4756 = f47 * ay + f56 * by;
        out[(l0 + i) * 4 + j] = (f0312 * az + f4756 * bz) * w;
      }
    }
  }
}

// Degree-4 real spherical harmonics of (d + 1) / 2 (sh_encoding.cu), for samples whose direction is not the ray's
__device__ __forceinline__ void sh16_of_direction(float dx, float dy, float dz, float (&o)[16]) {
  const float x = (dx + 1.0f) * 0.5f, y = (dy + 1.0f) * 0.5f, z = (dz + 1.0f) * 0.5f;
  const float xx = x * x, yy = y * y, zz = z * z;
  o[0] = 0.28209479177387814f;
  o[1] = 0.4886025119029199f * y;
  o[2] = 0.4886025119029199f * z;
  o[3] = 0.4886025119029199f * x;
  o[4] = 1.0925484305920792f * x * y;
  o[5] = 1.0925484305920792f * y * z;
  o[6] = 0.9461746957575601f * zz - 0.31539156525251999f;
  o[7] = 1.0925484305920792f * x * z;
  o[8] = 0.5462742152960396f * (xx - yy);
  o[9] = 0.5900435899266435f * y * (3.0f * xx - yy);
  o[10] = 2.890611442640554f * x * y * z;
  o[11] = 0.4570457994644658f * y * (5.0f * zz - 1.0f);
  o[12] = 0.3731763325901154f * z * (5.0f * zz - 3.0f);
  o[13] = 0.4570457994644658f * x * (5.0f * zz - 1.0f);
  o[14] = 1.445305721320277f * z * (xx - yy);
  o[15] = 0.5900435899266435f * x * (xx - 3.0f * yy);
}

}  // namespace nrb
