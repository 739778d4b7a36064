// Shared device helpers and launch plumbing for libneuradar_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "neuradar_b200.h"

namespace nrb {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---- host side -----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch();
int finish_launch(const char* what);  // cudaGetLastError -> return code, records the message

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

#define NRB_REQUIRE(cond, code, ...) \
  do {                               \
    if (!(cond)) {                   \
      ::nrb::set_error(__VA_ARGS__); \
      return (code);                 \
    }                                \
  } while (0)

int check_grid(const nrb_grid_t* g);
int check_rays(const nrb_rays_t* r);
int check_intervals(const char* who, const nrb_intervals_t* iv);

// Grid sizes for element-wise kernels: plain ceil-div (the hot kernels size themselves in multiples of the SM count).
inline unsigned blocks_for(int64_t work, int threads) { return static_cast<unsigned>((work + threads - 1) / threads); }
int sm_count();
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize), issued once per (device, kernel): the attribute is sticky, and the call is
// not permitted while a stream is being captured into a CUDA graph.
cudaError_t ensure_dynamic_smem(const void* kernel, int bytes);

// ---- device side ---------------------------------------------------------------------------------------------
// Geometry feeds integer outputs (hash-table rows), so it is evaluated with explicitly rounded fp32 operations in
// the exact order of the reference's torch expressions; the compiler must not contract them into FMAs.
__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }

constexpr float kThird = 0.333333343267440796f;  // float(1/3): torch evaluates x.pow(1/3) with an fp32 exponent

struct Gaussian {
  float x, y, z;  // contracted mean in [0,1]^3
  float std;      // contracted standard deviation
};

// ScaledSceneContraction(order=inf, scale) on GaussiansStd with normalize=True (spatial_distortions.py:103-113,132-136):
// world-space mean / std -> the hash grid's unit cube.
__device__ __forceinline__ Gaussian contract_gaussian(float mx, float my, float mz, float std, float scale) {
  mx = div(mx, scale);
  my = div(my, scale);
  mz = div(mz, scale);
  std = div(std, scale);
  const float mag = fmaxf(fmaxf(fabsf(mx), fabsf(my)), fabsf(mz));
  if (!(mag < 1.0f)) {
    const float cm = fmaxf(mag, 1.0f);
    const float k = sub(2.0f, div(1.0f, cm));
    mx = mul(k, div(mx, cm));
    my = mul(k, div(my, cm));
    mz = mul(k, div(mz, cm));
    const float r = div(powf(sub(mul(2.0f, cm), 1.0f), kThird), cm);
    std = mul(std, mul(r, r));
  }
  Gaussian g;
  g.x = mul(add(mx, 2.0f), 0.25f);
  g.y = mul(add(my, 2.0f), 0.25f);
  g.z = mul(add(mz, 2.0f), 0.25f);
  g.std = mul(std, 0.25f);
  return g;
}

// Frustums.get_fast_isotropic_gaussian(1) (cameras/rays.py:109-124): world-space mean and standard deviation of a sample
__device__ __forceinline__ Gaussian world_gaussian(float ox, float oy, float oz, float dx, float dy, float dz,
                                                   float pixel_area, float start, float end) {
  const float dist = mul(sub(end, start), 0.5f);
  const float t = add(start, dist);
  Gaussian g;
  g.x = add(ox, mul(dx, t));
  g.y = add(oy, mul(dy, t));
  g.z = add(oz, mul(dz, t));
  const float area = mul(pixel_area, mul(t, t));
  g.std = powf(mul(area, dist), kThird);
  return g;
}

// ... followed by the contraction
__device__ __forceinline__ Gaussian sample_gaussian(float ox, float oy, float oz, float dx, float dy, float dz,
                                                    float pixel_area, float start, float end, float scale) {
  const Gaussian w = world_gaussian(ox, oy, oz, dx, dy, dz, pixel_area, start, end);
  return contract_gaussian(w.x, w.y, w.z, w.std, scale);
}

// 1 / max(1, 2*scal*std): neurad_encoding.py:314  ((scalings * 2) * std).clamp_min(1)
__device__ __forceinline__ float level_weight(float scal, float std) {
  return div(1.0f, fmaxf(mul(mul(scal, 2.0f), std), 1.0f));
}

constexpr uint32_t kPrimeY = 2654435761u;
constexpr uint32_t kPrimeZ = 805459861u;

// One level of HashEncoding.pytorch_fwd (encodings.py:428-443): cell corners, in-cell offsets and the 8 table rows
// (relative to the level's first row) in the reference's corner order
//   0:(c,c,c) 1:(c,f,c) 2:(f,f,c) 3:(f,c,c) 4:(c,c,f) 5:(c,f,f) 6:(f,f,f) 7:(f,c,f).
// int64 hashing with Python modulo in the reference == uint32 wrap-around and a mask for power-of-two tables.
struct Cell {
  uint32_t row[8];
  float ox, oy, oz;
};

__device__ __forceinline__ Cell locate_cell(float px, float py, float pz, float scal, uint32_t mask) {
  const float sx = mul(px, scal), sy = mul(py, scal), sz = mul(pz, scal);
  const float fx = floorf(sx), fy = floorf(sy), fz = floorf(sz);
  Cell c;
  c.ox = sub(sx, fx);
  c.oy = sub(sy, fy);
  c.oz = sub(sz, fz);
  const uint32_t xf = static_cast<uint32_t>(static_cast<int32_t>(fx));
  const uint32_t xc = static_cast<uint32_t>(static_cast<int32_t>(ceilf(sx)));
  const uint32_t yf = static_cast<uint32_t>(static_cast<int32_t>(fy)) * kPrimeY;
  const uint32_t yc = static_cast<uint32_t>(static_cast<int32_t>(ceilf(sy))) * kPrimeY;
  const uint32_t zf = static_cast<uint32_t>(static_cast<int32_t>(fz)) * kPrimeZ;
  const uint32_t zc = static_cast<uint32_t>(static_cast<int32_t>(ceilf(sz))) * kPrimeZ;
  c.row[0] = (xc ^ yc ^ zc) & mask;
  c.row[1] = (xc ^ yf ^ zc) & mask;
  c.row[2] = (xf ^ yf ^ zc) & mask;
  c.row[3] = (xf ^ yc ^ zc) & mask;
  c.row[4] = (xc ^ yc ^ zf) & mask;
  c.row[5] = (xc ^ yf ^ zf) & mask;
  c.row[6] = (xf ^ yf ^ zf) & mask;
  c.row[7] = (xf ^ yc ^ zf) & mask;
  return c;
}

// Trilinear weights of the 8 corners in the same order (products of o / 1-o factors, encodings.py:454-464).
__device__ __forceinline__ void corner_weights(const Cell& c, float w[8]) {
  const float ax = c.ox, bx = 1.0f - c.ox, ay = c.oy, by = 1.0f - c.oy, az = c.oz, bz = 1.0f - c.oz;
  w[0] = ax * ay * az;
  w[1] = ax * by * az;
  w[2] = bx * by * az;
  w[3] = bx * ay * az;
  w[4] = ax * ay * bz;
  w[5] = ax * by * bz;
  w[6] = bx * by * bz;
  w[7] = bx * ay * bz;
}

template <int F>
struct Feat;
template <>
struct Feat<1> {
  using type = float;
};
template <>
struct Feat<2> {
  using type = float2;
};
template <>
struct Feat<4> {
  using type = float4;
};

template <int F>
__device__ __forceinline__ void load_row(const float* __restrict__ base, uint32_t row, float v[F]) {
  using V = typename Feat<F>::type;
  const V t = __ldg(reinterpret_cast<const V*>(base) + row);
  if constexpr (F == 1) {
    v[0] = t;
  } else if constexpr (F == 2) {
    v[0] = t.x;
    v[1] = t.y;
  } else {
    v[0] = t.x;
    v[1] = t.y;
    v[2] = t.z;
    v[3] = t.w;
  }
}

// The two rows of an x-corner pair (floor, ceil).  The x prime of the hash is 1, so whenever floor(x) is even the rows
// are r and r ^ 1: one aligned load of twice the width fetches both (the gather kernels are bound by the number of
// L1/TEX requests, not by bytes).
template <int F>
__device__ __forceinline__ void load_x_pair(const float* __restrict__ base, uint32_t row_f, uint32_t row_c, float vf[F],
                                            float vc[F]) {
  // F = 1 only: measured -6 % on the proposal gathers; for F = 2 (16-byte pairs) the divergent paths cost more than
  // the saved requests (+11 % on the main-grid forward)
  if constexpr (F == 1) {
    if (row_c == (row_f ^ 1u)) {
      const bool f_low = (row_f & 1u) == 0;
      const float2 t = __ldg(reinterpret_cast<const float2*>(base) + (row_f >> 1));
      vf[0] = f_low ? t.x : t.y;
      vc[0] = f_low ? t.y : t.x;
      return;
    }
  }
  load_row<F>(base, row_f, vf);
  load_row<F>(base, row_c, vc);
}

// Interpolate one level: lerp order of encodings.py:454-464 (x, then y, then z).
template <int F>
__device__ __forceinline__ void interpolate(const float* __restrict__ level_base, const Cell& c, float out[F]) {
  float f[8][F];
  // x pairs (floor, ceil): (3,0) (2,1) (7,4) (6,5)
  load_x_pair<F>(level_base, c.row[3], c.row[0], f[3], f[0]);
  load_x_pair<F>(level_base, c.row[2], c.row[1], f[2], f[1]);
  load_x_pair<F>(level_base, c.row[7], c.row[4], f[7], f[4]);
  load_x_pair<F>(level_base, c.row[6], c.row[5], f[6], f[5]);
  const float ax = c.ox, bx = 1.0f - c.ox, ay = c.oy, by = 1.0f - c.oy, az = c.oz, bz = 1.0f - c.oz;
#pragma unroll
  for (int j = 0; j < F; ++j) {
    const float f03 = f[0][j] * ax + f[3][j] * bx;
    const float f12 = f[1][j] * ax + f[2][j] * bx;
    const float f56 = f[5][j] * ax + f[6][j] * bx;
    const float f47 = f[4][j] * ax + f[7][j] * bx;
    const float f0312 = f03 * ay + f12 * by;
    const float f4756 = f47 * ay + f56 * by;
    out[j] = f0312 * az + f4756 * bz;
  }
}

// Gradient of one level's interpolated features with respect to the point's scaled position (x * scal), contracted
// with the upstream values g: the derivative of `interpolate` above.  Multiply by the level's scaling for the point.
template <int F>
__device__ __forceinline__ float3 position_grad(const float* __restrict__ level_base, const Cell& c, const float (&g)[F]) {
  float f[8][F];
#pragma unroll
  for (int k = 0; k < 8; ++k) load_row<F>(level_base, c.row[k], f[k]);
  const float ax = c.ox, bx = 1.0f - c.ox, ay = c.oy, by = 1.0f - c.oy, az = c.oz, bz = 1.0f - c.oz;
  float gx = 0.f, gy = 0.f, gz = 0.f;
#pragma unroll
  for (int j = 0; j < F; ++j) {
    const float f03 = f[0][j] * ax + f[3][j] * bx, f12 = f[1][j] * ax + f[2][j] * bx;
    const float f56 = f[5][j] * ax + f[6][j] * bx, f47 = f[4][j] * ax + f[7][j] * bx;
    const float f0312 = f03 * ay + f12 * by, f4756 = f47 * ay + f56 * by;
    gz += g[j] * (f0312 - f4756);
    gy += g[j] * ((f03 - f12) * az + (f47 - f56) * bz);
    gx += g[j] * (((f[0][j] - f[3][j]) * ay + (f[1][j] - f[2][j]) * by) * az +
                  ((f[4][j] - f[7][j]) * ay + (f[5][j] - f[6][j]) * by) * bz);
  }
  return make_float3(gx, gy, gz);
}

// The fused field backward's data-gradient tile image: [tile of 128 samples][8 chunks of 4 features][128 samples]
// float4.  Returns features 4c .. 4c+3 of sample m; a warp of consecutive samples reads 16-byte-strided, i.e. coalesced.
__device__ __forceinline__ const float* tile_image_chunk(const float* img, int64_t m, int c) {
  return img + ((m >> 7) * 1024 + (m & 127)) * 4 + c * 512;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

__device__ __forceinline__ float warp_inclusive_sum(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

__device__ __forceinline__ double warp_inclusive_sum(double v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double n = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

__device__ __forceinline__ float warp_inclusive_prod(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v *= n;
  }
  return v;
}

// torch.nan_to_num defaults: nan -> 0, +inf -> FLT_MAX, -inf -> -FLT_MAX
__device__ __forceinline__ float nan_to_num(float v) {
  if (isnan(v)) return 0.0f;
  if (isinf(v)) return v > 0 ? 3.402823466e+38f : -3.402823466e+38f;
  return v;
}

// power_fn / inv_power_fn of utils/math.py:541-580 for finite lambda not in {0, 1}.
__device__ __forceinline__ float power_fn(float x, float lam) {
  const float lam1 = fabsf(lam - 1.0f);
  const float base = add(div(x, lam1), 1.0f);
  const float p = (lam == -1.0f) ? div(1.0f, base) : powf(base, lam);
  return mul(div(lam1, lam), sub(p, 1.0f));
}

__device__ __forceinline__ float inv_power_fn(float x, float lam) {
  const float lam1 = fabsf(lam - 1.0f);
  const float base = fmaxf(add(div(mul(x, lam), lam1), 1.0f), 1e-10f);
  const float p = (lam == -1.0f) ? div(1.0f, base) : powf(base, div(1.0f, lam));
  return mul(sub(p, 1.0f), lam1);
}

// spacing_to_euclidean_fn of SpacedSampler (ray_samplers.py:117-120) composed with PowerSampler's inverse.
__device__ __forceinline__ float spacing_to_euclidean(float s, float s_near, float s_far, nrb_spacing_t sp) {
  const float v = add(mul(s, s_far), mul(sub(1.0f, s), s_near));
  return div(inv_power_fn(v, sp.lambda), sp.scaling);
}

}  // namespace nrb
