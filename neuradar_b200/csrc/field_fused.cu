// NeuRAD field, fused: hash-grid gather -> geometry MLP -> feature MLP (forward), and its backward with the
// activations RECOMPUTED on the tensor cores instead of saved.
// Semantics: NeuRADHashEncoding.forward + NeuRADField.forward (nerfstudio/field_components/neurad_encoding.py:152-189,
// 309-316; nerfstudio/fields/neurad_field.py:128-152; nerfstudio/field_components/encodings.py:425-466;
// nerfstudio/field_components/mlp.py:159-178; nerfstudio/model_components/utils.py:30-41).
//
// Measured on B200 with tools/mma_probe.cu (round 2), the facts this design rests on:
//   * one thread needs ~55 (kind::tf32) / ~85 (kind::f16) cycles to ISSUE one small tcgen05.mma (M 128, N 32..64); the
//     tensor pipe itself takes 16 (N = 32) .. 32 (N = 64) cycles when A comes from tensor memory and ~40 when A is read
//     from shared memory (128 B/cycle): with 4 issuing warps the pipe floor is reached.  Hence: several independent
//     128-sample tiles in flight per SM, each with its own issuing thread, and A operands in TMEM (".ts") wherever the
//     thread that owns a row can put it there;
//   * bf16 operands may be MN-major in shared memory (tf32 may not: all-zero accumulators), and a K-major image is the
//     MN-major image of the transposed matrix.  So ONE shared-memory image of an activation / delta tile serves the
//     weight-gradient GEMM (reduction over the 128 samples) with no transposes, and ONE image of each weight matrix
//     serves the forward recompute (K-major) and the data-gradient GEMM (MN-major);
//   * 16-bit A operands in TMEM are packed two per column (even element in the low half);
//   * an M = 64 accumulator uses lanes 0..15 of every 32-lane quarter; a second one can live at lane offset 16.
//
// Forward (field_fused_fwd_kernel): three groups of 128 threads per CTA, thread = sample.  Each thread gathers the 16
// levels of its sample straight into the layer-0 A operand in tensor memory (tf32 hi / lo; the [M,32] hash features never
// reach HBM in inference), runs the five layers as 3xTF32 tcgen05.mma with fp32 accumulation in TMEM, and writes
// feature / sdf / alpha.  In training it also leaves the bf16 hi / mid operand image of the hash features (16 KB per
// tile) and one ReLU bit mask per hidden layer: 140 B per sample instead of the 524 B of saved activations before.
//
// Backward (field_fused_bwd_kernel): two tiles in flight per CTA (2 x 128 worker threads) + five issuing warps, one per
// layer, for the weight-gradient GEMMs.  Per tile: recompute h1, emb, g1, g2 with the saved masks (bf16 hi / mid, three
// partial products, A via TMEM); every activation is written ONCE as a bf16 image that is the B operand of its layer's
// weight-gradient GEMM; then the delta chain runs back through the layers (A = delta via TMEM, B = the same weight
// images, MN-major), each delta also written once as the A image of the weight-gradient GEMM.  dW / db accumulate in
// TMEM across all tiles of the CTA (M = 64 accumulators, two per column range) and are flushed once.
#include <algorithm>
#include <cstdlib>

#include <cuda.h>
#include <cuda_bf16.h>

#include "actor_grid.cuh"
#include "hash_bwd_plan.cuh"
#include "tc_common.cuh"

namespace nrb {

using namespace tc;

struct FusedParams {
  const float* w[5];  // mlp_geo.layers.{0,1}.weight, mlp_feature.layers.{0,1,2}.weight   ([out, in] row-major)
  const float* b[5];
  const float* beta;  // sdf_to_density.beta [1]
  float beta_min;
};

__device__ constexpr int kLK[5] = {32, 32, 48, 32, 32};    // layer input width
__device__ constexpr int kLN[5] = {32, 48, 32, 32, 32};    // forward accumulator width (outputs padded to 16)
__device__ constexpr int kLOut[5] = {32, 33, 32, 32, 32};  // rows of the weight matrix

// ---------------------------------------------------------------------------------------------------------------
// shared helpers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void group_barrier(int g) { asm volatile("bar.sync %0, 128;" ::"r"(g + 1) : "memory"); }

// two consecutive features -> one packed bf16 word of the hi part (round to nearest) and of the residual
__device__ __forceinline__ void split_bf16_pair(float a0, float a1, uint32_t& hi, uint32_t& mid) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(a1), "f"(a0));
  const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xFFFF0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(mid) : "f"(a1 - h1), "f"(a0 - h0));
}

__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3])
               : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
}

// bulk asynchronous copy global -> shared (TMA engine, UBLKCP), completion counted on an mbarrier
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(mbar))
               : "memory");
}

__device__ __forceinline__ void mma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(static_cast<uint32_t>(acc))
      : "memory");
}

__device__ __forceinline__ void mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(static_cast<uint32_t>(acc))
      : "memory");
}

// kind::f16 instruction descriptor: bf16 x bf16 -> fp32
__device__ __forceinline__ uint32_t idesc_bf16(int m, int n, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

// ---------------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------------
constexpr int kFGroups = 3;
constexpr int kFThreads = kFGroups * kRows;
constexpr int kFCols = 144;  // TMEM columns per group: accumulator [0,48) | A hi [48,96) | A lo [96,144)
constexpr int kFAcc = 0, kFAHi = 48, kFALo = 96;

__host__ __device__ constexpr int ff_w_floats(int l) { return l == 0 ? 32 * 32 : l == 1 ? 48 * 32 : l == 2 ? 32 * 48 : 32 * 32; }
__host__ __device__ constexpr int ff_w_hi(int l) {
  int o = 0;
  for (int i = 0; i < l; ++i) o += 2 * ff_w_floats(i) * 4;
  return o;
}
__host__ __device__ constexpr int ff_w_lo(int l) { return ff_w_hi(l) + ff_w_floats(l) * 4; }

struct FusedFwdSmem {
  static constexpr int bias = ff_w_hi(5);                    // 5 x 48 floats
  static constexpr int bounce = bias + 5 * 48 * 4;           // one 4 KB row-I/O buffer per warp
  static constexpr int mbar = bounce + (kFThreads / 32) * 4096;
  static constexpr int tmem = mbar + 8 * kFGroups;
  static constexpr int total = tmem + 16;
};

struct FusedFwdArgs {
  const float* xyz;   // [M,3] contracted sample means (gather mode, F > 0)
  const float* std;   // [M] contracted standard deviations or null
  const float* x;     // [M,32] hash features (F == 0)
  const float* sh;    // [rays,16]
  int samples_per_ray;
  int64_t M;
  float* feature;     // [M,32]
  float* sdf;         // [M]
  float* alpha;       // [M]
  uint4* ximg;        // training: bf16 hi / mid operand image of the hash features, 16 KB per tile
  uint32_t* masks;    // training: [3][ld] ReLU bit masks of h1, g1, g2
  int64_t ld;
  ActorGridsDev ag;   // kActors: per-actor tables and the per-sample assignment (actors.cu)
  ActorSamplesDev as;
};

template <int F, bool kActors>
__global__ void __launch_bounds__(kFThreads, 1) field_fused_fwd_kernel(const __grid_constant__ FusedParams prm,
                                                                       const __grid_constant__ GridDev grid,
                                                                       const __grid_constant__ FusedFwdArgs a) {
  extern __shared__ __align__(128) char smem[];
  const int t = threadIdx.x, lane = t & 31, r = t & (kRows - 1);
  const int uwarp = uniform_warp_idx();
  const int g = uwarp >> 2;
  float* s_bias = reinterpret_cast<float*>(smem + FusedFwdSmem::bias);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + FusedFwdSmem::mbar) + g;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + FusedFwdSmem::tmem);
  char* bounce = smem + FusedFwdSmem::bounce + uwarp * 4096;

  for (int l = 0; l < 5; ++l) {
    stage_weight_split(prm.w[l], kLOut[l], kLN[l], kLK[l], smem + ff_w_hi(l), smem + ff_w_lo(l));
    for (int j = t; j < 48; j += kFThreads) s_bias[l * 48 + j] = (j < kLOut[l] && prm.b[l] != nullptr) ? __ldg(prm.b[l] + j) : 0.0f;
  }
  if (uwarp == 0) tmem_alloc<512>(tmem_slot);
  if (t == 0)
    for (int i = 0; i < kFGroups; ++i) mbar_init(reinterpret_cast<uint64_t*>(smem + FusedFwdSmem::mbar) + i, 1);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tg = *tmem_slot + static_cast<uint32_t>(g * kFCols);
  const uint32_t lane_base = tg + (static_cast<uint32_t>((uwarp & 3) * 32) << 16);
  const float beta = fabsf(__ldg(prm.beta)) + prm.beta_min;
  const bool train = a.ximg != nullptr;
  uint32_t phase = 0;

  auto run_layer = [&](int l) {
    fence_before_sync();
    group_barrier(g);
    if ((uwarp & 3) == 0) {
      if (elect_one()) {
        fence_after_sync();
        issue_gemm_ts(tg + kFAcc, kLN[l], tg + kFAHi, tg + kFALo, smem_u32(smem + ff_w_hi(l)), smem_u32(smem + ff_w_lo(l)),
                      kLK[l], kLK[l]);
        mma_commit(mbar);
      }
      __syncwarp();
    }
    mbar_wait(mbar, phase);
    phase ^= 1;
    fence_after_sync();
  };

  const int64_t tiles = (a.M + kRows - 1) / kRows;
  for (int64_t tile = blockIdx.x + static_cast<int64_t>(g) * gridDim.x; tile < tiles;
       tile += static_cast<int64_t>(kFGroups) * gridDim.x) {
    const int64_t row = tile * kRows + r;
    const bool ok = row < a.M;
    const int64_t rr = ok ? row : (a.M - 1);  // rows past the end compute on a valid row; nothing of theirs is stored
    // ---- layer-0 input: gather the levels (HashEncoding.pytorch_fwd + _rescale_grid_features) or read the given rows.
    // All 32 values are produced before anything is staged so that the compiler can keep the gathers of several levels
    // in flight (the tensor-memory stores below are ordering points for it).
    float v[32];
    int agid = -1;  // actor grid of this sample (-1: static world)
    if constexpr (kActors) agid = __ldg(a.as.grid_id + rr);
    if (kActors && agid >= 0) {
      // a sample inside an actor box: 16 features of that actor's grid, zero-padded, replace the static ones
      // (neurad_encoding.py:181-187)
      float o16[16];
      actor_gather16(a.ag, agid, __ldg(a.as.pos + 3 * rr), __ldg(a.as.pos + 3 * rr + 1), __ldg(a.as.pos + 3 * rr + 2),
                     __ldg(a.as.std + rr), o16);
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        v[j] = o16[j];
        v[16 + j] = 0.0f;
      }
    } else if constexpr (F > 0) {
      const float px = __ldg(a.xyz + 3 * rr), py = __ldg(a.xyz + 3 * rr + 1), pz = __ldg(a.xyz + 3 * rr + 2);
      const float sd = a.std != nullptr ? __ldg(a.std + rr) : 0.0f;
      const uint32_t hmask = (1u << grid.log2_size) - 1u;
      // kBatch levels at a time: all their 8 x kBatch corner rows are requested before the first one is used (the
      // tables are L2 resident: ~300-600 cycles per request, and only 12 warps per SM are there to hide it)
      constexpr int kBatch = 8 / F;
#pragma unroll
      for (int l0 = 0; l0 < 32 / F; l0 += kBatch) {
        Cell c[kBatch];
        float f[kBatch][8][F];
#pragma unroll
        for (int i = 0; i < kBatch; ++i) {
          c[i] = locate_cell(px, py, pz, grid.scalings[l0 + i], hmask);
          const float* base = grid.table + (static_cast<size_t>(l0 + i) << grid.log2_size) * F;
#pragma unroll
          for (int k = 0; k < 8; ++k) load_row<F>(base, c[i].row[k], f[i][k]);
        }
#pragma unroll
        for (int i = 0; i < kBatch; ++i) {
          const float ax = c[i].ox, bx = 1.0f - c[i].ox, ay = c[i].oy, by = 1.0f - c[i].oy, az = c[i].oz, bz = 1.0f - c[i].oz;
          const float w = a.std != nullptr ? level_weight(grid.scalings[l0 + i], sd) : 1.0f;
#pragma unroll
          for (int j = 0; j < F; ++j) {  // lerp order of encodings.py:454-464 (x, then y, then z), as common.cuh:interpolate
            const float f03 = f[i][0][j] * ax + f[i][3][j] * bx;
            const float f12 = f[i][1][j] * ax + f[i][2][j] * bx;
            const float f56 = f[i][5][j] * ax + f[i][6][j] * bx;
            const float f47 = f[i][4][j] * ax + f[i][7][j] * bx;
            const float f0312 = f03 * ay + f12 * by;
            const float f4756 = f47 * ay + f56 * by;
            v[(l0 + i) * F + j] = (f0312 * az + f4756 * bz) * w;
          }
        }
      }
    } else {
      float4 pf[8];
      warp_load_rows_coalesced(a.x, tile * kRows + (uwarp & 3) * 32, a.M, lane, pf);
      warp_bounce_to_rows(bounce, lane, pf, v);
    }
    // tf32 hi / lo into the A operand, bf16 hi / mid into the saved image
    tmem_store_row_split<32>(tg, uwarp, kFAHi, kFALo, 0, v);
    if (train) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t h[4], m[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) split_bf16_pair(v[8 * q + 2 * c], v[8 * q + 2 * c + 1], h[c], m[c]);
        uint4* dst = a.ximg + tile * 1024 + q * 128 + r;
        dst[0] = make_uint4(h[0], h[1], h[2], h[3]);
        dst[512] = make_uint4(m[0], m[1], m[2], m[3]);
      }
    }
    auto relu_mask = [&](const float* bias) {
      uint32_t m = 0;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        v[j] = fmaxf(v[j] + bias[j], 0.0f);
        m |= (v[j] > 0.0f ? 1u : 0u) << j;
      }
      return m;
    };
    // ---- mlp_geo layer 0: 32 -> 32, ReLU
    run_layer(0);
    tmem_load_row<32>(tg + kFAcc, uwarp, 0, v);
    const uint32_t m_h1 = relu_mask(s_bias);
    tmem_store_row_split<32>(tg, uwarp, kFAHi, kFALo, 0, v);
    // ---- mlp_geo layer 1: 32 -> 33 (sdf | embedding), no activation
    run_layer(1);
    float sdf_v;
    float emb[32];
    {
      float geo[48];
      tmem_load_row<48>(tg + kFAcc, uwarp, 0, geo);
      sdf_v = geo[0] + s_bias[48];
#pragma unroll
      for (int j = 0; j < 32; ++j) emb[j] = geo[1 + j] + s_bias[48 + 1 + j];
    }
    // ---- mlp_feature layer 0: [emb | sh] 48 -> 32, ReLU
    tmem_store_row_split<32>(tg, uwarp, kFAHi, kFALo, 0, emb);
    {
      float shv[16];
      if (kActors && agid >= 0) {  // the view direction was rotated into the actor's frame: its own SH basis
        sh16_of_direction(__ldg(a.as.dirs + 3 * rr), __ldg(a.as.dirs + 3 * rr + 1), __ldg(a.as.dirs + 3 * rr + 2), shv);
      } else {
        const float4* shp = reinterpret_cast<const float4*>(a.sh + (rr / a.samples_per_ray) * 16);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float4 q4 = __ldg(shp + c);
          shv[4 * c] = q4.x;
          shv[4 * c + 1] = q4.y;
          shv[4 * c + 2] = q4.z;
          shv[4 * c + 3] = q4.w;
        }
      }
      tmem_store_row_split<16>(tg, uwarp, kFAHi, kFALo, 32, shv);
    }
    run_layer(2);
    tmem_load_row<32>(tg + kFAcc, uwarp, 0, v);
    const uint32_t m_g1 = relu_mask(s_bias + 2 * 48);
    tmem_store_row_split<32>(tg, uwarp, kFAHi, kFALo, 0, v);
    // ---- mlp_feature layer 1: 32 -> 32, ReLU
    run_layer(3);
    tmem_load_row<32>(tg + kFAcc, uwarp, 0, v);
    const uint32_t m_g2 = relu_mask(s_bias + 3 * 48);
    tmem_store_row_split<32>(tg, uwarp, kFAHi, kFALo, 0, v);
    if (train && ok) {
      a.masks[row] = m_h1;
      a.masks[a.ld + row] = m_g1;
      a.masks[2 * a.ld + row] = m_g2;
    }
    // ---- mlp_feature layer 2: 32 -> 32, no activation; residual with the embedding
    run_layer(4);
    tmem_load_row<32>(tg + kFAcc, uwarp, 0, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = emb[j] + (v[j] + s_bias[4 * 48 + j]);
    warp_store_rows_coalesced(a.feature, tile * kRows + (uwarp & 3) * 32, a.M, bounce, lane, v);
    if (ok) {
      a.sdf[row] = sdf_v;
      a.alpha[row] = 1.0f / (1.0f + expf(sdf_v * beta));  // sigmoid(-sdf * beta)
    }
  }
  fence_before_sync();
  __syncthreads();
  if (uwarp == 0) tmem_free<512>(*tmem_slot);
}

// ---------------------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------------------
constexpr int kBGroups = 2;
constexpr int kBWorkers = kBGroups * kRows;  // 256
constexpr int kBIssuers = 1;                 // one polling warp issues every weight-gradient chain
constexpr int kBThreads = kBWorkers + kBIssuers * 32;
// TMEM columns of a group: accumulator [0,32) | A hi [32,56) | A mid [56,80) | delta hi [80,96) | delta mid [96,112)
constexpr int kBCols = 112;
constexpr int kBAcc = 0, kBAHi = 32, kBAMid = 56, kBDHi = 80, kBDMid = 96;
// weight-gradient accumulators (M = 64: 16 lanes per quarter, so two share a column range at lane offsets 0 / 16).
// Columns of one accumulator: [0,K) delta x input hi | K: delta x ones (bias gradient) | [K+8, 2K+8) delta x input mid.
__device__ constexpr int kDwCol[5] = {224, 224, 368, 296, 296};
__device__ constexpr int kDwLane[5] = {0, 16, 0, 0, 16};
constexpr int kSdfCol = 368, kSdfLane = 16;  // sdf row of W1: rows 0 (hi) and 1 (mid) of an accumulator next to layer 2's

// shared-memory map.  An "image" of a [128 samples x J features] bf16 matrix stores feature group q = j / 8 of sample s at
// byte q * 2048 + s * 16 + (j % 8) * 2: K-major with LBO 2048 / SBO 128 when samples are the rows, MN-major with
// LBO 128 / SBO 2048 when samples are the reduction dimension.  An input slot is [hi groups | ones group | mid groups],
// contiguous, so that ONE instruction per 16 samples multiplies delta with [in hi | 1 | in mid] (N = 72 or 104).
struct FusedBwdSmem {
  // per group
  static constexpr int d_hi = 0, d_mid = 8192;                       // delta: 32 hi rows | 32 mid rows = ONE 64-row operand
  static constexpr int d_sdf = 16384;                                // one more group: features (d sdf hi, d sdf mid, 0 ..)
  static constexpr int d_bytes = 18432;                              // (the first 16 KB are also the landing zone of the d feature tile)
  static constexpr int h1 = d_bytes;                                 // 4 + 1 + 4 groups
  static constexpr int emb = h1 + 18432;                             // 6 + 1 + 6 groups
  static constexpr int g1 = emb + 26624;
  static constexpr int g2x = g1 + 18432;                             // g2, later the hash features x
  static constexpr int group_bytes = g2x + 18432;                    // 100352 = 98 KB
  // shared
  static constexpr int w = kBGroups * group_bytes;                   // weight images [hi | mid] per layer
  static constexpr int w_bytes = 4 * 4096 + 6144;
  static constexpr int w1row0 = w + w_bytes;                         // sdf row of W1, 32 floats
  static constexpr int bias = w1row0 + 128;                          // 5 x 48 floats
  static constexpr int mbar = bias + 5 * 48 * 4;                  // data[2], xfull[2], dfull[2], ready[2][5], done[2][5]
  static constexpr int tmem = mbar + 8 * 26;
  static constexpr int total = tmem + 16;
};
__host__ __device__ constexpr int fb_w_off(int l) { return l <= 2 ? l * 4096 : 4096 * 2 + 6144 + (l - 3) * 4096; }
__host__ __device__ constexpr int fb_w_half(int l) { return l == 2 ? 3072 : 2048; }
__device__ constexpr int kSlotOff[5] = {FusedBwdSmem::g2x, FusedBwdSmem::h1, FusedBwdSmem::emb, FusedBwdSmem::g1,
                                        FusedBwdSmem::g2x};          // input image of layer l
__device__ constexpr int kSlotMid[5] = {10240, 10240, 14336, 10240, 10240};  // offset of the mid half inside the slot

struct FusedBwdArgs {
  const uint4* ximg;
  const uint32_t* masks;
  int64_t ld;
  const float* sh;
  const float* sdf;
  const float* alpha;
  const float* dfeature;   // [M,32] or null (then read through the tensor map)
  const float* dfeat_ray;  // [rays,32]: dfeature[m] = weights[m] * dfeat_ray[m / S] (compositor folded in)
  const float* weights;    // [M]
  const float* dsdf;       // [M] or null
  const float* dalpha;     // [M] or null
  int samples_per_ray;
  int64_t M;
  const int32_t* actor_grid_id;  // [M] or null: samples >= 0 use their own direction's SH basis
  const float* actor_dirs;       // [M,3]
  float4* dximg;           // [tiles][8 chunks][128 rows] float4, or null
  float* dw[5];
  float* db[5];
  float* dbeta;
};

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}

// TMA tile load (UTMALDG): box {32 features, 128 samples} of the row-major [M,32] fp32 matrix behind `map`, 128-byte
// swizzle (16-byte chunk c of row r lands at chunk c ^ (r & 7)), rows past the end of the matrix are filled with zeros
__device__ __forceinline__ void tma_load_rows(void* dst_smem, const CUtensorMap* map, int32_t row0, uint64_t* mbar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst_smem)),
      "l"(map), "r"(0), "r"(row0), "r"(smem_u32(mbar))
      : "memory");
}

#ifdef NRB_FUSED_TRACE
// debug build only (tools/trace_fused_bwd.py): thread 0 of CTA 0 and the layer-4 issuer stamp clock64() at phase boundaries
__device__ long long g_fused_trace[4096];
#define NRB_FT(slot)                                                                                            \
  do {                                                                                                          \
    if (blockIdx.x == 0 && t == 0 && trace_n < 2000) g_fused_trace[trace_n++] = (static_cast<long long>(slot) << 48) | (clock64() & 0xFFFFFFFFFFFFll); \
  } while (0)
#define NRB_FTI(slot)                                                                                           \
  do {                                                                                                          \
    if (blockIdx.x == 0 && uwarp == 8 && itrace_n < 4000) g_fused_trace[itrace_n++] = (static_cast<long long>(slot) << 48) | (clock64() & 0xFFFFFFFFFFFFll); \
  } while (0)
#else
#define NRB_FT(slot)
#define NRB_FTI(slot)
#endif

__global__ void __maxnreg__(128) field_fused_bwd_kernel(const __grid_constant__ FusedParams prm,
                                                                       const __grid_constant__ FusedBwdArgs a,
                                                                       const __grid_constant__ CUtensorMap dfeat_map) {
  extern __shared__ __align__(1024) char smem[];
  const int t = threadIdx.x, lane = t & 31, r = t & (kRows - 1);
  const int uwarp = uniform_warp_idx();
#ifdef NRB_FUSED_TRACE
  int trace_n = 0, itrace_n = 2000;
#endif
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem + FusedBwdSmem::mbar);
  uint64_t* mb_data = mbars;        // [2]
  uint64_t* mb_xfull = mbars + 2;   // [2]
  uint64_t* mb_dfull = mbars + 4;   // [2]
  uint64_t* mb_ready = mbars + 6;   // [2][5]
  uint64_t* mb_done = mbars + 16;   // [2][5]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + FusedBwdSmem::tmem);
  float* s_bias = reinterpret_cast<float*>(smem + FusedBwdSmem::bias);
  float* w1row0 = reinterpret_cast<float*>(smem + FusedBwdSmem::w1row0);

  // ---- one-time staging: weight images (bf16 hi / mid, K-major [out][in]), biases, the ones groups
  for (int l = 0; l < 5; ++l) {
    const int K = kLK[l];
    const float* src = prm.w[l] + (l == 1 ? 32 : 0);  // layer 1: rows 1..32 (embedding outputs); the sdf row is rank 1
    char* hi = smem + FusedBwdSmem::w + fb_w_off(l);
    char* mid = hi + fb_w_half(l);
    for (int e = t; e < 32 * K / 2; e += kBThreads) {
      const int n = e / (K / 2), k = 2 * (e - n * (K / 2));
      uint32_t h, m;
      split_bf16_pair(__ldg(src + n * K + k), __ldg(src + n * K + k + 1), h, m);
      const int off = (n >> 3) * (K / 8) * 128 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2;
      *reinterpret_cast<uint32_t*>(hi + off) = h;
      *reinterpret_cast<uint32_t*>(mid + off) = m;
    }
    for (int j = t; j < 48; j += kBThreads) s_bias[l * 48 + j] = (j < kLOut[l] && prm.b[l] != nullptr) ? __ldg(prm.b[l] + j) : 0.0f;
  }
  if (t < 32) w1row0[t] = __ldg(prm.w[1] + t);
  for (int gq = 0; gq < kBGroups; ++gq) {
    char* base = smem + gq * FusedBwdSmem::group_bytes;
    // ones groups: feature 0 of the group is 1.0 for every sample, features 1..7 are 0
    for (int e = t; e < 4 * 128; e += kBThreads) {
      const int slot = e >> 7, s = e & 127;
      const int off = slot == 0 ? FusedBwdSmem::h1 + 8192 : slot == 1 ? FusedBwdSmem::emb + 12288
                      : slot == 2 ? FusedBwdSmem::g1 + 8192 : FusedBwdSmem::g2x + 8192;
      *reinterpret_cast<uint4*>(base + off + s * 16) = make_uint4(0x00003F80u, 0u, 0u, 0u);
    }
  }
  if (uwarp == 0) tmem_alloc<512>(tmem_slot);
  if (t == 0) {
    for (int i = 0; i < 6; ++i) mbar_init(mbars + i, 1);
    for (int i = 0; i < 10; ++i) mbar_init(mb_ready + i, kRows);
    for (int i = 0; i < 10; ++i) mbar_init(mb_done + i, 1);
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const int64_t tiles = (a.M + kRows - 1) / kRows;
  // tiles of this CTA: blockIdx.x + k * gridDim.x, k = 0 .. mine-1; group g takes k = g, g + 2, ...
  const int64_t mine = static_cast<int64_t>(blockIdx.x) < tiles ? (tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;

  if (uwarp >= 8) {
    // ---- the weight-gradient issuer: ONE warp serves the chains of both groups and all layers (each accumulator is only
    // ever touched by this thread, so the accumulations are ordered).  It polls the two barriers that can fire next - every
    // group walks its layers 4 -> 0 - and backs off with nanosleep when neither has: the chains are short (8 instructions,
    // ~0.4 K cycles) and ~11 of them arrive per ~18 K-cycle tile period.
    // [dW | db | dW'] (+)= delta^T [in hi | 1 | in mid]: A = delta image (32 hi rows and 32 mid rows = one M = 64 operand),
    // B = the layer's input slot, both MN-major (reduction over the 128 samples): ONE instruction per 16 samples gives
    // all four partial products.  With 9 warps at <= 128 registers the CTA leaves a quarter of the register file free, so
    // blocks of the independent proposal-round backward (another stream) co-reside with this latency-bound kernel.
    const int64_t cnt[2] = {(mine + 1) / 2, mine / 2};
    int64_t it[2] = {0, 0};
    int lcur[2] = {4, 4};
    bool pend[2] = {false, false};  // x image to fetch once dW_4 has consumed g2
    uint32_t used = 0;              // accumulators that hold a partial sum already
    while (it[0] < cnt[0] || it[1] < cnt[1] || pend[0] || pend[1]) {
      bool progressed = false;
#pragma unroll
      for (int gq = 0; gq < 2; ++gq) {
        char* gsq = smem + gq * FusedBwdSmem::group_bytes;
        if (pend[gq] && mbar_test(mb_done + gq * 5 + 4, static_cast<uint32_t>(it[gq] & 1))) {
          if (elect_one()) {  // g2 has been consumed: its slot receives the hash-feature image for dW_0 (TMA bulk copy)
            const int64_t tile = blockIdx.x + (2 * it[gq] + gq) * gridDim.x;
            mbar_expect_tx(mb_xfull + gq, 16384);
            bulk_load(gsq + FusedBwdSmem::g2x, a.ximg + tile * 1024, 8192, mb_xfull + gq);
            bulk_load(gsq + FusedBwdSmem::g2x + 10240, a.ximg + tile * 1024 + 512, 8192, mb_xfull + gq);
          }
          __syncwarp();
          pend[gq] = false;
          progressed = true;
        }
        if (it[gq] < cnt[gq] && mbar_test(mb_ready + gq * 5 + lcur[gq], static_cast<uint32_t>(it[gq] & 1))) {
          const int l = lcur[gq];
          if (elect_one()) {
            NRB_FTI(100 + gq);
            fence_after_sync();
            const uint32_t base = smem_u32(gsq);
            const uint32_t d_tmem = tmem_base + (static_cast<uint32_t>(kDwLane[l]) << 16) + static_cast<uint32_t>(kDwCol[l]);
            const uint32_t idesc = idesc_bf16(64, 2 * kLK[l] + 8, 1, 1);
            uint64_t da = make_desc(base + FusedBwdSmem::d_hi, 128, 2048), db = make_desc(base + kSlotOff[l], 128, 2048);
            const bool acc0 = (used >> l) & 1u;
#pragma unroll
            for (int ks = 0; ks < kRows / 16; ++ks) {  // 16 samples per instruction = two 8-sample groups = 256 bytes
              mma_bf16_ss(d_tmem, da, db, idesc, acc0 || ks > 0);
              da += 16;
              db += 16;
            }
            if (l == 1) {  // the sdf row of W1: the same GEMM with the one-group image (d sdf hi, d sdf mid, 0 ..) as A
              const uint32_t s_tmem = tmem_base + (static_cast<uint32_t>(kSdfLane) << 16) + static_cast<uint32_t>(kSdfCol);
              uint64_t sa = make_desc(base + FusedBwdSmem::d_sdf, 128, 2048), sb = make_desc(base + kSlotOff[1], 128, 2048);
#pragma unroll
              for (int ks = 0; ks < kRows / 16; ++ks) {
                mma_bf16_ss(s_tmem, sa, sb, idesc, acc0 || ks > 0);
                sa += 16;
                sb += 16;
              }
            }
            mma_commit(mb_done + gq * 5 + l);
            NRB_FTI(110 + gq);
          }
          __syncwarp();
          used |= 1u << l;
          if (l == 4) pend[gq] = true;
          if (l == 0) {
            lcur[gq] = 4;
            // (a pending x fetch of this tile was served long ago: dW_0 needs the x image)
            ++it[gq];
          } else {
            lcur[gq] = l - 1;
          }
          progressed = true;
        }
      }
      if (!progressed) __nanosleep(64);
    }
  } else {
    // ---- workers: group g = warps 4g .. 4g+3, thread = sample row r of the group's current tile
    const int g = uwarp >> 2, wq = uwarp & 3;
    char* gs = smem + g * FusedBwdSmem::group_bytes;
    const uint32_t tg = tmem_base + static_cast<uint32_t>(g * kBCols);
    const uint32_t lane_base = tg + (static_cast<uint32_t>(wq * 32) << 16);
    const float beta = fabsf(__ldg(prm.beta)) + prm.beta_min;
    const bool rank1 = a.dfeature == nullptr;
    uint32_t ph_data = 0;
    float dbeta_acc = 0.0f;

    // one data-path GEMM of this group: all rows staged -> elected thread issues -> everybody waits for the accumulator
    auto data_step = [&](auto&& issue) {
      fence_before_sync();
      group_barrier(g);
      if (wq == 0) {
        if (elect_one()) {
          fence_after_sync();
          issue();
          mma_commit(mb_data + g);
        }
        __syncwarp();
      }
      mbar_wait(mb_data + g, ph_data);
      ph_data ^= 1;
      fence_after_sync();
    };
    // forward recompute of layer l: acc[128, 32] = A (TMEM, bf16 hi / mid) * W_l^T, W image K-major
    auto issue_fwd = [&](int l) {
      const int K = kLK[l];
      const uint32_t idesc = idesc_bf16(128, 32, 0, 0);
      const uint32_t wb = smem_u32(smem + FusedBwdSmem::w + fb_w_off(l));
      uint64_t bh = make_desc(wb, 128, (K / 8) * 128), bm = make_desc(wb + fb_w_half(l), 128, (K / 8) * 128);
      for (int ks = 0; ks < K / 16; ++ks) {
        mma_bf16_ts(tg + kBAcc, tg + kBAMid + 8 * ks, bh, idesc, ks > 0);
        mma_bf16_ts(tg + kBAcc, tg + kBAHi + 8 * ks, bm, idesc, true);
        mma_bf16_ts(tg + kBAcc, tg + kBAHi + 8 * ks, bh, idesc, true);
        bh += 16;
        bm += 16;
      }
    };
    // data gradient of layer l: acc[128, 32] = delta (TMEM) * W_l, the same image read MN-major (reduction over outputs)
    auto issue_din = [&](int l) {
      const int K = kLK[l];
      const uint32_t idesc = idesc_bf16(128, 32, 0, 1);
      const uint32_t wb = smem_u32(smem + FusedBwdSmem::w + fb_w_off(l));
      const uint32_t kgroup = static_cast<uint32_t>((K / 8) * 128);  // stride between groups of 8 outputs
      uint64_t bh = make_desc(wb, kgroup, 128), bm = make_desc(wb + fb_w_half(l), kgroup, 128);
      for (int ks = 0; ks < 2; ++ks) {
        mma_bf16_ts(tg + kBAcc, tg + kBDMid + 8 * ks, bh, idesc, ks > 0);
        mma_bf16_ts(tg + kBAcc, tg + kBDHi + 8 * ks, bm, idesc, true);
        mma_bf16_ts(tg + kBAcc, tg + kBDHi + 8 * ks, bh, idesc, true);
        bh += (2 * kgroup) >> 4;
        bm += (2 * kgroup) >> 4;
      }
    };
    // split 32 values of this thread's row: packed words to TMEM columns [col_hi, +16) / [col_mid, +16) (when col_hi >= 0)
    // and to the shared-memory image at img_hi / img_mid
    auto stage_row32 = [&](const float (&v)[32], int col_hi, int col_mid, char* img_hi, char* img_mid) {
      uint32_t h[16], m[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) split_bf16_pair(v[2 * c], v[2 * c + 1], h[c], m[c]);
      if (col_hi >= 0) {
        tmem_st16(lane_base + static_cast<uint32_t>(col_hi), h);
        tmem_st16(lane_base + static_cast<uint32_t>(col_mid), m);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        *reinterpret_cast<uint4*>(img_hi + q * 2048 + r * 16) = make_uint4(h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]);
        *reinterpret_cast<uint4*>(img_mid + q * 2048 + r * 16) = make_uint4(m[4 * q], m[4 * q + 1], m[4 * q + 2], m[4 * q + 3]);
      }
      if (col_hi >= 0) tmem_st_wait();
    };
    auto load_acc = [&](float (&v)[32]) { tmem_load_row<32>(tg + kBAcc, uwarp, 0, v); };
    auto wait_done = [&](int l, int64_t it) { mbar_wait(mb_done + g * 5 + l, static_cast<uint32_t>(it & 1)); };
    auto signal_ready = [&](int l) {
      fence_async_smem();
      mbar_arrive(mb_ready + g * 5 + l);
    };

    // head of a tile, loaded one tile ahead: this row of the saved hash-feature image and the three ReLU masks
    uint4 xq[8];
    uint32_t m_h1 = 0, m_g1 = 0, m_g2 = 0;
    auto load_head = [&](int64_t tile) {
      const int64_t rc = min(tile * kRows + r, a.M - 1);
      const uint4* src = a.ximg + tile * 1024 + r;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        xq[q] = __ldg(src + q * 128);
        xq[4 + q] = __ldg(src + 512 + q * 128);
      }
      m_h1 = __ldg(a.masks + rc), m_g1 = __ldg(a.masks + a.ld + rc), m_g2 = __ldg(a.masks + 2 * a.ld + rc);
    };
    if (g < mine) load_head(blockIdx.x + static_cast<int64_t>(g) * gridDim.x);

    int64_t it = 0;
    for (int64_t k = g; k < mine; k += 2, ++it) {
      const int64_t tile = blockIdx.x + k * gridDim.x;
      const int64_t row = tile * kRows + r;
      const bool ok = row < a.M;
      const int64_t rc = ok ? row : (a.M - 1);
      float v[32];
      NRB_FT(0);
      // the previous tile's last weight-gradient chain read the delta image and x: both are free again after this
      if (it > 0) wait_done(0, it - 1);
      if (!rank1 && r == 0) {  // d feature rows of this tile: TMA into the (free) delta image area, needed after layer 3
        mbar_expect_tx(mb_dfull + g, 16384);
        tma_load_rows(gs + FusedBwdSmem::d_hi, &dfeat_map, static_cast<int32_t>(tile * kRows), mb_dfull + g);
      }
      // ---- recompute, layer 0: A = this row of the saved hash-feature image
      {
        const uint32_t ha[16] = {xq[0].x, xq[0].y, xq[0].z, xq[0].w, xq[1].x, xq[1].y, xq[1].z, xq[1].w,
                                 xq[2].x, xq[2].y, xq[2].z, xq[2].w, xq[3].x, xq[3].y, xq[3].z, xq[3].w};
        const uint32_t ma[16] = {xq[4].x, xq[4].y, xq[4].z, xq[4].w, xq[5].x, xq[5].y, xq[5].z, xq[5].w,
                                 xq[6].x, xq[6].y, xq[6].z, xq[6].w, xq[7].x, xq[7].y, xq[7].z, xq[7].w};
        tmem_st16(lane_base + kBAHi, ha);
        tmem_st16(lane_base + kBAMid, ma);
        tmem_st_wait();
      }
      const uint32_t mh1 = m_h1, mg1 = m_g1, mg2 = m_g2;
      // the ray's SH basis (inputs 32..47 of layer 2), requested two layers before it is used
      float4 shq[4];
      if (a.actor_grid_id != nullptr && __ldg(a.actor_grid_id + rc) >= 0) {
        float o[16];
        sh16_of_direction(__ldg(a.actor_dirs + 3 * rc), __ldg(a.actor_dirs + 3 * rc + 1), __ldg(a.actor_dirs + 3 * rc + 2), o);
#pragma unroll
        for (int c = 0; c < 4; ++c) shq[c] = make_float4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
      } else {
        const float4* shp = reinterpret_cast<const float4*>(a.sh + (rc / a.samples_per_ray) * 16);
#pragma unroll
        for (int c = 0; c < 4; ++c) shq[c] = __ldg(shp + c);
      }
      NRB_FT(10);
      data_step([&] { issue_fwd(0); });
      NRB_FT(20);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((mh1 >> j) & 1u) ? v[j] + s_bias[j] : 0.0f;
      stage_row32(v, kBAHi, kBAMid, gs + FusedBwdSmem::h1, gs + FusedBwdSmem::h1 + 10240);  // (dW_1 of the last tile is done)
      // ---- layer 1 (embedding rows only; sdf is a saved output)
      NRB_FT(11);
      data_step([&] { issue_fwd(1); });
      NRB_FT(21);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += s_bias[48 + 1 + j];
      stage_row32(v, kBAHi, kBAMid, gs + FusedBwdSmem::emb, gs + FusedBwdSmem::emb + 14336);
      {
        uint32_t h[8], m[8];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          split_bf16_pair(shq[c].x, shq[c].y, h[2 * c], m[2 * c]);
          split_bf16_pair(shq[c].z, shq[c].w, h[2 * c + 1], m[2 * c + 1]);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const uint32_t hq[4] = {h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]};
          const uint32_t mq[4] = {m[4 * q], m[4 * q + 1], m[4 * q + 2], m[4 * q + 3]};
          tmem_st4(lane_base + static_cast<uint32_t>(kBAHi + 16 + 4 * q), hq);
          tmem_st4(lane_base + static_cast<uint32_t>(kBAMid + 16 + 4 * q), mq);
          *reinterpret_cast<uint4*>(gs + FusedBwdSmem::emb + (4 + q) * 2048 + r * 16) = make_uint4(hq[0], hq[1], hq[2], hq[3]);
          *reinterpret_cast<uint4*>(gs + FusedBwdSmem::emb + 14336 + (4 + q) * 2048 + r * 16) = make_uint4(mq[0], mq[1], mq[2], mq[3]);
        }
        tmem_st_wait();
      }
      // ---- layer 2
      NRB_FT(12);
      data_step([&] { issue_fwd(2); });
      NRB_FT(22);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((mg1 >> j) & 1u) ? v[j] + s_bias[2 * 48 + j] : 0.0f;
      stage_row32(v, kBAHi, kBAMid, gs + FusedBwdSmem::g1, gs + FusedBwdSmem::g1 + 10240);
      // ---- layer 3: g2 is only needed as the input image of dW_4
      NRB_FT(13);
      data_step([&] { issue_fwd(3); });
      NRB_FT(23);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((mg2 >> j) & 1u) ? v[j] + s_bias[3 * 48 + j] : 0.0f;
      stage_row32(v, -1, -1, gs + FusedBwdSmem::g2x, gs + FusedBwdSmem::g2x + 10240);

      // ---- backward sweep.  delta_4 = d feature
      float demb[32];
      NRB_FT(50);
      if (!rank1) {
        mbar_wait(mb_dfull + g, static_cast<uint32_t>(it & 1));
        const char* rowp = gs + FusedBwdSmem::d_hi + r * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 q4 = *reinterpret_cast<const float4*>(rowp + ((c ^ (r & 7)) << 4));
          demb[4 * c] = q4.x;
          demb[4 * c + 1] = q4.y;
          demb[4 * c + 2] = q4.z;
          demb[4 * c + 3] = q4.w;
        }
        group_barrier(g);  // every row has been read: the area turns into the delta image
      } else {
        const float wgt = __ldg(a.weights + rc);
        const float4* dfp = reinterpret_cast<const float4*>(a.dfeat_ray + (rc / a.samples_per_ray) * 32);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 q4 = __ldg(dfp + c);
          demb[4 * c] = wgt * q4.x;
          demb[4 * c + 1] = wgt * q4.y;
          demb[4 * c + 2] = wgt * q4.z;
          demb[4 * c + 3] = wgt * q4.w;
        }
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) demb[j] = ok ? demb[j] : 0.0f;
      stage_row32(demb, kBDHi, kBDMid, gs + FusedBwdSmem::d_hi, gs + FusedBwdSmem::d_mid);
      signal_ready(4);
      // the scalar inputs of the sdf / alpha head, requested two layers before they are used
      float a_v = 0.0f, sd_v = 0.0f, da_v = 0.0f, ds_v = 0.0f;
      if (ok) {
        a_v = __ldg(a.alpha + row), sd_v = __ldg(a.sdf + row);
        da_v = a.dalpha != nullptr ? __ldg(a.dalpha + row) : 0.0f;
        ds_v = a.dsdf != nullptr ? __ldg(a.dsdf + row) : 0.0f;
      }
      NRB_FT(34);
      data_step([&] { issue_din(4); });
      NRB_FT(44);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((mg2 >> j) & 1u) ? v[j] : 0.0f;
      // ---- layer 3
      NRB_FT(54);
      wait_done(4, it);
      NRB_FT(64);
      stage_row32(v, kBDHi, kBDMid, gs + FusedBwdSmem::d_hi, gs + FusedBwdSmem::d_mid);
      signal_ready(3);
      NRB_FT(33);
      data_step([&] { issue_din(3); });
      NRB_FT(43);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((mg1 >> j) & 1u) ? v[j] : 0.0f;
      // ---- layer 2 (only the embedding inputs carry a gradient; the SH basis is evaluated without one)
      NRB_FT(53);
      wait_done(3, it);
      NRB_FT(63);
      stage_row32(v, kBDHi, kBDMid, gs + FusedBwdSmem::d_hi, gs + FusedBwdSmem::d_mid);
      signal_ready(2);
      NRB_FT(32);
      data_step([&] { issue_din(2); });
      NRB_FT(42);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) demb[j] += v[j];
      // ---- layer 1: delta = [d emb | d sdf]; alpha = sigmoid(-sdf * beta)
      float dsdf_v = 0.0f;
      if (ok) {
        const float sg = a_v * (1.0f - a_v);
        dsdf_v = ds_v - da_v * beta * sg;
        dbeta_acc -= da_v * sd_v * sg;
      }
      NRB_FT(52);
      wait_done(2, it);
      NRB_FT(62);
      stage_row32(demb, kBDHi, kBDMid, gs + FusedBwdSmem::d_hi, gs + FusedBwdSmem::d_mid);
      {  // d sdf (row 0 of W1) has its own operand group: features (hi, mid, 0 ...)
        uint32_t h, m;
        split_bf16_pair(dsdf_v, 0.0f, h, m);
        *reinterpret_cast<uint4*>(gs + FusedBwdSmem::d_sdf + r * 16) = make_uint4((h & 0xFFFFu) | (m << 16), 0u, 0u, 0u);
      }
      signal_ready(1);
      NRB_FT(31);
      data_step([&] { issue_din(1); });
      NRB_FT(41);
      load_acc(v);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float d = fmaf(dsdf_v, w1row0[j], v[j]);
        v[j] = ((mh1 >> j) & 1u) ? d : 0.0f;
      }
      // ---- layer 0
      NRB_FT(51);
      wait_done(1, it);
      NRB_FT(61);
      stage_row32(v, kBDHi, kBDMid, gs + FusedBwdSmem::d_hi, gs + FusedBwdSmem::d_mid);
      NRB_FT(70);
      mbar_wait(mb_xfull + g, static_cast<uint32_t>(it & 1));  // x image landed
      NRB_FT(71);
      signal_ready(0);
      if (k + 2 < mine) load_head(blockIdx.x + (k + 2) * gridDim.x);  // next tile's head while the last GEMM runs
      if (a.dximg != nullptr) {
        NRB_FT(30);
        data_step([&] { issue_din(0); });
        NRB_FT(40);
        load_acc(v);
        float4* dst = a.dximg + tile * 1024 + r;
#pragma unroll
        for (int c = 0; c < 8; ++c) dst[c * 128] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
      }
    }
    if (it > 0) wait_done(0, it - 1);
    const float sb = warp_sum(dbeta_acc);
    if (lane == 0 && a.dbeta != nullptr && sb != 0.0f) {
      const float b0 = __ldg(prm.beta);  // d(|beta| + beta_min) / d beta = sign(beta)
      atomicAdd(a.dbeta, sb * (b0 > 0.0f ? 1.0f : (b0 < 0.0f ? -1.0f : 0.0f)));
    }
  }
  // ---- flush: weight and bias gradients from TMEM.  Row j of an M = 64 accumulator sits in lane (j / 16) * 32 + j % 16
  // (+ 16 for the second accumulator of a column range); rows j and 32 + j (hi and mid parts of delta) and the column
  // blocks [0,K) and [K+8, 2K+8) (hi and mid parts of the input) all belong to gradient element (j % 32, k).
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (mine > 0 && uwarp < 4) {
    const int wq = uwarp, half = lane >> 4, j = wq * 16 + (lane & 15);  // accumulator row held by this TMEM lane
#pragma unroll
    for (int u = 0; u < 6; ++u) {  // the five layers, then the sdf row of W1; every tcgen05.ld address is warp-uniform
      const int l = u < 5 ? u : 1;
      const int K = u < 5 ? kLK[u] : 32;
      const int col = u < 5 ? kDwCol[u] : kSdfCol, lane_off = u < 5 ? kDwLane[u] : kSdfLane;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + static_cast<uint32_t>(col);
      const int wrow = u == 5 ? 0 : (u == 1 ? (j & 31) + 1 : (j & 31));  // layer 1's accumulator holds rows 1..32 of W1
      const bool mine_row = (half == (lane_off >> 4)) && (u == 5 ? j < 2 : true);
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        if (c * 8 < K) {
          float hi8[8], mid8[8];
          tmem_ld8(taddr + c * 8, hi8);
          tmem_ld8(taddr + K + 8 + c * 8, mid8);
          tmem_ld_wait();
          if (mine_row && a.dw[l] != nullptr) {
#pragma unroll
            for (int i = 0; i < 8; ++i) atomicAdd(a.dw[l] + wrow * K + c * 8 + i, hi8[i] + mid8[i]);
          }
        }
      }
      float b8[8];
      tmem_ld8(taddr + K, b8);
      tmem_ld_wait();
      if (mine_row && a.db[l] != nullptr) atomicAdd(a.db[l] + wrow, b8[0]);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (uwarp == 0) tmem_free<512>(tmem_base);
}

}  // namespace nrb

using namespace nrb;

static FusedParams fused_params(const nrb_field_mlp_t* p) {
  FusedParams prm;
  for (int l = 0; l < 5; ++l) {
    prm.w[l] = p->weights[l];
    prm.b[l] = p->biases[l];
  }
  prm.beta = p->beta;
  prm.beta_min = p->beta_min;
  return prm;
}


// Tensor map of a row-major [M,32] fp32 matrix for TMA tile loads of 128 rows (cuTensorMapEncodeTiled through the
// runtime's driver entry point: the library links no libcuda).
static int make_rows_tensor_map(CUtensorMap* map, const float* base, int64_t M) {
  using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (encode == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    NRB_REQUIRE(e == cudaSuccess && fn != nullptr, NRB_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled is not available: %s",
                cudaGetErrorString(e));
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  const cuuint64_t dims[2] = {32, static_cast<cuuint64_t>(M)};
  const cuuint64_t strides[1] = {128};
  const cuuint32_t box[2] = {32, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  NRB_REQUIRE(r == CUDA_SUCCESS, NRB_ERR_BAD_ARG, "cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
  return NRB_OK;
}

extern "C" int64_t nrb_field_saved_ld(int64_t M) { return (M + tc::kRows - 1) / tc::kRows * tc::kRows; }

extern "C" int64_t nrb_field_fused_image_bytes(int64_t M) { return (M + tc::kRows - 1) / tc::kRows * 16384; }

extern "C" int nrb_field_fused_fwd(const nrb_field_mlp_t* p, const nrb_grid_t* grid, const float* xyz, const float* std,
                                   const float* x, const float* sh, int32_t samples_per_ray, int64_t M, float* feature,
                                   float* sdf, float* alpha, const nrb_field_fused_saved_t* saved,
                                   const nrb_actor_grids_t* actor_grids, const nrb_actor_samples_t* actor_samples,
                                   nrb_stream_t stream) {
  NRB_REQUIRE(p && sh && feature && sdf && alpha && M >= 0 && samples_per_ray > 0, NRB_ERR_BAD_ARG,
              "nrb_field_fused_fwd: null pointer or bad size");
  for (int l = 0; l < 5; ++l) NRB_REQUIRE(p->weights[l] != nullptr, NRB_ERR_BAD_ARG, "nrb_field_fused_fwd: weights[%d] is null", l);
  NRB_REQUIRE(p->beta != nullptr, NRB_ERR_BAD_ARG, "nrb_field_fused_fwd: beta is null");
  NRB_REQUIRE((grid != nullptr) != (x != nullptr), NRB_ERR_BAD_ARG,
              "nrb_field_fused_fwd: pass either a grid (+ xyz) to gather from or the hash features x");
  int F = 0;
  GridDev gd{};
  if (grid != nullptr) {
    if (int rc = check_grid(grid)) return rc;
    NRB_REQUIRE(xyz != nullptr, NRB_ERR_BAD_ARG, "nrb_field_fused_fwd: xyz is null");
    F = grid->features_per_level;
    NRB_REQUIRE((F == 2 || F == 4) && grid->num_levels * F == 32, NRB_ERR_UNSUPPORTED,
                "nrb_field_fused_fwd: the fused gather needs num_levels * features_per_level == 32 with 2 or 4 features");
    gd = to_dev(grid);
  } else {
    NRB_REQUIRE(aligned16(x), NRB_ERR_ALIGNMENT, "nrb_field_fused_fwd: x must be 16-byte aligned");
  }
  NRB_REQUIRE(aligned16(sh) && aligned16(feature), NRB_ERR_ALIGNMENT, "nrb_field_fused_fwd: sh and feature must be 16-byte aligned");
  if (actor_grids != nullptr) {
    if (int rc = check_actor_grids("nrb_field_fused_fwd", actor_grids)) return rc;
  }
  if (M == 0) return NRB_OK;
  FusedFwdArgs a{};
  a.xyz = xyz, a.std = std, a.x = x, a.sh = sh, a.samples_per_ray = samples_per_ray, a.M = M;
  a.feature = feature, a.sdf = sdf, a.alpha = alpha;
  if (saved != nullptr && saved->ximg != nullptr) {
    NRB_REQUIRE(saved->masks != nullptr && saved->ld >= M && saved->ld % tc::kRows == 0 && aligned16(saved->ximg),
                NRB_ERR_BAD_ARG, "nrb_field_fused_fwd: saved.masks / saved.ld (nrb_field_saved_ld(M)) / alignment");
    a.ximg = static_cast<uint4*>(saved->ximg), a.masks = saved->masks, a.ld = saved->ld;
  }
  const bool actors = actor_grids != nullptr;
  if (actors) {
    NRB_REQUIRE(grid != nullptr && actor_samples && actor_samples->grid_id && actor_samples->pos && actor_samples->std &&
                    actor_samples->dirs,
                NRB_ERR_BAD_ARG, "nrb_field_fused_fwd: actors need the gather mode and all per-sample actor arrays");
    a.ag = to_dev(actor_grids);
    a.as = ActorSamplesDev{actor_samples->grid_id, actor_samples->pos, actor_samples->std, actor_samples->dirs};
  }
  const int64_t tiles = (M + tc::kRows - 1) / tc::kRows;
  const unsigned nblk = static_cast<unsigned>(std::min<int64_t>((tiles + kFGroups - 1) / kFGroups, sm_count()));
  auto s = static_cast<cudaStream_t>(stream);
#define NRB_FUSED_FWD(FF, AA)                                                                                                  \
  {                                                                                                                            \
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(field_fused_fwd_kernel<FF, AA>), FusedFwdSmem::total); \
    NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "nrb_field_fused_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));  \
    field_fused_fwd_kernel<FF, AA><<<nblk, kFThreads, FusedFwdSmem::total, s>>>(fused_params(p), gd, a);                       \
  }
  if (F == 2 && actors) NRB_FUSED_FWD(2, true) else if (F == 4 && actors) NRB_FUSED_FWD(4, true)
  else if (F == 2) NRB_FUSED_FWD(2, false) else if (F == 4) NRB_FUSED_FWD(4, false) else NRB_FUSED_FWD(0, false)
#undef NRB_FUSED_FWD
  return finish_launch("nrb_field_fused_fwd");
}

extern "C" int nrb_field_fused_bwd(const nrb_field_mlp_t* p, const nrb_field_fused_bwd_in_t* in,
                                   const nrb_field_fused_bwd_out_t* out, int32_t samples_per_ray, int64_t M,
                                   nrb_stream_t stream) {
  NRB_REQUIRE(p && in && out && M >= 0 && samples_per_ray > 0, NRB_ERR_BAD_ARG, "nrb_field_fused_bwd: null pointer or bad size");
  NRB_REQUIRE(in->saved.ximg && in->saved.masks && in->sh && in->sdf && in->alpha, NRB_ERR_BAD_ARG,
              "nrb_field_fused_bwd: a required input is null");
  NRB_REQUIRE((in->dfeature != nullptr) != (in->dfeat_ray != nullptr && in->weights != nullptr), NRB_ERR_BAD_ARG,
              "nrb_field_fused_bwd: pass either dfeature [M,32] or dfeat_ray [rays,32] with weights [M]");
  NRB_REQUIRE(in->saved.ld >= M && in->saved.ld % tc::kRows == 0, NRB_ERR_BAD_ARG,
              "nrb_field_fused_bwd: saved.ld must be nrb_field_saved_ld(M)");
  for (int l = 0; l < 5; ++l) NRB_REQUIRE(p->weights[l] != nullptr, NRB_ERR_BAD_ARG, "nrb_field_fused_bwd: weights[%d] is null", l);
  NRB_REQUIRE(p->beta != nullptr, NRB_ERR_BAD_ARG, "nrb_field_fused_bwd: beta is null");
  NRB_REQUIRE(aligned16(in->saved.ximg) && aligned16(in->sh) && (in->dfeature == nullptr || aligned16(in->dfeature)) &&
                  (in->dfeat_ray == nullptr || aligned16(in->dfeat_ray)) && (out->dximg == nullptr || aligned16(out->dximg)),
              NRB_ERR_ALIGNMENT, "nrb_field_fused_bwd: arrays must be 16-byte aligned");
  if (M == 0) return NRB_OK;
  FusedBwdArgs a{};
  a.ximg = static_cast<const uint4*>(in->saved.ximg), a.masks = in->saved.masks, a.ld = in->saved.ld;
  a.sh = in->sh, a.sdf = in->sdf, a.alpha = in->alpha;
  a.dfeature = in->dfeature, a.dfeat_ray = in->dfeat_ray, a.weights = in->weights, a.dsdf = in->dsdf, a.dalpha = in->dalpha;
  a.samples_per_ray = samples_per_ray, a.M = M;
  a.actor_grid_id = in->actor_grid_id, a.actor_dirs = in->actor_dirs;
  NRB_REQUIRE((a.actor_grid_id == nullptr) == (a.actor_dirs == nullptr), NRB_ERR_BAD_ARG,
              "nrb_field_fused_bwd: actor_grid_id and actor_dirs go together");
  a.dximg = reinterpret_cast<float4*>(out->dximg);
  for (int l = 0; l < 5; ++l) {
    a.dw[l] = out->dweights[l];
    a.db[l] = out->dbiases[l];
  }
  a.dbeta = out->dbeta;
  CUtensorMap map{};
  if (a.dfeature != nullptr) {
    if (int rc = make_rows_tensor_map(&map, a.dfeature, M)) return rc;
  }
  cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(field_fused_bwd_kernel), FusedBwdSmem::total);
  NRB_REQUIRE(e == cudaSuccess, static_cast<int>(e), "nrb_field_fused_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  const int64_t tiles = (M + tc::kRows - 1) / tc::kRows;
  const unsigned nblk = static_cast<unsigned>(std::min<int64_t>((tiles + 1) / 2, sm_count()));
  field_fused_bwd_kernel<<<nblk, kBThreads, FusedBwdSmem::total, static_cast<cudaStream_t>(stream)>>>(fused_params(p), a, map);
  return finish_launch("nrb_field_fused_bwd");
}

#ifdef NRB_FUSED_TRACE
extern "C" int nrb_debug_fused_trace(long long* host, int32_t n) {
  cudaDeviceSynchronize();
  return static_cast<int>(cudaMemcpyFromSymbol(host, nrb::g_fused_trace, sizeof(long long) * std::min(n, 4096)));
}
#endif
