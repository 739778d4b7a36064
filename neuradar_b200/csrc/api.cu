// Library plumbing: version, per-thread error string, launch counter, argument validation.
#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace nrb {

static thread_local char g_error[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int finish_launch(const char* what) {
  count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: kernel launch failed: %s", what, cudaGetErrorString(e));
    return static_cast<int>(e);
  }
  return NRB_OK;
}

int check_grid(const nrb_grid_t* g) {
  NRB_REQUIRE(g != nullptr && g->table != nullptr, NRB_ERR_BAD_ARG, "grid: null grid or table pointer");
  NRB_REQUIRE(g->num_levels >= 1 && g->num_levels <= NRB_MAX_LEVELS, NRB_ERR_BAD_ARG, "grid: num_levels %d not in [1,%d]",
              g->num_levels, NRB_MAX_LEVELS);
  NRB_REQUIRE(g->features_per_level == 1 || g->features_per_level == 2 || g->features_per_level == 4,
              NRB_ERR_UNSUPPORTED, "grid: features_per_level %d not in {1,2,4}", g->features_per_level);
  NRB_REQUIRE(g->log2_hashmap_size >= 1 && g->log2_hashmap_size <= 24, NRB_ERR_BAD_ARG,
              "grid: log2_hashmap_size %d not in [1,24]", g->log2_hashmap_size);
  NRB_REQUIRE(aligned16(g->table), NRB_ERR_ALIGNMENT, "grid: table must be 16-byte aligned");
  return NRB_OK;
}

int check_rays(const nrb_rays_t* r) {
  NRB_REQUIRE(r != nullptr, NRB_ERR_BAD_ARG, "rays: null");
  NRB_REQUIRE(r->num_rays >= 0, NRB_ERR_BAD_ARG, "rays: negative num_rays");
  NRB_REQUIRE(r->num_rays == 0 || (r->origins && r->directions && r->pixel_area), NRB_ERR_BAD_ARG,
              "rays: origins/directions/pixel_area must be set");
  return NRB_OK;
}

int check_intervals(const char* who, const nrb_intervals_t* iv) {
  NRB_REQUIRE(iv != nullptr && iv->starts != nullptr && iv->ends != nullptr, NRB_ERR_BAD_ARG, "%s: null intervals", who);
  NRB_REQUIRE(iv->num_samples > 0 && iv->num_samples <= NRB_MAX_SAMPLES, NRB_ERR_BAD_ARG,
              "%s: num_samples %d not in [1,%d]", who, iv->num_samples, NRB_MAX_SAMPLES);
  NRB_REQUIRE(iv->row_stride >= iv->num_samples, NRB_ERR_BAD_ARG, "%s: row_stride smaller than num_samples", who);
  return NRB_OK;
}

cudaError_t ensure_dynamic_smem(const void* kernel, int bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, int> done;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) (void)cudaGetLastError();
  std::lock_guard<std::mutex> lock(mu);
  auto key = std::make_pair(dev, kernel);
  auto it = done.find(key);
  if (it != done.end() && it->second >= bytes) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done[key] = bytes;
  return e;
}

int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
      cached = n;
    } else {
      (void)cudaGetLastError();
      return 148;  // B200
    }
  }
  return cached;
}

}  // namespace nrb

extern "C" int nrb_version(void) { return NRB_VERSION; }

extern "C" int32_t nrb_max_actors(void) { return NRB_MAX_ACTORS; }
extern "C" const char* nrb_last_error_string(void) { return nrb::g_error; }
extern "C" int64_t nrb_launch_count(void) { return nrb::g_launches.load(std::memory_order_relaxed); }
