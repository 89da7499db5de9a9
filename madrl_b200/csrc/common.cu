// Library-wide host helpers: error string, launch counter, device queries, the env handle core.
#include <math.h>
#include <stdarg.h>
#include <string.h>
#include <new>

#include "common.cuh"
#include "host_pipeline.cuh"

namespace madrl {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
std::atomic<size_t> g_host_chunk_bytes{(size_t)32 << 20};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count(int device) {
  int n = 0;
  cudaError_t e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) {
    set_error("cudaDeviceGetAttribute(SM count): %s", cudaGetErrorString(e));
    return -1;
  }
  return n;
}

// ---- handle core (host_pipeline.cuh) ------------------------------------------------------------
int core_init(EnvCore* h, void* state_dev, size_t total_bytes) {
  cudaError_t e = cudaGetDevice(&h->device);
  if (e != cudaSuccess) { set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return MADRL_ECUDA; }
  h->sms = sm_count(h->device);
  if (h->sms <= 0) return MADRL_ECUDA;
  if (state_dev) {
    h->state = (char*)state_dev;
  } else {
    char* p = nullptr;
    e = cudaMalloc((void**)&p, total_bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu): %s", total_bytes, cudaGetErrorString(e)); return MADRL_ENOMEM; }
    h->state = p;
    h->owns_state = true;
  }
  e = cudaMemset(h->state, 0, total_bytes);
  if (e != cudaSuccess) { set_error("cudaMemset: %s", cudaGetErrorString(e)); return MADRL_ECUDA; }
  return MADRL_OK;
}

void core_release(EnvCore* h) {
  if (h->owns_state && h->state) cudaFree(h->state);
  h->pipe.destroy();
}

int core_clear_counters(EnvCore* h, size_t rng_counter_off, int n_envs, void* stream) {
  MADRL_CUDA_CHECK(cudaMemsetAsync(h->state + rng_counter_off, 0, 8 * (size_t)n_envs, (cudaStream_t)stream));
  return MADRL_OK;
}

int core_set_terminal_obs(EnvCore* h, void* term_obs_dev) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  h->term_obs = term_obs_dev;
  return MADRL_OK;
}

int core_set_launch(EnvCore* h, int warps_per_block, int blocks_per_sm) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  // warps_per_block is ignored (blocks are one warp) but still range-checked: the ABI has always refused > 4
  MADRL_REQUIRE(warps_per_block >= 0 && warps_per_block <= 4, "warps_per_block must be in [0,4]");
  MADRL_REQUIRE(blocks_per_sm >= 0 && blocks_per_sm <= 32, "blocks_per_sm must be in [0,32]");
  h->blocks_per_sm = blocks_per_sm;
  return MADRL_OK;
}

template <typename real>
static int upload_sensor_table_t(char* dst_dev, int K) {
  real* tab = new (std::nothrow) real[2 * (size_t)K];
  if (!tab) return MADRL_ENOMEM;
  const double step = (2.0 * M_PI - 0.0) / (double)K;
  for (int k = 0; k < K; ++k) {
    const double a = (double)k * step + 0.0;
    tab[k] = (real)cos(a);
    tab[K + k] = (real)sin(a);
  }
  cudaError_t e = cudaMemcpy(dst_dev, tab, sizeof(real) * 2 * K, cudaMemcpyHostToDevice);
  delete[] tab;
  MADRL_CUDA_CHECK(e);
  return MADRL_OK;
}

int upload_sensor_table(char* dst_dev, int K, bool fp64) {
  return fp64 ? upload_sensor_table_t<double>(dst_dev, K) : upload_sensor_table_t<float>(dst_dev, K);
}

}  // namespace madrl

extern "C" const char* madrl_last_error(void) { return madrl::g_err; }
extern "C" int madrl_version(void) { return 200; }
// sizeof of every struct that crosses the ABI: a binding built against another header refuses to run
extern "C" void madrl_abi_sizes(int32_t* out6) {
  out6[0] = (int32_t)sizeof(madrl_ww_config); out6[1] = (int32_t)sizeof(madrl_ww_layout);
  out6[2] = (int32_t)sizeof(madrl_pursuit_config); out6[3] = (int32_t)sizeof(madrl_pursuit_layout);
  out6[4] = (int32_t)sizeof(madrl_hostage_config); out6[5] = (int32_t)sizeof(madrl_hostage_layout);
}
extern "C" uint64_t madrl_launch_count(void) { return madrl::g_launches.load(); }
extern "C" void madrl_set_host_chunk_bytes(size_t bytes) { madrl::g_host_chunk_bytes.store(bytes ? bytes : ((size_t)32 << 20)); }

// ---- CUDA IPC helpers for the fused multi-GPU exchange (madrl_b200/dist.py PeerGather) -----------
// Buffers are cudaMalloc'ed here (not sub-allocated by a framework allocator) so that the IPC
// handle refers to exactly this buffer, and peers open it with THEIR device current, which is what
// makes the mapping usable from kernels running on the importing device.
extern "C" int madrl_ipc_alloc(size_t bytes, void** ptr, unsigned char* handle64) {
  MADRL_REQUIRE(ptr != nullptr && handle64 != nullptr && bytes > 0, "bad arguments");
  MADRL_CUDA_CHECK(cudaMalloc(ptr, bytes));
  MADRL_CUDA_CHECK(cudaMemset(*ptr, 0, bytes));
  cudaIpcMemHandle_t h;
  MADRL_CUDA_CHECK(cudaIpcGetMemHandle(&h, *ptr));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64, &h, 64);
  return MADRL_OK;
}

extern "C" int madrl_ipc_open(const unsigned char* handle64, void** ptr) {
  MADRL_REQUIRE(ptr != nullptr && handle64 != nullptr, "bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  MADRL_CUDA_CHECK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return MADRL_OK;
}

extern "C" int madrl_ipc_close(void* ptr) {
  if (ptr) MADRL_CUDA_CHECK(cudaIpcCloseMemHandle(ptr));
  return MADRL_OK;
}

extern "C" int madrl_ipc_free(void* ptr) {
  if (ptr) MADRL_CUDA_CHECK(cudaFree(ptr));
  return MADRL_OK;
}
