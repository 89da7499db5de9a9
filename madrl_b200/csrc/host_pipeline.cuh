// Host side shared by the three env families: the handle core every `madrl_*` handle derives from,
// the persistent launch policy, and the host-buffer rollout (the `*_rollout_host` entry points).
//
// A host-buffer rollout takes HOST pointers (pinned for full speed); the copies are part of the call.  The
// rollout is cut into chunks of lockstep steps: chunk c+1 is computed on one stream while the copy
// engines drain chunk c's trajectory rows on another, and the action upload rides in front on the
// compute stream (H2D and D2H use different copy engines).  With the full observation tensor
// returned, the call runs at the PCIe D2H rate (the kernel is ~1.5 % of it); with
// MADRL_HOST_OBS_LAST (policy on the device: only the last step's observations are needed on the
// host to continue) it runs at the kernel's rate.
#pragma once
#include <cmath>

#include "common.cuh"

namespace madrl {

struct HostPipe {
  void* stage = nullptr;
  size_t stage_bytes = 0;
  cudaStream_t compute = nullptr, copy = nullptr;
  cudaEvent_t done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};

  // Blocking (default-flag) streams: ordered after earlier work on the legacy default stream (e.g. a
  // reset launched there), unordered with each other.
  int ensure(size_t bytes) {
    if (!compute) {
      MADRL_CUDA_CHECK(cudaStreamCreate(&compute));
      MADRL_CUDA_CHECK(cudaStreamCreate(&copy));
      for (int i = 0; i < 8; ++i) MADRL_CUDA_CHECK(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
    }
    if (stage_bytes >= bytes) return MADRL_OK;
    if (stage) cudaFree(stage);
    stage = nullptr;
    stage_bytes = 0;
    cudaError_t e = cudaMalloc(&stage, bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc(stage %zu): %s", bytes, cudaGetErrorString(e)); return MADRL_ENOMEM; }
    stage_bytes = bytes;
    return MADRL_OK;
  }
  void destroy() {
    if (stage) cudaFree(stage);
    if (compute) cudaStreamDestroy(compute);
    if (copy) cudaStreamDestroy(copy);
    for (int i = 0; i < 8; ++i) if (done[i]) cudaEventDestroy(done[i]);
    stage = nullptr; compute = copy = nullptr;
  }
};

// Bytes of ONE lockstep step of each trajectory tensor (all tensors are time-major, so a chunk of
// steps is one contiguous slice of each).
struct StepBytes { size_t act, obs, rew, done, info; };

// launch(t0, Tc, act_dev, obs_dev, rew_dev, done_dev, info_dev, stream) -> rc runs Tc lockstep steps.
template <class Launch>
int host_rollout(HostPipe& hp, int T, const StepBytes& sb, const void* act_h, void* obs_h, void* rew_h, void* done_h,
                 void* info_h, int obs_last_only, Launch launch) {
  const size_t TT = (size_t)T;
  const size_t o_obs = align_up(TT * sb.act, 256), o_rew = align_up(o_obs + TT * sb.obs, 256);
  const size_t o_done = align_up(o_rew + TT * sb.rew, 256), o_info = align_up(o_done + TT * sb.done, 256);
  int rc = hp.ensure(o_info + TT * sb.info);
  if (rc) return rc;
  char* st = (char*)hp.stage;
  // chunks of >= 32 MB (madrl_set_host_chunk_bytes) of device->host traffic -- below that a copy is
  // latency-dominated -- and at most 8
  const size_t out_step = (obs_last_only ? 0 : sb.obs) + sb.rew + sb.done + sb.info;
  size_t n_chunks = (TT * out_step) / g_host_chunk_bytes.load();
  if (n_chunks < 1) n_chunks = 1;
  if (n_chunks > 8) n_chunks = 8;
  if (n_chunks > TT) n_chunks = TT;
  // done / info rows are sliced at chunk boundaries: keep the 8-byte alignment of the info rows
  size_t Tc = (TT + n_chunks - 1) / n_chunks;
  while ((Tc * sb.info) % 8 != 0) ++Tc;
  MADRL_CUDA_CHECK(cudaMemcpyAsync(st, act_h, TT * sb.act, cudaMemcpyHostToDevice, hp.compute));
  int c = 0;
  for (size_t t0 = 0; t0 < TT; t0 += Tc, ++c) {
    const size_t n = (t0 + Tc <= TT) ? Tc : TT - t0;
    rc = launch((int)t0, (int)n, st + t0 * sb.act, st + o_obs + t0 * sb.obs, st + o_rew + t0 * sb.rew,
                st + o_done + t0 * sb.done, st + o_info + t0 * sb.info, hp.compute);
    if (rc) return rc;
    MADRL_CUDA_CHECK(cudaEventRecord(hp.done[c], hp.compute));
    MADRL_CUDA_CHECK(cudaStreamWaitEvent(hp.copy, hp.done[c], 0));
    if (!obs_last_only)
      MADRL_CUDA_CHECK(cudaMemcpyAsync((char*)obs_h + t0 * sb.obs, st + o_obs + t0 * sb.obs, n * sb.obs,
                                       cudaMemcpyDeviceToHost, hp.copy));
    else if (t0 + n == TT)
      MADRL_CUDA_CHECK(cudaMemcpyAsync(obs_h, st + o_obs + (TT - 1) * sb.obs, sb.obs, cudaMemcpyDeviceToHost, hp.copy));
    MADRL_CUDA_CHECK(cudaMemcpyAsync((char*)rew_h + t0 * sb.rew, st + o_rew + t0 * sb.rew, n * sb.rew,
                                     cudaMemcpyDeviceToHost, hp.copy));
    MADRL_CUDA_CHECK(cudaMemcpyAsync((char*)done_h + t0 * sb.done, st + o_done + t0 * sb.done, n * sb.done,
                                     cudaMemcpyDeviceToHost, hp.copy));
    MADRL_CUDA_CHECK(cudaMemcpyAsync((char*)info_h + t0 * sb.info, st + o_info + t0 * sb.info, n * sb.info,
                                     cudaMemcpyDeviceToHost, hp.copy));
  }
  MADRL_CUDA_CHECK(cudaStreamSynchronize(hp.copy));
  MADRL_CUDA_CHECK(cudaStreamSynchronize(hp.compute));
  return MADRL_OK;
}

// ---- handle core ----------------------------------------------------------------------------------
// The fields every env handle has; madrl_ww / madrl_pursuit / madrl_hostage derive from it and add their
// config, layout and own fields.
struct EnvCore {
  char* state = nullptr;     // the env state blob (layout.total_bytes)
  bool owns_state = false;   // allocated by core_init (not adopted from the caller)
  int device = 0, sms = 0;
  int blocks_per_sm = 0;     // madrl_*_set_launch (0 = as many as the occupancy allows)
  HostPipe pipe;             // staging + streams of the host-buffer entry points (lazily created)
  void* term_obs = nullptr;  // madrl_*_set_terminal_obs (NULL = off)
};

// Current device and its SM count; adopt `state_dev` or cudaMalloc `total_bytes`; zero the blob.  On
// failure the caller releases the handle (core_release + delete).
int core_init(EnvCore* h, void* state_dev, size_t total_bytes);
void core_release(EnvCore* h);
// seed(): every env's Philox draw counter back to 0.
int core_clear_counters(EnvCore* h, size_t rng_counter_off, int n_envs, void* stream);
int core_set_terminal_obs(EnvCore* h, void* term_obs_dev);
int core_set_launch(EnvCore* h, int warps_per_block, int blocks_per_sm);
// cos / sin of K sensor angles linspace(0, 2pi, K+1)[:-1] (ww:29-31, hw:27-29) as 2K reals at `dst_dev`.
int upload_sensor_table(char* dst_dev, int K, bool fp64);

// Largest representable t with correctly-rounded sqrt(t) <= thr: `sqrt(d2) <= thr` (what
// scipy's cdist + `<=` computes in the reference) is then exactly `d2 <= t`.
template <typename real>
real exact_sq_threshold(double thr_d) {
  const real thr = (real)thr_d;
  real t = thr * thr;
  const real up = (real)INFINITY, dn = -(real)INFINITY;
  while (std::sqrt(t) <= thr) t = std::nextafter(t, up);
  while (std::sqrt(t) > thr) t = std::nextafter(t, dn);
  return t;
}

// Launch a persistent warp-per-env kernel: 32-thread blocks, as many resident per SM as the occupancy
// allows (capped by set_launch's blocks_per_sm), grid = one block per env or a single persistent wave.
template <class Kernel, class Params>
int launch_persistent(const EnvCore* h, Kernel kfn, int E, size_t smem, cudaStream_t stream, const Params& p) {
  if (smem > 48 * 1024)
    MADRL_CUDA_CHECK(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int resident = 0;
  MADRL_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kfn, 32, smem));
  if (resident < 1) resident = 1;
  if (h->blocks_per_sm > 0 && h->blocks_per_sm < resident) resident = h->blocks_per_sm;
  int grid = E;                                        // one warp (= one 32-thread block) per env ...
  if (grid > h->sms * resident) grid = h->sms * resident;   // ... or a single persistent wave
  MADRL_LAUNCH(kfn, grid, 32, smem, stream, p);
  g_launches.fetch_add(1);
  MADRL_CUDA_CHECK(cudaGetLastError());
  return MADRL_OK;
}

// reset() with host buffers: stage the mask and, when masked, the caller's obs (rows of unmasked envs must
// survive); reset_fn(mask_dev, obs_dev) -> rc launches the device reset on the legacy default stream.
template <class ResetFn>
int core_reset_host(EnvCore* h, size_t E, size_t obs_bytes, const uint8_t* mask_host, void* obs_host, ResetFn reset_fn) {
  const size_t mask_off = align_up(obs_bytes, 256);
  int rc = h->pipe.ensure(mask_off + E);
  if (rc) return rc;
  char* st = (char*)h->pipe.stage;
  uint8_t* mask_dev = nullptr;
  if (mask_host) {
    mask_dev = (uint8_t*)(st + mask_off);
    MADRL_CUDA_CHECK(cudaMemcpyAsync(mask_dev, mask_host, E, cudaMemcpyHostToDevice, 0));
    MADRL_CUDA_CHECK(cudaMemcpyAsync(st, obs_host, obs_bytes, cudaMemcpyHostToDevice, 0));
  }
  rc = reset_fn(mask_dev, st);
  if (rc) return rc;
  MADRL_CUDA_CHECK(cudaMemcpyAsync(obs_host, st, obs_bytes, cudaMemcpyDeviceToHost, 0));
  MADRL_CUDA_CHECK(cudaStreamSynchronize(0));
  return MADRL_OK;
}

// rollout() with host buffers: argument checks, then host_rollout with the terminal-obs side tensor off
// (the kernel would index it with chunk-relative offsets: it is a device-API feature).
template <class Launch>
int core_rollout_host(EnvCore* h, int T, const StepBytes& sb, const void* act_h, void* obs_h, void* rew_h,
                      void* done_h, void* info_h, int flags, Launch launch) {
  MADRL_REQUIRE(T >= 1, "T must be >= 1");
  MADRL_REQUIRE(act_h && obs_h && rew_h && done_h && info_h, "NULL trajectory buffer");
  MADRL_REQUIRE((flags & ~MADRL_HOST_OBS_LAST) == 0, "unknown flags %d", flags);
  void* const keep = h->term_obs;
  h->term_obs = nullptr;
  const int rc = host_rollout(h->pipe, T, sb, act_h, obs_h, rew_h, done_h, info_h, flags & MADRL_HOST_OBS_LAST, launch);
  h->term_obs = keep;
  return rc;
}

}  // namespace madrl
