// Shared helpers for the lfmq CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

namespace lfmq {

extern thread_local char g_err[512];
extern long long g_launches;

#define LFMQ_SET_ERR(...) snprintf(::lfmq::g_err, sizeof(::lfmq::g_err), __VA_ARGS__)

#define LFMQ_CUDA_CHECK(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      LFMQ_SET_ERR("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));  \
      return 2; /* LFMQ_ERR_CUDA */                                                        \
    }                                                                                      \
  } while (0)

// Programmatic dependent launch.  Device side: every kernel launched through launch_pdl() calls pdl_sync() before it
// touches anything its predecessors wrote -- wait for the previous kernel of the stream, THEN let the next one's CTAs be
// dispatched (in that order: when a kernel starts, its predecessor has seen ITS predecessor complete, so only the
// immediate predecessor can still be running).  A kernel launched without the attribute sees both as no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_sync() {
  pdl_wait();
  pdl_release();
}

// Every kernel launch goes through this so bench.py can report gpu_launches.
// LFMQ_DEBUG_SYNC=1: synchronise after every launch and say where (finds the kernel that hangs or faults).
inline bool debug_sync_on() {
  static const bool on = getenv("LFMQ_DEBUG_SYNC") && atoi(getenv("LFMQ_DEBUG_SYNC")) != 0;
  return on;
}
#define LFMQ_DEBUG_SYNC()                                                                              \
  do {                                                                                                 \
    if (::lfmq::debug_sync_on()) {                                                                     \
      fprintf(stderr, "[lfmq launch] %s:%d ...", __FILE__, __LINE__);                                  \
      fflush(stderr);                                                                                  \
      cudaError_t _e = cudaDeviceSynchronize();                                                        \
      fprintf(stderr, " %s\n", cudaGetErrorString(_e));                                               \
      fflush(stderr);                                                                                  \
    }                                                                                                  \
  } while (0)

#define LFMQ_LAUNCH_CHECK()                                   \
  do {                                                        \
    ::lfmq::g_launches++;                                     \
    LFMQ_CUDA_CHECK(cudaGetLastError());                      \
    LFMQ_DEBUG_SYNC();                                        \
  } while (0)

// Host side: launch with the programmatic-stream-serialization attribute (LFMQ_PDL=0 turns it off).  `attrs_extra` lets
// the cluster kernels add their cluster dimension.
inline bool pdl_on() {
  static const bool on = !(getenv("LFMQ_PDL") && atoi(getenv("LFMQ_PDL")) == 0);
  return on;
}
template <typename... KArgs, typename... Args>
inline int launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, int cluster_x,
                      Args&&... args) {
  const bool on = pdl_on();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (on) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  LFMQ_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
  g_launches++;
  LFMQ_DEBUG_SYNC();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011) -- bit-identical to oracle/lfm_oracle.py:philox4x32_10.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Dropout scale factors for the 4 consecutive elements of quad q = (global_row * inner + j) / 4.
struct DropoutKey {
  uint32_t k0, k1;     // seed
  uint32_t stream;     // 2*layer (Dropout) or 2*layer+1 (recurrent dropout)
  uint32_t step;
  uint32_t thr;        // keep iff (r >> 8) >= thr, thr = (uint32)(rate * 2^24)
  float scale;         // 1 / (1 - rate)
};

__device__ __forceinline__ void dropout_quad(const DropoutKey& k, uint64_t q, float m[4]) {
  uint32_t r[4];
  philox4x32_10((uint32_t)q, (uint32_t)(q >> 32), k.stream, k.step, k.k0, k.k1, r);
#pragma unroll
  for (int i = 0; i < 4; ++i) m[i] = ((r[i] >> 8) >= k.thr) ? k.scale : 0.0f;
}

// Event brackets around the regions of a step (include/lfmq.h LFMQ_REGION_*).
struct Profiler {
  static constexpr int kRegions = 5, kCap = 256;
  bool enabled = false;
  bool created = false;
  cudaEvent_t a[kRegions][kCap], b[kRegions][kCap];
  int n[kRegions] = {0, 0, 0, 0, 0};
  void begin(int r, cudaStream_t s) {
    if (enabled && n[r] < kCap) cudaEventRecord(a[r][n[r]], s);
  }
  void end(int r, cudaStream_t s) {
    if (enabled && n[r] < kCap) cudaEventRecord(b[r][n[r]++], s);
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace lfmq
