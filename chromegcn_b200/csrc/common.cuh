// Shared device / host helpers for libchromegcn (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/chromegcn.h"

namespace cgcn {

// ------------------------------------------------------------------ errors / bookkeeping
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return CGCN_ERR_CUDA;
  }
  return CGCN_OK;
}

#define CGCN_CUDA(expr)                                                        \
  do {                                                                         \
    cudaError_t e__ = (expr);                                                  \
    if (e__ != cudaSuccess) {                                                  \
      cgcn::set_error("%s: %s", #expr, cudaGetErrorString(e__));               \
      return CGCN_ERR_CUDA;                                                    \
    }                                                                          \
  } while (0)

#define CGCN_TRY(expr)                                                         \
  do {                                                                         \
    int s__ = (expr);                                                          \
    if (s__ != CGCN_OK) return s__;                                            \
  } while (0)

#define CGCN_REQUIRE(cond, ...)                                                \
  do {                                                                         \
    if (!(cond)) {                                                             \
      cgcn::set_error(__VA_ARGS__);                                            \
      return CGCN_ERR_INVALID;                                                 \
    }                                                                          \
  } while (0)

int sm_count();                       // cached, current device

// "set once per device" helper for cudaFuncSetAttribute: the attribute belongs to the device's context, so a
// process that drives several GPUs must set it on each of them.
inline bool first_use_on_device(bool (&done)[64]) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
  if (done[dev]) return false;
  done[dev] = true;
  return true;
}

// ------------------------------------------------------------------ programmatic dependent launch
// One chromosome step is ~34 kernels of 5..60 us each on one stream: the drain / launch / ramp-up bubble between
// two dependent kernels is a measurable share of it.  Every kernel of the model path starts with pdl_grid_sync()
// (griddepcontrol.wait: the whole previous grid has completed and its writes are visible; then
// griddepcontrol.launch_dependents: the next kernel's CTAs may be scheduled as soon as all of this grid's CTAs have
// started) and is launched through launch_k() with cudaLaunchAttributeProgrammaticStreamSerialization, so the next
// kernel's launch latency and prologue (barrier init, TMEM allocation, argument fetch) overlap this kernel's tail.
// Nothing that touches global memory may precede pdl_grid_sync().  CGCN_NO_PDL=1 turns the attribute off.
bool pdl_enabled();
void pdl_plain_next(cudaStream_t stream);   // the next launch_k on `stream` is an ordinary launch (after event waits)
bool pdl_take_plain(cudaStream_t stream);

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_enabled() && !pdl_take_plain(stream)) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// one weight operand of a tcgen05 row-panel contraction, to be split (hi/lo TF32) and swizzled into `img`
struct TcImageSpec {
  const float* B;
  int b_transposed, n, k;
  void* img;
};
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Peer gather (one graph row-partitioned over the GPUs of an NVLink box): the gathered panel lives in the ranks'
// exchange buffers (cgcn_peer_panel); rank r owns global rows [begin[r], begin[r+1]) at base[r].  Passed by value in
// kernel parameters, read with peer_row().
struct PeerTable {
  int world;
  int begin[CGCN_MAX_PEERS + 1];
  const float* base[CGCN_MAX_PEERS];
};

// Fills *t from pp and checks it against this rank's graph of n_local rows; error messages start with `who`.
int peer_table(PeerTable* t, const cgcn_peer_panel* pp, int n_local, const char* who);

// bump allocator over a caller-provided workspace
struct Arena {
  char* base;
  size_t cap;
  size_t off;
  Arena(void* p, size_t bytes) : base(static_cast<char*>(p)), cap(bytes), off(0) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* r = reinterpret_cast<T*>(base + off);
    off += count * sizeof(T);
    return r;
  }
  bool ok() const { return off <= cap; }
};

// ------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

__device__ __forceinline__ void pdl_grid_sync() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float inv_degree(const int32_t* __restrict__ rowptr, int row) {
  // float32(1.0 / float64(deg)) of utils/util_methods.py:101-105,122 == correctly rounded 1.0f / (float)deg
  const int deg = __ldg(rowptr + row + 1) - __ldg(rowptr + row);
  return deg > 0 ? __fdiv_rn(1.0f, static_cast<float>(deg)) : 0.0f;
}

// 1/deg from the pattern, or the stored 1/rowsum of a weighted graph
__device__ __forceinline__ float row_scale(const int32_t* __restrict__ rowptr, const float* __restrict__ row_inv, int row) {
  return row_inv != nullptr ? __ldg(row_inv + row) : inv_degree(rowptr, row);
}

// Row c of a panel of pitch_floats floats per row, spread over the ranks of t: the owner is counted with
// CGCN_MAX_PEERS - 1 compares.  A kernel that takes the table as a parameter of its own declares it __grid_constant__;
// dynamically indexed, a by-value parameter of this size is otherwise copied to local memory.
__device__ __forceinline__ const float* peer_row(const PeerTable& t, int c, size_t pitch_floats) {
  int o = 0;
#pragma unroll
  for (int r = 1; r < CGCN_MAX_PEERS; ++r) o += (r < t.world && c >= t.begin[r]) ? 1 : 0;
  return t.base[o] + static_cast<size_t>(c - t.begin[o]) * pitch_floats;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// Philox4x32-10: counter-based, so the dropout keep-mask is a pure function of
// (seed, step, site, element index) and is re-derived in the backward pass instead of stored.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}

struct DropoutCfg {
  uint32_t threshold;   // keep iff rnd >= threshold   (threshold = p * 2^32)
  float scale;          // 1 / (1 - p)
  uint2 key;            // seed
  uint32_t step_lo, step_hi_site;   // counter words 2,3
  int enabled;
  unsigned long long elem4_offset;  // added to the local float4 index: global position of a row-partitioned panel
};

inline DropoutCfg make_dropout(float p, uint64_t seed, uint64_t step, int site, bool training,
                               unsigned long long elem4_offset = 0) {
  DropoutCfg c;
  c.elem4_offset = elem4_offset;
  c.enabled = (training && p > 0.0f) ? 1 : 0;
  double t = static_cast<double>(p) * 4294967296.0;
  if (t > 4294967295.0) t = 4294967295.0;
  if (t < 0.0) t = 0.0;
  c.threshold = static_cast<uint32_t>(t);
  c.scale = p < 1.0f ? 1.0f / (1.0f - p) : 0.0f;
  c.key = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  c.step_lo = static_cast<uint32_t>(step);
  c.step_hi_site = (static_cast<uint32_t>(step >> 32) << 4) | static_cast<uint32_t>(site & 0xF);
  return c;
}

// keep-mask multipliers for the 4 consecutive floats starting at flat element index `elem4 * 4`
__device__ __forceinline__ float4 dropout_mult4(const DropoutCfg& c, uint64_t elem4) {
  elem4 += c.elem4_offset;
  const uint4 r = philox4x32_10(
      make_uint4(static_cast<uint32_t>(elem4), static_cast<uint32_t>(elem4 >> 32), c.step_lo, c.step_hi_site), c.key);
  float4 m;
  m.x = r.x >= c.threshold ? c.scale : 0.0f;
  m.y = r.y >= c.threshold ? c.scale : 0.0f;
  m.z = r.z >= c.threshold ? c.scale : 0.0f;
  m.w = r.w >= c.threshold ? c.scale : 0.0f;
  return m;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

#endif  // __CUDACC__

}  // namespace cgcn
