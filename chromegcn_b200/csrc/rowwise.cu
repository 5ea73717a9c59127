// Row-wise (HBM-streaming) kernels of the gated GCN: everything in ChromeGCN.forward
// (models/ChromeModels.py:34-52) and its autograd that is neither the SpMM nor a dense
// contraction, fused so that each activation panel is read and written once per stage.
//
// Layout: panels are [n][S][D] fp32 (S strands interleaved, D = DV*128).  One warp owns one
// window row at a time; lane l holds, per strand and per 128-column block v, the float4 at
// column v*128 + 4*l, so every access is a coalesced 512 B request and the per-row gate
// dot-product is one 5-step shuffle reduction.  Column reductions (bias / gate / BatchNorm
// statistics and gradients) are accumulated in registers across the rows a warp visits,
// combined per CTA in shared memory, written as per-CTA partials and summed in a fixed order
// in fp64 by a small finalize kernel: deterministic, no fp32 atomics.
#include "common.cuh"
#include "rowwise_args.cuh"

namespace cgcn {

constexpr int RW_WARPS = 8;
constexpr int RW_THREADS = RW_WARPS * 32;

int rowwise_grid(int n) {
  const int by_rows = (n + RW_WARPS - 1) / RW_WARPS;
  const int cap = sm_count() * 8;
  return by_rows < cap ? (by_rows > 0 ? by_rows : 1) : cap;
}
int rowwise_max_grid() { return sm_count() * 8; }

__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ void add4(float4& a, float4 b) {
  a.x += b.x;
  a.y += b.y;
  a.z += b.z;
  a.w += b.w;
}

// Combine per-warp register accumulators (K floats per warp, laid out by `store`) into one
// per-CTA partial row.  red: [RW_WARPS][K] floats of dynamic shared memory.
__device__ __forceinline__ void block_combine(float* red, int K, float* __restrict__ dst) {
  __syncthreads();
  for (int idx = threadIdx.x; idx < K; idx += RW_THREADS) {
    float t = red[idx];
#pragma unroll
    for (int w = 1; w < RW_WARPS; ++w) t += red[w * K + idx];
    dst[idx] = t;
  }
}


// Fixed-order parallel reduction of per-CTA partials.  A CTA is (32 columns) x (FIN_SLICES slices of the parts
// axis); a thread-block CLUSTER of gridDim.y CTAs (cluster dims 1 x gridDim.y x 1) shares one column block: slice
// (cluster rank, threadIdx.y) sums parts q = rank*FIN_SLICES + y, stepping by gridDim.y*FIN_SLICES, in fp64; the
// slices of a CTA are combined in slice order in its shared memory, and cluster rank 0 then reads the other CTAs'
// sums through distributed shared memory in rank order.  One launch, >= 8x the CTAs of a single-CTA-per-column-
// block reduction (these kernels sit on the critical path between two panel kernels), and still deterministic.
// Every thread of every CTA must call this; the result is valid in threads with threadIdx.y == 0 of cluster rank 0
// (`owner`).
constexpr int FIN_SLICES = 32;
constexpr int FIN_MAX_CLUSTER = 8;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ double ld_dsmem_f64(const double* local_smem_ptr, uint32_t cta_rank) {
  const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(local_smem_ptr));
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(cta_rank));
  double v;
  asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(ra) : "memory");
  return v;
}

template <int NV>
__device__ __forceinline__ bool reduce_parts(const float* __restrict__ partial, int parts, size_t stride,
                                             const int (&offs)[NV], bool active, double (&out)[NV]) {
  __shared__ double sh[FIN_SLICES][32][NV];
  __shared__ double cta_sum[32][NV];
  const uint32_t crank = cluster_ctarank(), csize = cluster_nctarank();
  const int step = static_cast<int>(csize) * FIN_SLICES;
  double acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = 0.0;
  if (active) {
    int q = static_cast<int>(crank) * FIN_SLICES + threadIdx.y;
    for (; q + 3 * step < parts; q += 4 * step) {                    // 4 x NV independent loads in flight
      float t[4][NV];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < NV; ++v) t[u][v] = partial[static_cast<size_t>(q + u * step) * stride + offs[v]];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] += static_cast<double>(t[u][v]);
    }
    for (; q < parts; q += step) {
#pragma unroll
      for (int v = 0; v < NV; ++v) acc[v] += static_cast<double>(partial[static_cast<size_t>(q) * stride + offs[v]]);
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) sh[threadIdx.y][threadIdx.x][v] = acc[v];
  __syncthreads();
  if (threadIdx.y == 0) {
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      double t = 0.0;
      for (int y = 0; y < FIN_SLICES; ++y) t += sh[y][threadIdx.x][v];
      cta_sum[threadIdx.x][v] = t;
    }
  }
  cluster_sync_all();                                               // every CTA's cta_sum is written and visible
  const bool owner = (crank == 0) && (threadIdx.y == 0);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    double t = 0.0;
    if (owner)
      for (uint32_t r = 0; r < csize; ++r) t += ld_dsmem_f64(&cta_sum[threadIdx.x][v], r);
    out[v] = t;
  }
  cluster_sync_all();                                               // nobody exits while rank 0 still reads its memory
  return owner;
}

// Launch a finalize kernel with cluster dims (1, cy, 1) over grid (gx, cy): cy CTAs share one column block.
static int finalize_cluster_y(int parts) {
  int cy = (parts + FIN_SLICES - 1) / FIN_SLICES;
  if (cy < 1) cy = 1;
  if (cy > FIN_MAX_CLUSTER) cy = FIN_MAX_CLUSTER;
  while (cy & (cy - 1)) cy &= cy - 1;                               // power of two <= 8
  return cy;
}
template <typename... KArgs, typename... Args>
static int launch_finalize(void (*kernel)(KArgs...), int gx, int cy, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(gx, cy, 1);
  cfg.blockDim = dim3(32, FIN_SLICES, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = cy;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_enabled() && !pdl_take_plain(stream)) ? 2 : 1;
  CGCN_CUDA(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
  return CGCN_OK;
}

// ------------------------------------------------------------------------------- gate forward

template <int DV, int S, bool STATS>
__global__ void __launch_bounds__(RW_THREADS) gate_fwd_kernel(const GateFwdArgs a) {
  pdl_grid_sync();
  constexpr int D = DV * 128;
  constexpr int K = 2 * S * D;
  extern __shared__ __align__(16) float red[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 wg[DV];
#pragma unroll
  for (int v = 0; v < DV; ++v) wg[v] = ldg4(a.wg + v * 128 + lane * 4);
  const float bg = __ldg(a.bg);
  float4 ssum[STATS ? S : 1][STATS ? DV : 1], ssq[STATS ? S : 1][STATS ? DV : 1];
  if constexpr (STATS) {
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
      for (int v = 0; v < DV; ++v) ssum[s][v] = ssq[s][v] = f4_zero();
  }
  for (int row = blockIdx.x * RW_WARPS + warp; row < a.n; row += gridDim.x * RW_WARPS) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const size_t base = (static_cast<size_t>(row) * S + s) * D + lane * 4;
      float4 z[DV];
      float dot = 0.f;
#pragma unroll
      for (int v = 0; v < DV; ++v) {
        const float4 y = ld4(a.y + base + v * 128);
        z[v] = make_float4(tanhf(y.x), tanhf(y.y), tanhf(y.z), tanhf(y.w));
        dot += dot4(z[v], wg[v]);
      }
      dot = warp_sum(dot);
      const float g = a.gate_off ? 1.0f : sigmoidf_(dot + bg);
      const float omg = 1.0f - g;
      if (lane == 0) a.g[static_cast<size_t>(row) * S + s] = g;
#pragma unroll
      for (int v = 0; v < DV; ++v) {
        const float4 x = ldg4(a.x + base + v * 128);
        float4 h = make_float4(omg * x.x + g * z[v].x, omg * x.y + g * z[v].y, omg * x.z + g * z[v].z,
                               omg * x.w + g * z[v].w);
        if (a.drop.enabled) {
          const float4 m = dropout_mult4(a.drop, (base + v * 128) >> 2);
          h = make_float4(h.x * m.x, h.y * m.y, h.z * m.z, h.w * m.w);
        }
        st4(a.z + base + v * 128, z[v]);
        st4(a.xo + base + v * 128, h);
        if constexpr (STATS) {
          const float4 r = make_float4(fmaxf(h.x, 0.f), fmaxf(h.y, 0.f), fmaxf(h.z, 0.f), fmaxf(h.w, 0.f));
          add4(ssum[s][v], r);
          add4(ssq[s][v], make_float4(r.x * r.x, r.y * r.y, r.z * r.z, r.w * r.w));
        }
      }
    }
  }
  if constexpr (STATS) {
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
      for (int v = 0; v < DV; ++v) {
        st4(red + warp * K + (0 * S + s) * D + v * 128 + lane * 4, ssum[s][v]);
        st4(red + warp * K + (1 * S + s) * D + v * 128 + lane * 4, ssq[s][v]);
      }
    block_combine(red, K, a.stats_partial + static_cast<size_t>(blockIdx.x) * K);
  }
}

// BatchNorm1d statistics (models/ChromeModels.py:49): per strand call, batch mean / biased variance
// over the n rows; running stats updated once per strand, in strand order, with the unbiased
// variance (torch.nn.BatchNorm1d semantics).  Eval mode: running stats.
template <int S>
__global__ void __launch_bounds__(32 * FIN_SLICES)
bn_finalize_kernel(const float* __restrict__ partial, int parts, int64_t n, int D, float eps, float momentum, int training,
                   float* __restrict__ running_mean, float* __restrict__ running_var, int64_t* __restrict__ num_batches,
                   float* __restrict__ mean_out, float* __restrict__ rstd_out, const double* __restrict__ presummed,
                   double* __restrict__ sums_out) {
  pdl_grid_sync();
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool active = c < D;
  const int K = 2 * S * D;
  if (!training) {
    if (active && threadIdx.y == 0 && blockIdx.y == 0) {
      const float m = running_mean[c];
      const float r = static_cast<float>(1.0 / sqrt(static_cast<double>(running_var[c]) + static_cast<double>(eps)));
      for (int s = 0; s < S; ++s) {
        mean_out[s * D + c] = m;
        rstd_out[s * D + c] = r;
      }
    }
    return;
  }
  int offs[2 * S];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    offs[2 * s] = (0 * S + s) * D + c;
    offs[2 * s + 1] = (1 * S + s) * D + c;
  }
  double sums[2 * S];
  bool owner = threadIdx.y == 0 && blockIdx.y == 0;
  if (presummed != nullptr) {                       // row-partitioned mode: sums already reduced over CTAs and ranks
#pragma unroll
    for (int v = 0; v < 2 * S; ++v) sums[v] = active ? presummed[offs[v]] : 0.0;
  } else {
    owner = reduce_parts<2 * S>(partial, parts, K, offs, active, sums);
  }
  if (!active || !owner) return;
  if (sums_out != nullptr) {                        // row-partitioned mode, first half: publish this rank's sums
#pragma unroll
    for (int v = 0; v < 2 * S; ++v) sums_out[offs[v]] = sums[v];
    return;
  }
  float rm = running_mean[c], rv = running_var[c];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const double mean = sums[2 * s] / n;
    double var = sums[2 * s + 1] / n - mean * mean;
    if (var < 0.0) var = 0.0;
    mean_out[s * D + c] = static_cast<float>(mean);
    rstd_out[s * D + c] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const double unbiased = n > 1 ? var * n / (n - 1.0) : var;
    rm = (1.0f - momentum) * rm + momentum * static_cast<float>(mean);
    rv = (1.0f - momentum) * rv + momentum * static_cast<float>(unbiased);
  }
  running_mean[c] = rm;
  running_var[c] = rv;
  if (c == 0 && num_batches != nullptr) *num_batches += S;
}

// hb = dropout(gamma * (relu(h) - mean) * rstd + beta)      (models/ChromeModels.py:48-50)

__global__ void __launch_bounds__(256) bn_apply_kernel(const BnApplyArgs a) {
  pdl_grid_sync();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < a.total4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t e = i * 4;
    const int c = static_cast<int>(e % a.D);
    const int s = static_cast<int>((e / a.D) % a.S);
    const float4 h = ldg4(a.h + e);
    const float4 mu = ldg4(a.mean + s * a.D + c), rs = ldg4(a.rstd + s * a.D + c);
    const float4 ga = ldg4(a.gamma + c), be = ldg4(a.beta + c);
    float4 o = make_float4((fmaxf(h.x, 0.f) - mu.x) * rs.x * ga.x + be.x, (fmaxf(h.y, 0.f) - mu.y) * rs.y * ga.y + be.y,
                           (fmaxf(h.z, 0.f) - mu.z) * rs.z * ga.z + be.z, (fmaxf(h.w, 0.f) - mu.w) * rs.w * ga.w + be.w);
    if (a.drop.enabled) {
      const float4 m = dropout_mult4(a.drop, static_cast<uint64_t>(i));
      o = make_float4(o.x * m.x, o.y * m.y, o.z * m.z, o.w * m.w);
    }
    st4(a.hb + e, o);
  }
}

// ------------------------------------------------------------------------------ BN backward sums

template <int DV, int S>
__global__ void __launch_bounds__(RW_THREADS, (DV == 1) ? 4 : 1) bn_bwd_reduce_kernel(const BnBwdReduceArgs a) {
  pdl_grid_sync();
  constexpr int D = DV * 128;
  constexpr int K = 2 * S * D;
  extern __shared__ __align__(16) float red[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 s1[S][DV], s2[S][DV];
#pragma unroll
  for (int s = 0; s < S; ++s)
#pragma unroll
    for (int v = 0; v < DV; ++v) s1[s][v] = s2[s][v] = f4_zero();
  for (int row = blockIdx.x * RW_WARPS + warp; row < a.n; row += gridDim.x * RW_WARPS) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const size_t base = (static_cast<size_t>(row) * S + s) * D + lane * 4;
#pragma unroll
      for (int v = 0; v < DV; ++v) {
        float4 g = ldg4(a.dhb + base + v * 128);
        if (a.drop.enabled) {
          const float4 m = dropout_mult4(a.drop, (base + v * 128) >> 2);
          g = make_float4(g.x * m.x, g.y * m.y, g.z * m.z, g.w * m.w);
        }
        const float4 h = ldg4(a.h + base + v * 128);
        const float4 mu = ldg4(a.mean + s * D + v * 128 + lane * 4), rs = ldg4(a.rstd + s * D + v * 128 + lane * 4);
        const float4 xh = make_float4((fmaxf(h.x, 0.f) - mu.x) * rs.x, (fmaxf(h.y, 0.f) - mu.y) * rs.y,
                                      (fmaxf(h.z, 0.f) - mu.z) * rs.z, (fmaxf(h.w, 0.f) - mu.w) * rs.w);
        add4(s1[s][v], g);
        add4(s2[s][v], make_float4(g.x * xh.x, g.y * xh.y, g.z * xh.z, g.w * xh.w));
      }
    }
  }
#pragma unroll
  for (int s = 0; s < S; ++s)
#pragma unroll
    for (int v = 0; v < DV; ++v) {
      st4(red + warp * K + (0 * S + s) * D + v * 128 + lane * 4, s1[s][v]);
      st4(red + warp * K + (1 * S + s) * D + v * 128 + lane * 4, s2[s][v]);
    }
  block_combine(red, K, a.partial + static_cast<size_t>(blockIdx.x) * K);
}

// c1 = mean(dbn), c2 = mean(dbn * xhat) per strand (zero in eval mode: running stats are constants);
// d gamma = sum_s sum dbn*xhat ; d beta = sum_s sum dbn.
template <int S>
__global__ void __launch_bounds__(32 * FIN_SLICES)
bn_bwd_finalize_kernel(const float* __restrict__ partial, int parts, int64_t n, int D, int training, float* __restrict__ c1,
                       float* __restrict__ c2, float* __restrict__ dgamma, float* __restrict__ dbeta,
                       const double* __restrict__ presummed, double* __restrict__ sums_out) {
  pdl_grid_sync();
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool active = c < D;
  const int K = 2 * S * D;
  int offs[2 * S];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    offs[2 * s] = (0 * S + s) * D + c;
    offs[2 * s + 1] = (1 * S + s) * D + c;
  }
  double sums[2 * S];
  bool owner = threadIdx.y == 0 && blockIdx.y == 0;
  if (presummed != nullptr) {
#pragma unroll
    for (int v = 0; v < 2 * S; ++v) sums[v] = active ? presummed[offs[v]] : 0.0;
  } else {
    owner = reduce_parts<2 * S>(partial, parts, K, offs, active, sums);
  }
  if (!active || !owner) return;
  if (presummed != nullptr) {                       // second half: c1 / c2 from the all-reduced sums; d gamma / d beta stay local
#pragma unroll
    for (int s = 0; s < S; ++s) {
      c1[s * D + c] = training ? static_cast<float>(sums[2 * s] / n) : 0.f;
      c2[s * D + c] = training ? static_cast<float>(sums[2 * s + 1] / n) : 0.f;
    }
    return;
  }
  if (sums_out != nullptr) {
#pragma unroll
    for (int v = 0; v < 2 * S; ++v) sums_out[offs[v]] = sums[v];
  }
  double tg = 0.0, tb = 0.0;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    if (sums_out == nullptr) {
      c1[s * D + c] = training ? static_cast<float>(sums[2 * s] / n) : 0.f;
      c2[s * D + c] = training ? static_cast<float>(sums[2 * s + 1] / n) : 0.f;
    }
    tb += sums[2 * s];
    tg += sums[2 * s + 1];
  }
  dgamma[c] = static_cast<float>(tg);
  dbeta[c] = static_cast<float>(tb);
}

// ------------------------------------------------------------------------------ gate backward

template <int DV, int S, int HEAD>
__global__ void __launch_bounds__(RW_THREADS, (DV == 1) ? 3 : 1) gate_bwd_kernel(const GateBwdArgs a) {
  pdl_grid_sync();
  constexpr int D = DV * 128;
  constexpr int K = 2 * D + 4;
  extern __shared__ __align__(16) float red[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 wg[DV], db[DV], dwg[DV];
  float dbg = 0.f;
#pragma unroll
  for (int v = 0; v < DV; ++v) {
    wg[v] = ldg4(a.wg + v * 128 + lane * 4);
    db[v] = dwg[v] = f4_zero();
  }
  for (int row = blockIdx.x * RW_WARPS + warp; row < a.n; row += gridDim.x * RW_WARPS) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const size_t base = (static_cast<size_t>(row) * S + s) * D + lane * 4;
      float4 dh[DV], z[DV], x[DV];
      float part = 0.f;
#pragma unroll
      for (int v = 0; v < DV; ++v) {
        float4 d = ldg4(a.dsrc + base + v * 128);
        if (a.drop.enabled) {
          const float4 m = dropout_mult4(a.drop, (base + v * 128) >> 2);
          d = make_float4(d.x * m.x, d.y * m.y, d.z * m.z, d.w * m.w);
        }
        if (HEAD) {
          const int co = s * D + v * 128 + lane * 4;
          const float4 h = ldg4(a.h + base + v * 128);
          const float4 mu = ldg4(a.mean + co), rs = ldg4(a.rstd + co), k1 = ldg4(a.c1 + co), k2 = ldg4(a.c2 + co);
          const float4 ga = ldg4(a.gamma + v * 128 + lane * 4);
          float4 r;
          r.x = h.x > 0.f ? ga.x * rs.x * (d.x - k1.x - (h.x - mu.x) * rs.x * k2.x) : 0.f;
          r.y = h.y > 0.f ? ga.y * rs.y * (d.y - k1.y - (h.y - mu.y) * rs.y * k2.y) : 0.f;
          r.z = h.z > 0.f ? ga.z * rs.z * (d.z - k1.z - (h.z - mu.z) * rs.z * k2.z) : 0.f;
          r.w = h.w > 0.f ? ga.w * rs.w * (d.w - k1.w - (h.w - mu.w) * rs.w * k2.w) : 0.f;
          d = r;
        }
        dh[v] = d;
        z[v] = ldg4(a.z + base + v * 128);
        x[v] = ldg4(a.x + base + v * 128);
        part += d.x * (z[v].x - x[v].x) + d.y * (z[v].y - x[v].y) + d.z * (z[v].z - x[v].z) + d.w * (z[v].w - x[v].w);
      }
      part = warp_sum(part);
      const float g = __ldg(a.g + static_cast<size_t>(row) * S + s);
      const float dgp = part * g * (1.0f - g);
      const float omg = 1.0f - g;
      const float inv = a.scale_rowptr != nullptr ? inv_degree(a.scale_rowptr, row) : 1.0f;
#pragma unroll
      for (int v = 0; v < DV; ++v) {
        const float4 dz = make_float4(g * dh[v].x + dgp * wg[v].x, g * dh[v].y + dgp * wg[v].y,
                                      g * dh[v].z + dgp * wg[v].z, g * dh[v].w + dgp * wg[v].w);
        const float4 dy = make_float4(dz.x * (1.0f - z[v].x * z[v].x), dz.y * (1.0f - z[v].y * z[v].y),
                                      dz.z * (1.0f - z[v].z * z[v].z), dz.w * (1.0f - z[v].w * z[v].w));
        st4(a.dy + base + v * 128, make_float4(dy.x * inv, dy.y * inv, dy.z * inv, dy.w * inv));
        if (a.dxd != nullptr)
          st4(a.dxd + base + v * 128, make_float4(omg * dh[v].x, omg * dh[v].y, omg * dh[v].z, omg * dh[v].w));
        add4(db[v], dy);
        add4(dwg[v], make_float4(dgp * z[v].x, dgp * z[v].y, dgp * z[v].z, dgp * z[v].w));
      }
      dbg += dgp;                      // identical in every lane
    }
  }
#pragma unroll
  for (int v = 0; v < DV; ++v) {
    st4(red + warp * K + v * 128 + lane * 4, db[v]);
    st4(red + warp * K + D + v * 128 + lane * 4, dwg[v]);
  }
  if (lane < 4) red[warp * K + 2 * D + lane] = (lane == 0) ? dbg : 0.f;
  block_combine(red, K, a.partial + static_cast<size_t>(blockIdx.x) * K);
}

// out[k] = sum over parts of partial[part*stride + k], routed to up to three destinations
struct ColFinalizeArgs {
  const float* partial;
  int parts, stride;
  float* dst[3];
  int begin[3], len[3];
};

__global__ void __launch_bounds__(32 * FIN_SLICES) col_finalize_kernel(const ColFinalizeArgs a) {
  pdl_grid_sync();
  const int t = blockIdx.x * 32 + threadIdx.x;        // index into the concatenation of the segments
  int q = -1, local = 0, base = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (q < 0 && a.dst[i] != nullptr && t >= base && t < base + a.len[i]) {
      q = i;
      local = t - base;
    }
    if (a.dst[i] != nullptr) base += a.len[i];
  }
  const bool active = q >= 0;
  int offs[1] = {active ? a.begin[q] + local : 0};
  double out[1];
  const bool owner = reduce_parts<1>(a.partial, a.parts, a.stride, offs, active, out);
  if (active && owner) a.dst[q][local] = static_cast<float>(out[0]);
}

// ------------------------------------------------------------------------------ generic column sum
// dst[c] = sum_r X[r][c], X [rows][cols] with arbitrary cols <= 128 (d out.bias = column sums of the
// logit gradient).  One thread per column, 8 rows in flight.
__global__ void __launch_bounds__(128) colsum_partial_kernel(const float* __restrict__ X, int64_t rows, int cols, int ld,
                                                             int64_t rows_per_cta, float* __restrict__ partial) {
  pdl_grid_sync();
  const int c = threadIdx.x;
  const int64_t r0 = blockIdx.x * rows_per_cta;
  const int64_t r1 = min(r0 + rows_per_cta, rows);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c < cols) {
    int64_t r = r0;
    for (; r + 8 <= r1; r += 8) {
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] += __ldg(X + (r + u) * ld + c);
    }
    for (; r < r1; ++r) acc[0] += __ldg(X + r * ld + c);
  }
  const float t = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
  partial[static_cast<size_t>(blockIdx.x) * 128 + c] = (c < cols) ? t : 0.f;
}

// ------------------------------------------------------------------------------ BCE-with-logits
struct BceArgs {
  const float* out;    // [n][S][C]
  const float* target; // [n][C], or NULL when target_bits is set
  const uint32_t* target_bits;   // [n][(C+31)/32] little-endian bit rows (bit c of a row = label c), or NULL
  float* probs;        // [n][C] or NULL
  float* out_grad;     // [n][S][C] or NULL
  float* partial;      // [grid]
  int64_t total;       // n*ld
  int C, S, ld;        // ld = floats per (row, strand) of out / out_grad
  float inv_count;     // 1 / (n*C)
};

template <int SS>
__global__ void __launch_bounds__(256) bce_kernel(const BceArgs a) {
  pdl_grid_sync();
  __shared__ float wsum[8];
  float local = 0.f;
  constexpr uint32_t S = SS;                                    // compile-time: the strand loads issue back to back
  const float inv_s = 1.0f / S;
  const uint32_t total = static_cast<uint32_t>(a.total), C = static_cast<uint32_t>(a.C);
  const uint32_t LD = static_cast<uint32_t>(a.ld);
  const uint32_t WPR = (C + 31u) >> 5;                           // words per bit-packed target row
  // flat over the n x ld elements (padding columns only get a zero gradient), 4 independent elements per
  // thread per trip (coalesced, 32-bit index math)
  for (uint32_t e0 = blockIdx.x * 1024u + threadIdx.x; e0 < total; e0 += gridDim.x * 1024u) {
    float p[4], t[4];
    uint32_t ob[4], rr[4], cc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t e = e0 + u * 256u;
      p[u] = 0.f;
      t[u] = 0.f;
      ob[u] = rr[u] = cc[u] = 0;
      if (e < total) {
        rr[u] = e / LD;
        cc[u] = e - rr[u] * LD;
        ob[u] = rr[u] * S * LD + cc[u];                         // (r*S + 0)*ld + c
        if (cc[u] < C) {
          float ps[SS];
#pragma unroll
          for (uint32_t s = 0; s < S; ++s) ps[s] = __ldg(a.out + ob[u] + s * LD);
          t[u] = (a.target_bits != nullptr)
                     ? static_cast<float>((__ldg(a.target_bits + rr[u] * WPR + (cc[u] >> 5)) >> (cc[u] & 31u)) & 1u)
                     : __ldg(a.target + rr[u] * C + cc[u]);
#pragma unroll
          for (uint32_t s = 0; s < S; ++s) p[u] += ps[s];
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t e = e0 + u * 256u;
      if (e >= total) continue;
      if (cc[u] >= C) {
        if (a.out_grad != nullptr) {
#pragma unroll
          for (uint32_t s = 0; s < S; ++s) a.out_grad[ob[u] + s * LD] = 0.f;
        }
        continue;
      }
      const float pm = p[u] * inv_s;                            // (pred_f + pred_r) / 2, finetune.py:43
      const float en = expf(-fabsf(pm));                        // one exponential serves the loss and the sigmoid
      local += fmaxf(pm, 0.f) - pm * t[u] + log1pf(en);         // BCE-with-logits, finetune.py:45
      const float rinv = 1.0f / (1.0f + en);
      const float pr = pm >= 0.f ? rinv : en * rinv;
      if (a.probs != nullptr) a.probs[rr[u] * C + cc[u]] = pr;  // F.sigmoid(pred), finetune.py:52
      if (a.out_grad != nullptr) {
        const float gsc = (pr - t[u]) * a.inv_count * inv_s;
#pragma unroll
        for (uint32_t s = 0; s < S; ++s) a.out_grad[ob[u] + s * LD] = gsc;
      }
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += wsum[w];
    a.partial[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256) bce_finalize_kernel(const float* __restrict__ partial, int parts, float inv_count,
                                                            float* loss_sum) {
  pdl_grid_sync();
  __shared__ double sh[256];
  double s = 0.0;
  for (int p = threadIdx.x; p < parts; p += 256) s += static_cast<double>(partial[p]);
  sh[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 256; ++i) t += sh[i];
    *loss_sum += static_cast<float>(t * static_cast<double>(inv_count));
  }
}

// ------------------------------------------------------------------------------ optimisers
__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf, int64_t count,
                           float lr, float momentum, float wd, float gscale) {
  pdl_grid_sync();
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  const float w = p[i];
  float d = g[i] * gscale;
  d = fmaf(wd, w, d);                       // grad.add(param, alpha=weight_decay)
  const float b = momentum * buf[i] + d;    // buf.mul_(momentum).add_(grad)   (buf starts at 0 == first-step clone)
  buf[i] = b;
  p[i] = w - lr * b;                        // param.add_(buf, alpha=-lr)
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t count, float lr, float b1, float b2, float eps,
                            float bc1, float bc2_sqrt, float gscale) {
  pdl_grid_sync();
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  const float gr = g[i] * gscale;
  const float mi = m[i] + (gr - m[i]) * (1.0f - b1);          // exp_avg.lerp_(grad, 1 - beta1)
  const float vi = b2 * v[i] + (1.0f - b2) * gr * gr;          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1-beta2)
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] = p[i] - (lr / bc1) * (mi / denom);
}

// ------------------------------------------------------------------------------ utilities
__global__ void interleave_kernel(const float* s0, const float* s1, int S, int64_t n, int d4, float4* dst) {
  pdl_grid_sync();
  const int64_t total = n * S * d4;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % d4);
    const int s = static_cast<int>((i / d4) % S);
    const int64_t r = i / (static_cast<int64_t>(d4) * S);
    const float* src = s == 0 ? s0 : s1;
    dst[i] = __ldg(reinterpret_cast<const float4*>(src) + r * d4 + c);
  }
}

__global__ void deinterleave_kernel(const float* src, int S, int64_t n, int w, float* d0, float* d1) {
  pdl_grid_sync();
  const int64_t total = n * S * w;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % w);
    const int s = static_cast<int>((i / w) % S);
    const int64_t r = i / (static_cast<int64_t>(w) * S);
    (s == 0 ? d0 : d1)[r * w + c] = __ldg(src + i);
  }
}

__global__ void dropout_mask_kernel(float4* mask, int64_t total4, DropoutCfg cfg) {
  pdl_grid_sync();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    mask[i] = cfg.enabled ? dropout_mult4(cfg, static_cast<uint64_t>(i)) : make_float4(1.f, 1.f, 1.f, 1.f);
}

// Read-bandwidth probe (tools/l2_bw.py): the grid strides over the buffer `reps` times (each element is read once per
// repetition, by one thread) with 8 independent 128-bit loads in flight per thread.  A buffer that fits L2 (<= 64 MB) measures the L2 -> SM read rate the gather kernels
// can hope for; a buffer of several GB measures the HBM read rate.
__global__ void __launch_bounds__(256) membw_read_kernel(const float4* __restrict__ p, size_t n4, int reps, float* sink) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (int r = 0; r < reps; ++r) {
    size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    for (; i + 7 * stride < n4; i += 8 * stride) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldcg(p + i + u * stride);      // L2 only: a hit in L1 would not be an L2 read
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        acc.x += v[u].x;
        acc.y += v[u].y;
        acc.z += v[u].z;
        acc.w += v[u].w;
      }
    }
    for (; i < n4; i += stride) {
      const float4 v = __ldcg(p + i);
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
  }
  if (acc.x + acc.y + acc.z + acc.w == 1.2345e-30f) *sink = acc.x;      // keeps the loads alive
}

// =============================================================================== host launchers
static int flat_grid(int64_t work_items, int threads) {
  int64_t b = (work_items + threads - 1) / threads;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

template <typename KernelT>
static int ensure_smem(KernelT kernel, size_t bytes) {
  if (bytes > 48 * 1024) CGCN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
  return CGCN_OK;
}

#define DISPATCH_DV_S(DVV, SV, MACRO)                                                              \
  do {                                                                                             \
    if ((DVV) == 1 && (SV) == 1) { MACRO(1, 1); }                                                  \
    else if ((DVV) == 1 && (SV) == 2) { MACRO(1, 2); }                                             \
    else if ((DVV) == 2 && (SV) == 1) { MACRO(2, 1); }                                             \
    else if ((DVV) == 2 && (SV) == 2) { MACRO(2, 2); }                                             \
    else if ((DVV) == 4 && (SV) == 1) { MACRO(4, 1); }                                             \
    else if ((DVV) == 4 && (SV) == 2) { MACRO(4, 2); }                                             \
    else { set_error("unsupported d=%d strands=%d (d must be 128, 256 or 512; strands 1 or 2)", (DVV) * 128, (SV)); return CGCN_ERR_INVALID; } \
  } while (0)

int gate_fwd_launch(const GateFwdArgs& a, int d, int S, bool stats, int* grid_out, cudaStream_t stream) {
  const int grid = rowwise_grid(a.n);
  if (grid_out) *grid_out = grid;
  const int dv = d / 128;
  const size_t smem = stats ? static_cast<size_t>(RW_WARPS) * 2 * S * d * sizeof(float) : 0;
#define GF(DVC, SC)                                                                          \
  if (stats) {                                                                               \
    CGCN_TRY(ensure_smem(gate_fwd_kernel<DVC, SC, true>, smem));                             \
    CGCN_CUDA(launch_k(gate_fwd_kernel<DVC, SC, true>, dim3(grid), dim3(RW_THREADS), smem, stream, a)); \
  } else {                                                                                   \
    CGCN_CUDA(launch_k(gate_fwd_kernel<DVC, SC, false>, dim3(grid), dim3(RW_THREADS), 0, stream, a));   \
  }
  DISPATCH_DV_S(dv, S, GF);
#undef GF
  return check_launch("gate_fwd_kernel");
}

int bn_finalize_launch(const float* partial, int parts, int64_t n, int S, int D, float eps, float momentum, int training,
                       float* running_mean, float* running_var, int64_t* nbt, float* mean_out, float* rstd_out,
                       const double* presummed, double* sums_out, cudaStream_t stream) {
  const int cy = (training && presummed == nullptr) ? finalize_cluster_y(parts) : 1;
  if (S == 1)
    CGCN_TRY(launch_finalize(bn_finalize_kernel<1>, (D + 31) / 32, cy, stream, partial, parts, n, D, eps, momentum, training,
                             running_mean, running_var, nbt, mean_out, rstd_out, presummed, sums_out));
  else
    CGCN_TRY(launch_finalize(bn_finalize_kernel<2>, (D + 31) / 32, cy, stream, partial, parts, n, D, eps, momentum, training,
                             running_mean, running_var, nbt, mean_out, rstd_out, presummed, sums_out));
  return check_launch("bn_finalize_kernel");
}

int bn_apply_launch(const BnApplyArgs& a, cudaStream_t stream) {
  CGCN_CUDA(launch_k(bn_apply_kernel, dim3(flat_grid(a.total4, 256)), dim3(256), 0, stream, a));
  return check_launch("bn_apply_kernel");
}

int bn_bwd_reduce_launch(const BnBwdReduceArgs& a, int d, int S, int* grid_out, cudaStream_t stream) {
  const int grid = rowwise_grid(a.n);
  if (grid_out) *grid_out = grid;
  const int dv = d / 128;
  const size_t smem = static_cast<size_t>(RW_WARPS) * 2 * S * d * sizeof(float);
#define BR(DVC, SC)                                                    \
  CGCN_TRY(ensure_smem(bn_bwd_reduce_kernel<DVC, SC>, smem));          \
  CGCN_CUDA(launch_k(bn_bwd_reduce_kernel<DVC, SC>, dim3(grid), dim3(RW_THREADS), smem, stream, a));
  DISPATCH_DV_S(dv, S, BR);
#undef BR
  return check_launch("bn_bwd_reduce_kernel");
}

int bn_bwd_finalize_launch(const float* partial, int parts, int64_t n, int S, int D, int training, float* c1, float* c2,
                           float* dgamma, float* dbeta, const double* presummed, double* sums_out, cudaStream_t stream) {
  const int cy = (presummed == nullptr) ? finalize_cluster_y(parts) : 1;
  if (S == 1)
    CGCN_TRY(launch_finalize(bn_bwd_finalize_kernel<1>, (D + 31) / 32, cy, stream, partial, parts, n, D, training, c1, c2,
                             dgamma, dbeta, presummed, sums_out));
  else
    CGCN_TRY(launch_finalize(bn_bwd_finalize_kernel<2>, (D + 31) / 32, cy, stream, partial, parts, n, D, training, c1, c2,
                             dgamma, dbeta, presummed, sums_out));
  return check_launch("bn_bwd_finalize_kernel");
}

// The kernel only; its per-CTA partials are reduced by gate_bwd_finalize_launch (possibly on another stream:
// the bias / gate gradients are not on the critical path of the backward pass).
int gate_bwd_launch(const GateBwdArgs& a, int d, int S, bool head, int* grid_out, cudaStream_t stream) {
  const int grid = rowwise_grid(a.n);
  if (grid_out) *grid_out = grid;
  const int dv = d / 128;
  const int K = 2 * d + 4;
  const size_t smem = static_cast<size_t>(RW_WARPS) * K * sizeof(float);
#define GBW(DVC, SC)                                                            \
  if (head) {                                                                   \
    CGCN_TRY(ensure_smem(gate_bwd_kernel<DVC, SC, 1>, smem));                   \
    CGCN_CUDA(launch_k(gate_bwd_kernel<DVC, SC, 1>, dim3(grid), dim3(RW_THREADS), smem, stream, a)); \
  } else {                                                                      \
    CGCN_TRY(ensure_smem(gate_bwd_kernel<DVC, SC, 0>, smem));                   \
    CGCN_CUDA(launch_k(gate_bwd_kernel<DVC, SC, 0>, dim3(grid), dim3(RW_THREADS), smem, stream, a)); \
  }
  DISPATCH_DV_S(dv, S, GBW);
#undef GBW
  return check_launch("gate_bwd_kernel");
}

int gate_bwd_finalize_launch(const float* partial, int grid, int d, float* db, float* dwg, float* dbg,
                             cudaStream_t stream) {
  const int K = 2 * d + 4;
  ColFinalizeArgs f{};
  f.partial = partial;
  f.parts = grid;
  f.stride = K;
  f.dst[0] = db;  f.begin[0] = 0;      f.len[0] = d;
  f.dst[1] = dwg; f.begin[1] = d;      f.len[1] = d;
  f.dst[2] = dbg; f.begin[2] = 2 * d;  f.len[2] = 1;
  CGCN_TRY(launch_finalize(col_finalize_kernel, (2 * d + 1 + 31) / 32, finalize_cluster_y(grid), stream, f));
  return check_launch("col_finalize_kernel");
}

int colsum_launch(const float* X, int64_t rows, int cols, int ld, float* dst, float* partial, cudaStream_t stream) {
  CGCN_REQUIRE(cols >= 1 && cols <= 128, "colsum: cols=%d", cols);
  const int64_t max_parts = static_cast<int64_t>(sm_count()) * 8;
  int64_t rows_per = (rows + max_parts - 1) / max_parts;
  if (rows_per < 64) rows_per = 64;
  const int parts = static_cast<int>((rows + rows_per - 1) / rows_per);
  CGCN_CUDA(launch_k(colsum_partial_kernel, dim3(parts), dim3(128), 0, stream, X, rows, cols, ld, rows_per, partial));
  CGCN_TRY(check_launch("colsum_partial_kernel"));
  ColFinalizeArgs f{};
  f.partial = partial;
  f.parts = parts;
  f.stride = 128;
  f.dst[0] = dst; f.begin[0] = 0; f.len[0] = cols;
  CGCN_TRY(launch_finalize(col_finalize_kernel, (cols + 31) / 32, finalize_cluster_y(parts), stream, f));
  return check_launch("col_finalize_kernel");
}

int bce_grid() { return sm_count() * 8; }

int bce_launch(const float* out, const float* target, const uint32_t* target_bits, int n, int C, int S, int ld, float* probs,
               float* loss_sum, float* out_grad, float* partial, int64_t n_total, cudaStream_t stream) {
  if (n_total <= 0) n_total = n;                       // row-partitioned graphs normalise by the global row count
  BceArgs a{out, target, target_bits, probs, out_grad, partial, static_cast<int64_t>(n) * ld, C, S, ld,
            static_cast<float>(1.0 / (static_cast<double>(n_total) * C))};
  CGCN_REQUIRE(a.total * S < 4294967296LL, "cgcn_bce_loss: n * nclass * strands must fit 32 bits");
  int grid = static_cast<int>((a.total + 1023) / 1024);
  if (grid > bce_grid()) grid = bce_grid();
  if (grid < 1) grid = 1;
  if (S == 1) CGCN_CUDA(launch_k(bce_kernel<1>, dim3(grid), dim3(256), 0, stream, a));
  else CGCN_CUDA(launch_k(bce_kernel<2>, dim3(grid), dim3(256), 0, stream, a));
  CGCN_TRY(check_launch("bce_kernel"));
  CGCN_CUDA(launch_k(bce_finalize_kernel, dim3(1), dim3(256), 0, stream, partial, grid, a.inv_count, loss_sum));
  return check_launch("bce_finalize_kernel");
}

}  // namespace cgcn

using namespace cgcn;

extern "C" size_t cgcn_bce_workspace_bytes(int32_t n, int32_t nclass) {
  (void)n;
  (void)nclass;
  return static_cast<size_t>(bce_grid()) * sizeof(float) + 256;
}

extern "C" int cgcn_bce_loss(const float* out, const float* target, int32_t n, int32_t nclass, int32_t strands,
                             int32_t out_ld, int64_t n_total, float* probs, float* loss_sum_out, float* out_grad,
                             void* workspace, size_t workspace_bytes, cgcn_stream_t stream) {
  CGCN_REQUIRE(out && target && loss_sum_out, "cgcn_bce_loss: null argument");
  CGCN_REQUIRE(n >= 1 && nclass >= 1 && (strands == 1 || strands == 2), "cgcn_bce_loss: bad shape");
  if (out_ld <= 0) out_ld = nclass;
  CGCN_REQUIRE(out_ld >= nclass, "cgcn_bce_loss: out_ld %d < nclass %d", out_ld, nclass);
  if (workspace == nullptr || workspace_bytes < cgcn_bce_workspace_bytes(n, nclass)) {
    set_error("cgcn_bce_loss: workspace too small");
    return CGCN_ERR_WORKSPACE;
  }
  return bce_launch(out, target, nullptr, n, nclass, strands, out_ld, probs, loss_sum_out, out_grad,
                    static_cast<float*>(workspace), n_total, static_cast<cudaStream_t>(stream));
}

extern "C" int cgcn_bce_loss_bits(const float* out, const uint32_t* target_bits, int32_t n, int32_t nclass, int32_t strands,
                                  int32_t out_ld, int64_t n_total, float* probs, float* loss_sum_out, float* out_grad,
                                  void* workspace, size_t workspace_bytes, cgcn_stream_t stream) {
  CGCN_REQUIRE(out && target_bits && loss_sum_out, "cgcn_bce_loss_bits: null argument");
  CGCN_REQUIRE(n >= 1 && nclass >= 1 && (strands == 1 || strands == 2), "cgcn_bce_loss_bits: bad shape");
  if (out_ld <= 0) out_ld = nclass;
  CGCN_REQUIRE(out_ld >= nclass, "cgcn_bce_loss_bits: out_ld %d < nclass %d", out_ld, nclass);
  if (workspace == nullptr || workspace_bytes < cgcn_bce_workspace_bytes(n, nclass)) {
    set_error("cgcn_bce_loss_bits: workspace too small");
    return CGCN_ERR_WORKSPACE;
  }
  return bce_launch(out, nullptr, target_bits, n, nclass, strands, out_ld, probs, loss_sum_out, out_grad,
                    static_cast<float*>(workspace), n_total, static_cast<cudaStream_t>(stream));
}

extern "C" int cgcn_sgd_step(float* params, const float* grads, float* momentum_buf, int64_t count, float lr,
                             float momentum, float weight_decay, float grad_scale, cgcn_stream_t stream) {
  CGCN_REQUIRE(params && grads && momentum_buf && count >= 0, "cgcn_sgd_step: null argument");
  if (count == 0) return CGCN_OK;
  sgd_kernel<<<static_cast<int>((count + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      params, grads, momentum_buf, count, lr, momentum, weight_decay, grad_scale);
  return check_launch("sgd_kernel");
}

extern "C" int cgcn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t count,
                              float lr, float beta1, float beta2, float eps, int64_t step_index, float grad_scale,
                              cgcn_stream_t stream) {
  CGCN_REQUIRE(params && grads && exp_avg && exp_avg_sq && count >= 0 && step_index >= 1, "cgcn_adam_step: bad argument");
  if (count == 0) return CGCN_OK;
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), static_cast<double>(step_index));
  const double bc2 = 1.0 - pow(static_cast<double>(beta2), static_cast<double>(step_index));
  adam_kernel<<<static_cast<int>((count + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      params, grads, exp_avg, exp_avg_sq, count, lr, beta1, beta2, eps, static_cast<float>(bc1),
      static_cast<float>(sqrt(bc2)), grad_scale);
  return check_launch("adam_kernel");
}

extern "C" int cgcn_membw_read(const float* buf, size_t bytes, int32_t reps, float* sink, cgcn_stream_t stream) {
  CGCN_REQUIRE(buf && sink && bytes >= 16 && reps >= 1, "cgcn_membw_read: bad argument");
  membw_read_kernel<<<sm_count() * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const float4*>(buf), bytes / 16,
                                                                                reps, sink);
  return check_launch("membw_read_kernel");
}

extern "C" int cgcn_interleave_strands(const float* const* src_host, int32_t strands, int32_t n, int32_t d, float* dst,
                                       cgcn_stream_t stream) {
  CGCN_REQUIRE(src_host && dst && (strands == 1 || strands == 2) && d % 4 == 0, "cgcn_interleave_strands: bad argument");
  if (n <= 0) return CGCN_OK;
  const int64_t total = static_cast<int64_t>(n) * strands * (d / 4);
  interleave_kernel<<<flat_grid(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src_host[0], strands == 2 ? src_host[1] : src_host[0], strands, n, d / 4, reinterpret_cast<float4*>(dst));
  return check_launch("interleave_kernel");
}

extern "C" int cgcn_deinterleave_strands(const float* src, int32_t strands, int32_t n, int32_t width,
                                         float* const* dst_host, cgcn_stream_t stream) {
  CGCN_REQUIRE(src && dst_host && (strands == 1 || strands == 2) && width >= 1, "cgcn_deinterleave_strands: bad argument");
  if (n <= 0) return CGCN_OK;
  const int64_t total = static_cast<int64_t>(n) * strands * width;
  deinterleave_kernel<<<flat_grid(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, strands, n, width, dst_host[0], strands == 2 ? dst_host[1] : dst_host[0]);
  return check_launch("deinterleave_kernel");
}

extern "C" int cgcn_dropout_mask(float* mask, int32_t n, int32_t strands, int32_t d, float p, uint64_t seed,
                                 uint64_t step, int32_t site, cgcn_stream_t stream) {
  CGCN_REQUIRE(mask && d % 4 == 0 && p >= 0.f && p < 1.f, "cgcn_dropout_mask: bad argument");
  const int64_t total4 = static_cast<int64_t>(n) * strands * d / 4;
  if (total4 <= 0) return CGCN_OK;
  const DropoutCfg cfg = make_dropout(p, seed, step, site, true);
  dropout_mask_kernel<<<flat_grid(total4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<float4*>(mask), total4, cfg);
  return check_launch("dropout_mask_kernel");
}
