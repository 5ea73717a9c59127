// Pattern-only CSR SpMM over a strand-interleaved fp32 feature panel (sm_100a).
//
//   out[i,:] = scale_i * sum_{j in row i of bin(A+I)} x[j,:]  (+ residual[i,:])
//
// replaces torch.spmm(adj, support) of models/SubLayers.py:46 with adj = D^-1 bin(A+I) built by
// utils/util_methods.py:99-106,152-165 (scale_mode 1), and its autograd transpose
// A_hat^T G = P (D^-1 G) (scale_mode 0, the D^-1 having been applied upstream).
//
// There is no value array: every stored entry of row i equals 1/deg_i, and deg_i is
// rowptr[i+1]-rowptr[i], so the kernel's HBM/L2 traffic is colidx + one gathered row per entry
// + one written row per node.  One warp owns one row; a row of the panel is VEC*512 bytes and
// each lane reads VEC 128-bit words of it, so a gather is VEC fully coalesced 512 B requests.
// Column indices are fetched 32 at a time (coalesced) and broadcast by shuffle; 8 independent
// 128-bit loads per lane are kept in flight.  Summation runs in CSR (ascending column) order,
// so results are run-to-run deterministic.  Rows longer than LONG_ROW are split over the
// 8 warps of the CTA and combined in shared memory in a fixed order.
#include <cstring>

#include "common.cuh"

namespace cgcn {

constexpr int SPMM_WARPS = 8;
constexpr int LONG_ROW = 512;

// Where the gathered rows come from: the local panel x (pattern, or weighted by vals), or the panel spread over the
// ranks' exchange buffers (PeerTable).
constexpr int ROWS_PATTERN = 0, ROWS_WEIGHTED = 1, ROWS_PEER = 2;

__device__ __forceinline__ const float* shfl_ptr(const float* p, int src) {
  const unsigned long long v = reinterpret_cast<unsigned long long>(p);
  const unsigned lo = __shfl_sync(0xffffffffu, static_cast<unsigned>(v), src);
  const unsigned hi = __shfl_sync(0xffffffffu, static_cast<unsigned>(v >> 32), src);
  return reinterpret_cast<const float*>((static_cast<unsigned long long>(hi) << 32) | lo);
}

// acc += the rows of entries [begin, end), in CSR order.  The local sources broadcast the column index and form the
// address after the shuffle; the peer source resolves the owner of its lane's column once per 32 entries and
// broadcasts the 64-bit row pointer, which keeps the lookup off the per-neighbour path.
template <int VEC, int SRC>
__device__ __forceinline__ void gather_range(const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                             const float* __restrict__ x, const PeerTable& peer, int begin, int end,
                                             int lane, float4 (&acc)[VEC]) {
  constexpr bool WEIGHTED = SRC == ROWS_WEIGHTED;
  constexpr int UNROLL = (VEC >= 8) ? 1 : (8 / VEC);
  constexpr size_t PITCH = static_cast<size_t>(VEC) * 128;
  for (int base = begin; base < end; base += 32) {
    const int mine = (base + lane < end) ? __ldg(colidx + base + lane) : 0;
    float wmine = 1.0f;
    if (WEIGHTED) wmine = (base + lane < end) ? __ldg(vals + base + lane) : 0.0f;
    const float* pmine = nullptr;
    if (SRC == ROWS_PEER) pmine = peer_row(peer, mine, PITCH);   // lanes past the end: never broadcast
    auto row = [&](int k, float& w) -> const float* {       // this lane's part of the batch's k-th row, and its weight
      if (SRC == ROWS_PEER) {
        w = 1.0f;
        return shfl_ptr(pmine, k) + lane * 4;
      }
      const int c = __shfl_sync(0xffffffffu, mine, k);
      w = WEIGHTED ? __shfl_sync(0xffffffffu, wmine, k) : 1.0f;
      return x + static_cast<size_t>(c) * PITCH + lane * 4;
    };
    const int cnt = min(32, end - base);
    int k = 0;
    for (; k + UNROLL <= cnt; k += UNROLL) {
      float4 v[UNROLL][VEC];
      float w[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const float* p = row(k + u, w[u]);
#pragma unroll
        for (int q = 0; q < VEC; ++q) v[u][q] = ldg4(p + q * 128);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int q = 0; q < VEC; ++q) {
          if (WEIGHTED) {
            acc[q].x = fmaf(w[u], v[u][q].x, acc[q].x);
            acc[q].y = fmaf(w[u], v[u][q].y, acc[q].y);
            acc[q].z = fmaf(w[u], v[u][q].z, acc[q].z);
            acc[q].w = fmaf(w[u], v[u][q].w, acc[q].w);
          } else {
            acc[q].x += v[u][q].x;
            acc[q].y += v[u][q].y;
            acc[q].z += v[u][q].z;
            acc[q].w += v[u][q].w;
          }
        }
      }
    }
    for (; k < cnt; ++k) {                         // fmaf(1, v, acc) == acc + v: one tail for every source
      float w1;
      const float* p = row(k, w1);
#pragma unroll
      for (int q = 0; q < VEC; ++q) {
        const float4 v = ldg4(p + q * 128);
        acc[q].x = fmaf(w1, v.x, acc[q].x);
        acc[q].y = fmaf(w1, v.y, acc[q].y);
        acc[q].z = fmaf(w1, v.z, acc[q].z);
        acc[q].w = fmaf(w1, v.w, acc[q].w);
      }
    }
  }
}

// x (local sources) or peer (ROWS_PEER) is the gathered panel; vals / row_inv are read by ROWS_WEIGHTED only.
template <int VEC, int SRC>
__global__ void __launch_bounds__(SPMM_WARPS * 32, (VEC <= 2) ? 5 : 2)
spmm_pattern_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, int n,
                    const float* __restrict__ x, float* __restrict__ out, int scale_mode,
                    const float* __restrict__ residual, const float* __restrict__ vals,
                    const float* __restrict__ row_inv, const __grid_constant__ PeerTable peer) {
  pdl_grid_sync();
  constexpr bool WEIGHTED = SRC == ROWS_WEIGHTED;
  constexpr size_t PITCH = static_cast<size_t>(VEC) * 128;
  __shared__ float4 red[SPMM_WARPS][VEC][32];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int row0 = blockIdx.x * SPMM_WARPS;
  const int row = row0 + warp;
  auto scale = [&](int r, int d) {
    return (scale_mode != 1) ? 1.0f : (WEIGHTED ? __ldg(row_inv + r) : (d > 0 ? __fdiv_rn(1.0f, static_cast<float>(d)) : 1.0f));
  };
  auto finish = [&](int r, int q, float s, float4 t) {          // out[r] = s * sum (+ residual[r]), float4 q of the lane
    t = make_float4(t.x * s, t.y * s, t.z * s, t.w * s);
    if (residual != nullptr) {
      const float4 e = ldg4(residual + static_cast<size_t>(r) * PITCH + lane * 4 + q * 128);
      t.x += e.x;
      t.y += e.y;
      t.z += e.z;
      t.w += e.w;
    }
    st4(out + static_cast<size_t>(r) * PITCH + lane * 4 + q * 128, t);
  };

  int start = 0, end = 0;
  if (row < n) {
    start = __ldg(rowptr + row);
    end = __ldg(rowptr + row + 1);
  }
  const int deg = end - start;
  if (row < n && deg <= LONG_ROW) {
    float4 acc[VEC];
#pragma unroll
    for (int q = 0; q < VEC; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    gather_range<VEC, SRC>(colidx, vals, x, peer, start, end, lane, acc);
    const float s = scale(row, deg);
#pragma unroll
    for (int q = 0; q < VEC; ++q) finish(row, q, s, acc[q]);
  }

  // hub rows: any row of this CTA longer than LONG_ROW is shared by all 8 warps
  const int any_long = __syncthreads_or(row < n && deg > LONG_ROW);
  if (!any_long) return;
  for (int r = 0; r < SPMM_WARPS; ++r) {
    const int lrow = row0 + r;
    if (lrow >= n) break;                                     // uniform across the CTA
    const int ls = __ldg(rowptr + lrow), le = __ldg(rowptr + lrow + 1);
    const int ldeg = le - ls;
    if (ldeg <= LONG_ROW) continue;                           // uniform across the CTA
    const int chunk = (ldeg + SPMM_WARPS - 1) / SPMM_WARPS;
    const int b = min(ls + warp * chunk, le), e = min(b + chunk, le);
    float4 acc[VEC];
#pragma unroll
    for (int q = 0; q < VEC; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    gather_range<VEC, SRC>(colidx, vals, x, peer, b, e, lane, acc);
#pragma unroll
    for (int q = 0; q < VEC; ++q) red[warp][q][lane] = acc[q];
    __syncthreads();
    if (warp == 0) {
      const float s = scale(lrow, ldeg);
#pragma unroll
      for (int q = 0; q < VEC; ++q) {
        float4 t = red[0][q][lane];
        for (int w = 1; w < SPMM_WARPS; ++w) {
          const float4 u = red[w][q][lane];
          t.x += u.x;
          t.y += u.y;
          t.z += u.z;
          t.w += u.w;
        }
        finish(lrow, q, s, t);
      }
    }
    __syncthreads();
  }
}

// One launch of spmm_pattern_kernel over g->n > 0 rows, after the entry point has checked its arguments.
// cgcn_spmm takes widths 128 x {1, 2, 3, 4, 6, 8}, cgcn_spmm_peer 128 x {1, 2, 4, 8}.
static int spmm_run(const cgcn_graph* g, int src, const float* x, const PeerTable& peer, float* out, int width,
                    int scale_mode, const float* residual, cudaStream_t stream) {
  const dim3 grid((g->n + SPMM_WARPS - 1) / SPMM_WARPS), block(SPMM_WARPS * 32);
#define SPMM_CASE(SRC, V)                                                                                          \
  case SRC * 16 + V:                                                                                               \
    CGCN_CUDA(launch_k(spmm_pattern_kernel<V, SRC>, grid, block, 0, stream, g->rowptr, g->colidx, g->n, x, out,    \
                       scale_mode, residual, g->vals, g->row_inv, peer));                                          \
    break;
#define SPMM_LOCAL_CASES(SRC) SPMM_CASE(SRC, 1) SPMM_CASE(SRC, 2) SPMM_CASE(SRC, 3) SPMM_CASE(SRC, 4) SPMM_CASE(SRC, 6) SPMM_CASE(SRC, 8)
  switch (src * 16 + width / 128) {
    SPMM_LOCAL_CASES(ROWS_PATTERN)
    SPMM_LOCAL_CASES(ROWS_WEIGHTED)
    SPMM_CASE(ROWS_PEER, 1)
    SPMM_CASE(ROWS_PEER, 2)
    SPMM_CASE(ROWS_PEER, 4)
    SPMM_CASE(ROWS_PEER, 8)
    default:
      if (src == ROWS_PEER)
        set_error("cgcn_spmm_peer: unsupported width %d (128, 256, 512 or 1024)", width);
      else
        set_error("cgcn_spmm: unsupported width %d", width);
      return CGCN_ERR_INVALID;
  }
#undef SPMM_LOCAL_CASES
#undef SPMM_CASE
  return check_launch("spmm_pattern_kernel");
}

int peer_table(PeerTable* t, const cgcn_peer_panel* pp, int n_local, const char* who) {
  CGCN_REQUIRE(pp != nullptr, "%s: null peer panel", who);
  CGCN_REQUIRE(pp->world >= 1 && pp->world <= CGCN_MAX_PEERS && pp->rank >= 0 && pp->rank < pp->world,
               "%s: peer panel world=%d rank=%d", who, pp->world, pp->rank);
  *t = PeerTable{};
  t->world = pp->world;
  for (int r = 0; r < pp->world; ++r) {
    CGCN_REQUIRE(pp->base[r] != nullptr && pp->row_begin[r] <= pp->row_begin[r + 1], "%s: bad peer block %d", who, r);
    t->base[r] = pp->base[r];
    t->begin[r] = pp->row_begin[r];
  }
  t->begin[pp->world] = pp->row_begin[pp->world];
  const int rows = pp->row_begin[pp->rank + 1] - pp->row_begin[pp->rank];
  CGCN_REQUIRE(rows == n_local, "%s: graph has %d rows, peer block %d", who, n_local, rows);
  return CGCN_OK;
}

int spmm_peer_launch(const cgcn_graph* g, const cgcn_peer_panel* pp, float* out, int width, int scale_mode,
                     const float* residual, cudaStream_t stream) {
  CGCN_REQUIRE(g != nullptr && g->rowptr != nullptr && (g->colidx != nullptr || g->nnz == 0), "cgcn_spmm_peer: null graph");
  CGCN_REQUIRE(out != nullptr, "cgcn_spmm_peer: null panel");
  CGCN_REQUIRE(g->vals == nullptr, "cgcn_spmm_peer: weighted graphs are not row-partitioned");
  CGCN_REQUIRE(scale_mode == 0 || scale_mode == 1, "cgcn_spmm_peer: scale_mode %d", scale_mode);
  CGCN_REQUIRE(width > 0 && width % 128 == 0 && width <= 1024, "cgcn_spmm_peer: width %d must be a multiple of 128, <= 1024", width);
  PeerTable t;
  CGCN_TRY(peer_table(&t, pp, g->n, "cgcn_spmm_peer"));
  for (int r = 0; r < t.world; ++r) CGCN_REQUIRE(t.base[r] != out, "cgcn_spmm_peer: in-place aggregation is not possible");
  if (g->n <= 0) return CGCN_OK;
  return spmm_run(g, ROWS_PEER, nullptr, t, out, width, scale_mode, residual, stream);
}

// ---- exchange buffers (CUDA IPC)
static int ipc_alloc(size_t bytes, void** ptr, unsigned char* handle) {
  CGCN_REQUIRE(ptr != nullptr && handle != nullptr && bytes > 0, "cgcn_peer_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  void* p = nullptr;
  CGCN_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    set_error("cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    return CGCN_ERR_CUDA;
  }
  memcpy(handle, &h, 64);
  *ptr = p;
  return CGCN_OK;
}

// ------------------------------------------------------------------------------------------------
// SDDMM over the stored pattern: out[e] = sum_c G[row(e), c] * S[col(e), c] for every stored entry e (CSR order) --
// the gradient of  Y = A S  with respect to the VALUES of A (d loss / d a_ij = <G_i, S_j>), which the A-saliency
// analysis of the reference (scripts/visualize.py:30-45: adj.requires_grad, |adj * adj.grad|) asks for.  Warp per row:
// the row of G stays in registers, one gathered row of S per stored entry, warp-reduced dot product.
template <int VEC>
__global__ void __launch_bounds__(SPMM_WARPS * 32) sddmm_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                                int n, const float* __restrict__ G, const float* __restrict__ S,
                                                                float* __restrict__ out) {
  constexpr size_t PITCH = static_cast<size_t>(VEC) * 128;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * SPMM_WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  const int start = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
  float4 g[VEC];
#pragma unroll
  for (int q = 0; q < VEC; ++q) g[q] = ldg4(G + static_cast<size_t>(row) * PITCH + q * 128 + lane * 4);
  for (int base = start; base < end; base += 32) {
    const int mine = (base + lane < end) ? __ldg(colidx + base + lane) : 0;
    const int cnt = min(32, end - base);
    float keep = 0.f;
    for (int k = 0; k < cnt; ++k) {
      const int c = __shfl_sync(0xffffffffu, mine, k);
      const float* p = S + static_cast<size_t>(c) * PITCH + lane * 4;
      float d = 0.f;
#pragma unroll
      for (int q = 0; q < VEC; ++q) {
        const float4 v = ldg4(p + q * 128);
        d += g[q].x * v.x + g[q].y * v.y + g[q].z * v.z + g[q].w * v.w;
      }
      d = warp_sum(d);
      if (lane == k) keep = d;
    }
    if (lane < cnt) out[base + lane] = keep;
  }
}

int sddmm_launch(const cgcn_graph* g, const float* G, const float* S, int width, float* out, cudaStream_t stream) {
  CGCN_REQUIRE(g != nullptr && g->rowptr != nullptr && (g->colidx != nullptr || g->nnz == 0), "cgcn_sddmm: null graph");
  CGCN_REQUIRE(G != nullptr && S != nullptr && (out != nullptr || g->nnz == 0), "cgcn_sddmm: null operand");
  CGCN_REQUIRE(width > 0 && width % 128 == 0 && width <= 1024, "cgcn_sddmm: width %d must be a multiple of 128, <= 1024", width);
  if (g->n <= 0 || g->nnz <= 0) return CGCN_OK;
  const dim3 grid((g->n + SPMM_WARPS - 1) / SPMM_WARPS), block(SPMM_WARPS * 32);
  switch (width / 128) {
    case 1: sddmm_kernel<1><<<grid, block, 0, stream>>>(g->rowptr, g->colidx, g->n, G, S, out); break;
    case 2: sddmm_kernel<2><<<grid, block, 0, stream>>>(g->rowptr, g->colidx, g->n, G, S, out); break;
    case 4: sddmm_kernel<4><<<grid, block, 0, stream>>>(g->rowptr, g->colidx, g->n, G, S, out); break;
    case 8: sddmm_kernel<8><<<grid, block, 0, stream>>>(g->rowptr, g->colidx, g->n, G, S, out); break;
    default:
      set_error("cgcn_sddmm: unsupported width %d (128, 256, 512 or 1024)", width);
      return CGCN_ERR_INVALID;
  }
  return check_launch("sddmm_kernel");
}

int spmm_launch(const cgcn_graph* g, const float* x, float* out, int width, int scale_mode, const float* residual,
                cudaStream_t stream) {
  CGCN_REQUIRE(g != nullptr && g->rowptr != nullptr && (g->colidx != nullptr || g->nnz == 0), "cgcn_spmm: null graph");
  CGCN_REQUIRE(x != nullptr && out != nullptr, "cgcn_spmm: null panel");
  CGCN_REQUIRE(x != out, "cgcn_spmm: in-place aggregation is not possible");
  CGCN_REQUIRE(scale_mode == 0 || scale_mode == 1, "cgcn_spmm: scale_mode %d", scale_mode);
  CGCN_REQUIRE(width > 0 && width % 128 == 0 && width <= 1024, "cgcn_spmm: width %d must be a multiple of 128, <= 1024", width);
  if (g->n <= 0) return CGCN_OK;
  const bool weighted = g->vals != nullptr;
  CGCN_REQUIRE(!weighted || g->row_inv != nullptr, "cgcn_spmm: weighted graph without row_inv");
  return spmm_run(g, weighted ? ROWS_WEIGHTED : ROWS_PATTERN, x, PeerTable{}, out, width, scale_mode, residual, stream);
}

}  // namespace cgcn

extern "C" int cgcn_spmm(const cgcn_graph* g, const float* x, float* out, int32_t width, int32_t scale_mode,
                         const float* residual, cgcn_stream_t stream) {
  return cgcn::spmm_launch(g, x, out, width, scale_mode, residual, static_cast<cudaStream_t>(stream));
}

extern "C" int cgcn_sddmm(const cgcn_graph* g, const float* G, const float* S, int32_t width, float* out_vals, cgcn_stream_t stream) {
  return cgcn::sddmm_launch(g, G, S, width, out_vals, static_cast<cudaStream_t>(stream));
}

extern "C" int cgcn_spmm_peer(const cgcn_graph* g, const cgcn_peer_panel* panel, float* out, int32_t width, int32_t scale_mode,
                              const float* residual, cgcn_stream_t stream) {
  return cgcn::spmm_peer_launch(g, panel, out, width, scale_mode, residual, static_cast<cudaStream_t>(stream));
}

extern "C" int cgcn_peer_alloc(size_t bytes, void** ptr_host, unsigned char handle_host[64]) {
  return cgcn::ipc_alloc(bytes, ptr_host, handle_host);
}

extern "C" int cgcn_peer_open(const unsigned char handle_host[64], void** ptr_host) {
  CGCN_REQUIRE(handle_host != nullptr && ptr_host != nullptr, "cgcn_peer_open: null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle_host, 64);
  void* p = nullptr;
  CGCN_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *ptr_host = p;
  return CGCN_OK;
}

extern "C" int cgcn_peer_close(void* ptr) {
  if (ptr == nullptr) return CGCN_OK;
  CGCN_CUDA(cudaIpcCloseMemHandle(ptr));
  return CGCN_OK;
}

extern "C" int cgcn_peer_free(void* ptr) {
  if (ptr == nullptr) return CGCN_OK;
  CGCN_CUDA(cudaFree(ptr));
  return CGCN_OK;
}

extern "C" int cgcn_peer_publish(void* exchange_buffer, const void* local_panel, size_t bytes, cgcn_stream_t stream) {
  CGCN_REQUIRE(exchange_buffer != nullptr && local_panel != nullptr, "cgcn_peer_publish: null argument");
  if (bytes == 0) return CGCN_OK;
  CGCN_CUDA(cudaMemcpyAsync(exchange_buffer, local_panel, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return CGCN_OK;
}
