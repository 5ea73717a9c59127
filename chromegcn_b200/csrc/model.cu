// ChromeGCN.forward / its autograd / the finetune train step, as sequences of the kernels in
// spmm.cu, gemm_*.cu and rowwise.cu on one stream (models/ChromeModels.py:34-52,
// finetune.py:39-53).  Also the library-level entry points (version, errors, device info).
//
// Per layer the reference computes  A_hat (x W) + b ; this path computes (A_hat x) W + b
// (same value up to fp32 rounding, SURVEY.md 3.2) because it makes
//   d loss / d W = (A_hat x)^T (d loss / d y)
// SpMM-free and lets the first layer skip its backward SpMM when nobody needs d loss / d x_in.
#include <cstdarg>
#include <cstdlib>

#include "common.cuh"
#include "fused_layer.cuh"
#include "rowwise_args.cuh"

namespace cgcn {

// ---- declarations of the launchers defined in the other translation units
int spmm_launch(const cgcn_graph* g, const float* x, float* out, int width, int scale_mode, const float* residual,
                cudaStream_t stream);
int spmm_peer_launch(const cgcn_graph* g, const cgcn_peer_panel* pp, float* out, int width, int scale_mode,
                     const float* residual, cudaStream_t stream);
int gemm_rowpanel_ffma(const float* A, int64_t lda, const float* B, int b_transposed, const float* bias, float* C,
                       int64_t ldc, int64_t m, int n, int k, const int32_t* rowscale_rowptr, const float* rowscale_inv, int rowscale_group,
                       cudaStream_t stream, int64_t ldb = 0, int accumulate = 0);
int gemm_gram_ffma(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t m, int ka,
                   int nb, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t gram_workspace_bytes(int64_t m);
int gemm_rowpanel_tc(const float* A, int64_t lda, const float* B, int b_transposed, const float* bias, float* C,
                     int64_t ldc, int64_t m, int n, int k, const int32_t* rowscale_rowptr, const float* rowscale_inv, int rowscale_group,
                     void* workspace, size_t workspace_bytes, const void* ready_image, cudaStream_t stream, int64_t ldb = 0,
                     int accumulate = 0);
int tc_prep_images(const TcImageSpec* specs, int count, cudaStream_t stream);
int gemm_gram_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t m, int ka,
                 int nb, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t stream);
bool tc_rowpanel_supported(int64_t lda, int64_t ldc, int n, int k, const void* A, const void* C);
bool tc_gram_supported(int64_t lda, int64_t ldb, int ka, int nb, const void* A, const void* B);
size_t tc_workspace_bytes();

int rowwise_max_grid();
int bce_launch(const float* out, const float* target, const uint32_t* target_bits, int n, int C, int S, int ld, float* probs,
               float* loss_sum, float* out_grad, float* partial, int64_t n_total, cudaStream_t stream);
int colsum_launch(const float* X, int64_t rows, int cols, int ld, float* dst, float* partial, cudaStream_t stream);
int bn_finalize_launch(const float* partial, int parts, int64_t n, int S, int D, float eps, float momentum, int training,
                       float* running_mean, float* running_var, int64_t* nbt, float* mean_out, float* rstd_out,
                       const double* presummed, double* sums_out, cudaStream_t stream);
int bn_bwd_finalize_launch(const float* partial, int parts, int64_t n, int S, int D, int training, float* c1, float* c2,
                           float* dgamma, float* dbeta, const double* presummed, double* sums_out, cudaStream_t stream);

// ---- error string / counters
static thread_local char tls_error[512] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tls_error, sizeof(tls_error), fmt, ap);
  va_end(ap);
}

// ---- programmatic dependent launch switches (common.cuh)
bool pdl_enabled() {
  static const bool on = getenv("CGCN_NO_PDL") == nullptr;
  return on;
}
static thread_local cudaStream_t tls_plain[4] = {nullptr, nullptr, nullptr, nullptr};
static thread_local bool tls_plain_set[4] = {false, false, false, false};
void pdl_plain_next(cudaStream_t stream) {
  for (int i = 0; i < 4; ++i)
    if (tls_plain_set[i] && tls_plain[i] == stream) return;
  for (int i = 0; i < 4; ++i)
    if (!tls_plain_set[i]) {
      tls_plain_set[i] = true;
      tls_plain[i] = stream;
      return;
    }
}
bool pdl_take_plain(cudaStream_t stream) {
  for (int i = 0; i < 4; ++i)
    if (tls_plain_set[i] && tls_plain[i] == stream) {
      tls_plain_set[i] = false;
      return true;
    }
  return false;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    cached[dev] = v;
  }
  return cached[dev];
}

// ---- dense dispatch
// one <= 128 x 128 block of the weight operand; B (with leading dimension ldb) already points at the block
static int gemm_rowpanel_block(const float* A, int64_t lda, const float* B, int b_transposed, int64_t ldb, const float* bias, float* C,
                               int64_t ldc, int64_t m, int n, int k, const int32_t* rowscale_rowptr, const float* rowscale_inv,
                               int rowscale_group, int accumulate, int impl, void* ws, size_t ws_bytes, cudaStream_t stream,
                               const void* ready_image) {
  const bool tc_ok = tc_rowpanel_supported(lda, ldc, n, k, A, C) &&
                     (ready_image != nullptr || (ws != nullptr && ws_bytes >= tc_workspace_bytes()));
  if (impl == 2 && !tc_ok) {
    set_error("cgcn_gemm_rowpanel: tcgen05 path needs 16-byte aligned rows of a multiple of 4 floats and a workspace");
    return CGCN_ERR_INVALID;
  }
  if (impl == 2 || (impl == 0 && tc_ok))
    return gemm_rowpanel_tc(A, lda, B, b_transposed, bias, C, ldc, m, n, k, rowscale_rowptr, rowscale_inv, rowscale_group, ws, ws_bytes,
                            ready_image, stream, ldb, accumulate);
  return gemm_rowpanel_ffma(A, lda, B, b_transposed, bias, C, ldc, m, n, k, rowscale_rowptr, rowscale_inv, rowscale_group, stream, ldb,
                            accumulate);
}

// C[m x n] = rowscale * (A[m x k] op(B)) + bias for any n, k: the weight operand is cut into <= 128 x 128 blocks
// (d_model 256 / 512: BASELINE.json's stress configuration); the k-blocks of one column block accumulate into C
// (bias with the first one; the row scale distributes over the sum).
int gemm_rowpanel_dispatch(const float* A, int64_t lda, const float* B, int b_transposed, const float* bias, float* C,
                           int64_t ldc, int64_t m, int n, int k, const int32_t* rowscale_rowptr, const float* rowscale_inv, int rowscale_group,
                           int impl, void* ws, size_t ws_bytes, cudaStream_t stream, const void* ready_image = nullptr) {
  CGCN_REQUIRE(n >= 1 && k >= 1, "cgcn_gemm_rowpanel: n=%d k=%d", n, k);
  if (n <= 128 && k <= 128)
    return gemm_rowpanel_block(A, lda, B, b_transposed, b_transposed ? k : n, bias, C, ldc, m, n, k, rowscale_rowptr, rowscale_inv,
                               rowscale_group, 0, impl, ws, ws_bytes, stream, ready_image);
  const int64_t ldb = b_transposed ? k : n;
  for (int n0 = 0; n0 < n; n0 += 128) {
    const int nn = (n - n0) < 128 ? (n - n0) : 128;
    for (int k0 = 0; k0 < k; k0 += 128) {
      const int kk = (k - k0) < 128 ? (k - k0) : 128;
      const float* Bblk = b_transposed ? B + static_cast<int64_t>(n0) * ldb + k0 : B + static_cast<int64_t>(k0) * ldb + n0;
      CGCN_TRY(gemm_rowpanel_block(A + k0, lda, Bblk, b_transposed, ldb, (k0 == 0 && bias != nullptr) ? bias + n0 : nullptr, C + n0,
                                   ldc, m, nn, kk, rowscale_rowptr, rowscale_inv, rowscale_group, k0 > 0 ? 1 : 0, impl, ws, ws_bytes,
                                   stream, nullptr));
    }
  }
  return CGCN_OK;
}

static int gemm_gram_block(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t m,
                           int ka, int nb, int accumulate, int impl, void* ws, size_t ws_bytes, cudaStream_t stream) {
  const bool tc_ok = tc_gram_supported(lda, ldb, ka, nb, A, B);
  if (impl == 2 && !tc_ok) {
    set_error("cgcn_gemm_gram: tcgen05 path needs 16-byte aligned rows of a multiple of 4 floats");
    return CGCN_ERR_INVALID;
  }
  if (impl == 2 || (impl == 0 && tc_ok))
    return gemm_gram_tc(A, lda, B, ldb, C, ldc, m, ka, nb, accumulate, ws, ws_bytes, stream);
  return gemm_gram_ffma(A, lda, B, ldb, C, ldc, m, ka, nb, accumulate, ws, ws_bytes, stream);
}

// C[ka x nb] (+)= A^T B for any ka, nb: one <= 128 x 128 output block per launch pair (the reduction runs over all m rows
// inside a launch, so blocks never accumulate into each other).
int gemm_gram_dispatch(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t m,
                       int ka, int nb, int accumulate, int impl, void* ws, size_t ws_bytes, cudaStream_t stream) {
  CGCN_REQUIRE(ka >= 1 && nb >= 1, "cgcn_gemm_gram: ka=%d nb=%d", ka, nb);
  for (int a0 = 0; a0 < ka; a0 += 128)
    for (int b0 = 0; b0 < nb; b0 += 128)
      CGCN_TRY(gemm_gram_block(A + a0, lda, B + b0, ldb, C + static_cast<int64_t>(a0) * ldc + b0, ldc, m,
                               (ka - a0) < 128 ? (ka - a0) : 128, (nb - b0) < 128 ? (nb - b0) : 128, accumulate, impl, ws, ws_bytes,
                               stream));
  return CGCN_OK;
}

// ---- side stream: weight-gradient contractions and gradient finalizes are off the critical path of the
// backward pass (nothing downstream reads them before the optimiser step), so they run on a helper stream
// forked from / joined to the caller's stream with events.  One helper per host thread and device, created on
// first use (the only resources this library ever creates).
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t join = nullptr;
};
static int side_stream(SideStream** out) {
  static thread_local SideStream table[64];
  int dev = 0;
  CGCN_CUDA(cudaGetDevice(&dev));
  CGCN_REQUIRE(dev >= 0 && dev < 64, "device index %d out of range", dev);
  SideStream& s = table[dev];
  if (s.stream == nullptr) {
    CGCN_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    for (int i = 0; i < 4; ++i) CGCN_CUDA(cudaEventCreateWithFlags(&s.fork[i], cudaEventDisableTiming));
    CGCN_CUDA(cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming));
  }
  *out = &s;
  return CGCN_OK;
}

// ---- workspace layout (offsets in floats)
constexpr int ML = CGCN_MAX_LAYERS;
struct WsLayout {
  size_t ax[ML], z[ML], xo[ML], hb;
  size_t bn_mean, bn_rstd, bn_c1, bn_c2;
  size_t dy[ML], dX, dY, dC;           // backward: one dy panel per layer (the side stream reads it until the join) + 3 rotating
  size_t partial, partial_floats;      // main-stream reductions (BatchNorm)
  size_t partial_l[ML], partial_side;  // per-layer gate-backward partials and the side stream's own (column sums)
  size_t gram, gram_bytes;
  size_t tc, tc_bytes;                 // one tcgen05 weight image (hi/lo TF32, swizzled): 128 KB
  size_t img_fwd[ML + 1];              // GC_l.weight (l < L), out.weight^T          -- prepared once per forward
  size_t img_bwd[ML + 1];              // out.weight, GC_l.weight^T                  -- prepared once per backward
  size_t total_floats;
};

static WsLayout make_layout(int n, int d, int nclass, int layers, int strands) {
  (void)nclass;
  WsLayout L{};
  size_t off = 0;
  auto take = [&](size_t floats) {
    off = (off + 63) / 64 * 64;      // 256-byte alignment
    const size_t r = off;
    off += floats;
    return r;
  };
  const size_t panel = static_cast<size_t>(n) * strands * d;
  for (int l = 0; l < ML; ++l) {
    const bool used = l < layers;
    L.ax[l] = take(used ? panel : 0);
    L.z[l] = take(used ? panel : 0);
    L.xo[l] = take(used ? panel : 0);
  }
  L.hb = take(panel);
  L.bn_mean = take(static_cast<size_t>(strands) * d);
  L.bn_rstd = take(static_cast<size_t>(strands) * d);
  L.bn_c1 = take(static_cast<size_t>(strands) * d);
  L.bn_c2 = take(static_cast<size_t>(strands) * d);
  for (int l = 0; l < ML; ++l) L.dy[l] = take(l < layers ? panel : 0);
  L.dX = take(panel);
  L.dY = take(panel);
  L.dC = take(panel);
  size_t per = static_cast<size_t>(2) * strands * d;
  if (per < static_cast<size_t>(2 * d + 4)) per = 2 * d + 4;
  if (per < 128) per = 128;
  L.partial_floats = static_cast<size_t>(rowwise_max_grid()) * per;
  L.partial = take(L.partial_floats);
  for (int l = 0; l < ML; ++l) L.partial_l[l] = take(l < layers ? L.partial_floats : 0);
  L.partial_side = take(L.partial_floats);
  L.gram_bytes = gram_workspace_bytes(static_cast<int64_t>(n) * strands);
  L.gram = take((L.gram_bytes + 3) / 4);
  L.tc_bytes = tc_workspace_bytes();
  L.tc = take((L.tc_bytes + 3) / 4);
  for (int i = 0; i <= ML; ++i) {
    const bool used = i <= layers;
    L.img_fwd[i] = take(used ? (L.tc_bytes + 3) / 4 : 0);
    L.img_bwd[i] = take(used ? (L.tc_bytes + 3) / 4 : 0);
  }
  L.total_floats = (off + 63) / 64 * 64;
  return L;
}

static int validate(const cgcn_model* m, bool backward) {
  CGCN_REQUIRE(m != nullptr, "cgcn_model: null");
  CGCN_REQUIRE(m->graph.n >= 1 && m->graph.rowptr && m->graph.colidx, "cgcn_model: bad graph");
  CGCN_REQUIRE((m->graph.vals == nullptr) == (m->graph.row_inv == nullptr), "cgcn_model: weighted graphs need vals and row_inv");
  CGCN_REQUIRE(m->d == 128 || m->d == 256 || m->d == 512, "cgcn_model: d=%d (supported: 128 -- the width main.py:62 fixes -- 256, 512)", m->d);
  CGCN_REQUIRE(m->nclass >= 1 && m->nclass <= 128, "cgcn_model: nclass=%d must be in [1,128]", m->nclass);
  CGCN_REQUIRE(m->layers >= 1 && m->layers <= ML, "cgcn_model: layers=%d (1..%d)", m->layers, ML);
  CGCN_REQUIRE(m->gate_off == 0 || m->gate_off == 1, "cgcn_model: gate_off=%d", m->gate_off);
  CGCN_REQUIRE(m->strands == 1 || m->strands == 2, "cgcn_model: strands=%d", m->strands);
  CGCN_REQUIRE(m->dropout_p >= 0.f && m->dropout_p < 1.f, "cgcn_model: dropout_p=%f", m->dropout_p);
  CGCN_REQUIRE(m->out_ld == 0 || m->out_ld >= m->nclass, "cgcn_model: out_ld=%d < nclass=%d", m->out_ld, m->nclass);
  CGCN_REQUIRE(m->x_in && m->out, "cgcn_model: null activation pointer");
  for (int l = 0; l < m->layers; ++l) CGCN_REQUIRE(m->gate[l] != nullptr, "cgcn_model: null gate[%d]", l);
  CGCN_REQUIRE(m->bn_running_mean && m->bn_running_var, "cgcn_model: null BatchNorm running statistics");
  for (int l = 0; l < m->layers; ++l)
    CGCN_REQUIRE(m->params.gc_w[l] && m->params.gc_b[l] && m->params.gate_w[l] && m->params.gate_b[l],
                 "cgcn_model: null layer-%d parameter", l);
  CGCN_REQUIRE(m->params.bn_w && m->params.bn_b && m->params.out_w && m->params.out_b, "cgcn_model: null head parameter");
  CGCN_REQUIRE(!(m->training && (m->n_total > 0 ? m->n_total : m->graph.n) < 2),
               "cgcn_model: BatchNorm1d in training mode needs more than 1 row");
  const size_t need = cgcn_model_workspace_bytes(m->graph.n, m->d, m->nclass, m->layers, m->strands);
  if (m->workspace == nullptr || m->workspace_bytes < need) {
    set_error("cgcn_model: workspace %zu < %zu bytes", m->workspace_bytes, need);
    return CGCN_ERR_WORKSPACE;
  }
  if (backward) {
    CGCN_REQUIRE(m->out_grad != nullptr, "cgcn_model_backward: null out_grad");
    for (int l = 0; l < m->layers; ++l)
      CGCN_REQUIRE(m->grads.gc_w[l] && m->grads.gc_b[l] && m->grads.gate_w[l] && m->grads.gate_b[l],
                   "cgcn_model_backward: null layer-%d gradient", l);
    CGCN_REQUIRE(m->grads.bn_w && m->grads.bn_b && m->grads.out_w && m->grads.out_b, "cgcn_model_backward: null head gradient");
    CGCN_REQUIRE(!m->need_input_grad || m->x_in_grad, "cgcn_model_backward: need_input_grad without x_in_grad");
  }
  return CGCN_OK;
}


int gate_fwd_launch(const GateFwdArgs& a, int d, int S, bool stats, int* grid_out, cudaStream_t stream);
int bn_apply_launch(const BnApplyArgs& a, cudaStream_t stream);
int bn_bwd_reduce_launch(const BnBwdReduceArgs& a, int d, int S, int* grid_out, cudaStream_t stream);
int gate_bwd_launch(const GateBwdArgs& a, int d, int S, bool head, int* grid_out, cudaStream_t stream);
int gate_bwd_finalize_launch(const float* partial, int grid, int d, float* db, float* dwg, float* dbg, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// The model as stages.  cgcn_model_forward / _backward run them back to back on one GPU.  For one graph
// row-partitioned over several GPUs (m->n_total > 0: graph.n local rows, global column indices) the host calls
// cgcn_model_phase() stage by stage and performs the exchange step in between: an all-gather of the panel the
// next SpMM gathers from (into m->x_full), or an all-reduce of the BatchNorm sums (m->bn_sums).
// ------------------------------------------------------------------------------------------------
struct Ctx {
  const cgcn_model* m;
  WsLayout lay;
  cudaStream_t st;
  int n, d, S, C, L, W;
  int ldo;                          // leading dimension of out / out_grad
  int64_t M, n_total;
  bool dist;
  bool images;                      // tcgen05 weight images prepared once per pass
  bool fused;                       // fused layer kernels instead of SpMM + contraction + gate kernel
  float* ws;
  void* tcws;
  unsigned long long drop_off;      // float4 offset of the first local row in the global panel
};

// The fused layer kernels (fused_layer.cu): one launch per layer and direction instead of SpMM + contraction + gate
// kernel.  In this mode the saved `ax` panels hold the UN-normalised neighbour sums and the `dy` panels hold
// D^-1 dy, so that d W = ax^T dy is unchanged while the backward gather needs no per-neighbour scale.  A fused forward
// is always followed by the fused backward.  Measured on B200, whole genome (mean degree 10.7), ms per pass: three
// kernels 16.9, fused 15.7 (profiles/r02_layer_modes.md).  The all-in-one kernel keeps ~200 gather loads in flight per
// SM against the SpMM's ~320, so once the gather dominates (mean degree 51: fused 6.5 ms per layer vs SpMM 2.15 + 0.6 +
// 0.9) the three kernels win: graphs with more than FUSED_MAX_DEGREE stored entries per row on average use them.
constexpr int64_t FUSED_MAX_DEGREE = 24;
static bool use_fused(const cgcn_model* m, bool images) {
  static const bool off = getenv("CGCN_NO_FUSED") != nullptr;       // developer aid / A-B measurements
  if (off || !images || !fused_layer_supported(m->d, &m->graph)) return false;
  const int64_t nnz = m->graph.nnz, n = m->graph.n > 0 ? m->graph.n : 1;
  return nnz <= FUSED_MAX_DEGREE * n;
}

static Ctx make_ctx(const cgcn_model* m) {
  Ctx c;
  c.m = m;
  c.st = static_cast<cudaStream_t>(m->stream);
  c.n = m->graph.n; c.d = m->d; c.S = m->strands; c.C = m->nclass; c.L = m->layers;
  c.W = c.S * c.d;
  c.ldo = m->out_ld > 0 ? m->out_ld : c.C;
  c.M = static_cast<int64_t>(c.n) * c.S;
  c.dist = m->n_total > 0;
  c.n_total = c.dist ? m->n_total : c.n;
  c.lay = make_layout(c.n, c.d, c.C, c.L, c.S);
  c.ws = m->workspace;
  c.tcws = c.ws + c.lay.tc;
  c.drop_off = c.dist ? static_cast<unsigned long long>(m->row_begin) * c.W / 4 : 0ull;
  // Weight images of the tcgen05 contractions, one launch per pass (the weights change only at the optimiser step).
  // Wider models prepare each 128 x 128 weight block in place.
  c.images = m->gemm_impl != 1 && c.d == 128;
  c.fused = use_fused(m, c.images);
  return c;
}

// dropout site ids (cgcn_dropout_mask): 0 = after layer 1, 1 = after BatchNorm, l + 1 = after layer l + 1 (l >= 1)
static int layer_drop_site(int l) { return l == 0 ? 0 : l + 1; }

static const void* fwd_image(const Ctx& c, int i) { return c.images ? c.ws + c.lay.img_fwd[i] : nullptr; }
static const void* bwd_image(const Ctx& c, int i) { return c.images ? c.ws + c.lay.img_bwd[i] : nullptr; }

static int prep_fwd_images(const Ctx& c) {
  pdl_plain_next(c.st);              // first kernel of a pass: ordinary stream order against whatever ran before
  if (!c.images) return CGCN_OK;
  TcImageSpec sp[ML + 1];
  int k = 0;
  for (int l = 0; l < c.L; ++l) sp[k++] = TcImageSpec{c.m->params.gc_w[l], 0, c.d, c.d, c.ws + c.lay.img_fwd[l]};
  sp[k++] = TcImageSpec{c.m->params.out_w, 1, c.C, c.d, c.ws + c.lay.img_fwd[c.L]};
  return tc_prep_images(sp, k, c.st);
}
static int prep_bwd_images(const Ctx& c) {
  if (!c.images) return CGCN_OK;
  TcImageSpec sp[ML + 1];
  int k = 0;
  sp[k++] = TcImageSpec{c.m->params.out_w, 0, c.d, c.C, c.ws + c.lay.img_bwd[0]};
  for (int l = c.m->need_input_grad ? 0 : 1; l < c.L; ++l)
    sp[k++] = TcImageSpec{c.m->params.gc_w[l], 1, c.d, c.d, c.ws + c.lay.img_bwd[1 + l]};
  return tc_prep_images(sp, k, c.st);
}

// BatchNorm statistics from the last layer's per-CTA column sums (`parts` partial rows in lay.partial)
static int fwd_layer_stats(const Ctx& c, bool last, int parts) {
  const cgcn_model* m = c.m;
  const WsLayout& lay = c.lay;
  float* ws = c.ws;
  if (!last) return CGCN_OK;
  if (c.dist && m->training)         // publish this rank's column sums; the host all-reduces m->bn_sums
    return bn_finalize_launch(ws + lay.partial, parts, c.n_total, c.S, c.d, m->bn_eps, m->bn_momentum, 1, m->bn_running_mean,
                              m->bn_running_var, nullptr, ws + lay.bn_mean, ws + lay.bn_rstd, nullptr, m->bn_sums, c.st);
  if (!c.dist)
    return bn_finalize_launch(ws + lay.partial, parts, c.n, c.S, c.d, m->bn_eps, m->bn_momentum, m->training,
                              m->bn_running_mean, m->bn_running_var, m->bn_num_batches_tracked, ws + lay.bn_mean,
                              ws + lay.bn_rstd, nullptr, nullptr, c.st);
  return CGCN_OK;
}

// layer l: ax = A_hat x ; y = ax W + b ; gate.  `gather_src` is the panel the SpMM reads neighbours from (the
// layer input itself on one GPU, the all-gathered copy of it when row-partitioned).
static int fwd_layer(const Ctx& c, int l, const float* gather_src) {
  const cgcn_model* m = c.m;
  const WsLayout& lay = c.lay;
  float* ws = c.ws;
  const float* xin = (l == 0) ? m->x_in : ws + lay.xo[l - 1];
  const bool last = (l == c.L - 1);
  int grid = 0;
  if (c.fused) {
    // gather -> (A_hat x) W + b -> tanh -> gate -> blend -> dropout (-> BatchNorm column sums) in one kernel
    fl::Args a{};
    a.rowptr = m->graph.rowptr;
    a.colidx = m->graph.colidx;
    a.n = c.n;
    a.gsrc = gather_src;
    if (c.dist && m->peer != nullptr) CGCN_TRY(peer_table(&a.peer, m->peer, c.n, "fused layer"));  // neighbour rows over NVLink
    a.w = m->params.gc_w[l];
    a.w_transposed = 0;
    a.xin = xin;
    a.bias = m->params.gc_b[l];
    a.wg = m->params.gate_w[l];
    a.bg = m->params.gate_b[l];
    a.sx = ws + lay.ax[l];
    a.z = ws + lay.z[l];
    a.xo = ws + lay.xo[l];
    a.g = m->gate[l];
    a.partial = ws + lay.partial;
    a.gate_off = m->gate_off;
    a.drop = make_dropout(m->dropout_p, m->seed, m->step, layer_drop_site(l), m->training && !last, c.drop_off);
    CGCN_TRY(fused_layer_launch(a, c.S, (last && m->training) ? fl::FWD_STATS : fl::FWD, &grid, c.st));
    return fwd_layer_stats(c, last, grid);
  }
  // ax = A_hat x                                   (torch.spmm, models/SubLayers.py:46)
  if (c.dist && m->peer != nullptr)  // neighbour rows straight from the owners' exchange buffers (NVLink loads)
    CGCN_TRY(spmm_peer_launch(&m->graph, m->peer, ws + lay.ax[l], c.W, 1, nullptr, c.st));
  else
    CGCN_TRY(spmm_launch(&m->graph, gather_src, ws + lay.ax[l], c.W, 1, nullptr, c.st));
  // y = ax W + b                                   (torch.mm + bias, models/SubLayers.py:43,50)
  CGCN_TRY(gemm_rowpanel_dispatch(ws + lay.ax[l], c.d, m->params.gc_w[l], 0, m->params.gc_b[l], ws + lay.z[l], c.d, c.M, c.d,
                                  c.d, nullptr, nullptr, 1, m->gemm_impl, c.tcws, lay.tc_bytes, c.st, fwd_image(c, l)));
  // z = tanh(y); g = sigmoid(W z); x' = (1-g) x + g z; dropout between the layers
  //                                                (models/ChromeModels.py:38-42 / 44-46)
  GateFwdArgs a{};
  a.y = ws + lay.z[l];
  a.x = xin;
  a.wg = m->params.gate_w[l];
  a.bg = m->params.gate_b[l];
  a.z = ws + lay.z[l];
  a.g = m->gate[l];
  a.xo = ws + lay.xo[l];
  a.stats_partial = ws + lay.partial;
  a.n = c.n;
  a.gate_off = m->gate_off;
  a.drop = make_dropout(m->dropout_p, m->seed, m->step, layer_drop_site(l), m->training && !last, c.drop_off);
  CGCN_TRY(gate_fwd_launch(a, c.d, c.S, last && m->training, &grid, c.st));
  return fwd_layer_stats(c, last, grid);
}

static int fwd_head(const Ctx& c) {
  const cgcn_model* m = c.m;
  const WsLayout& lay = c.lay;
  float* ws = c.ws;
  if (c.dist)                        // statistics from the all-reduced sums (or the running stats in eval mode)
    CGCN_TRY(bn_finalize_launch(ws + lay.partial, 0, c.n_total, c.S, c.d, m->bn_eps, m->bn_momentum, m->training,
                                m->bn_running_mean, m->bn_running_var, m->bn_num_batches_tracked, ws + lay.bn_mean,
                                ws + lay.bn_rstd, m->training ? m->bn_sums : nullptr, nullptr, c.st));
  // hb = dropout(BatchNorm(relu(x)))                 (models/ChromeModels.py:48-50)
  BnApplyArgs b{};
  b.h = ws + lay.xo[c.L - 1];
  b.mean = ws + lay.bn_mean;
  b.rstd = ws + lay.bn_rstd;
  b.gamma = m->params.bn_w;
  b.beta = m->params.bn_b;
  b.hb = ws + lay.hb;
  b.total4 = static_cast<int64_t>(c.n) * c.W / 4;
  b.S = c.S;
  b.D = c.d;
  b.drop = make_dropout(m->dropout_p, m->seed, m->step, 1, m->training, c.drop_off);
  CGCN_TRY(bn_apply_launch(b, c.st));
  // out = hb Wout^T + bout                           (models/ChromeModels.py:51)
  return gemm_rowpanel_dispatch(ws + lay.hb, c.d, m->params.out_w, 1, m->params.out_b, m->out, c.ldo, c.M, c.C, c.d, nullptr, nullptr,
                                1, m->gemm_impl, c.tcws, lay.tc_bytes, c.st, fwd_image(c, c.L));
}

static int model_forward(const cgcn_model* m) {
  CGCN_TRY(validate(m, false));
  CGCN_REQUIRE(m->n_total <= 0, "cgcn_model_forward: row-partitioned graphs (n_total > 0) run through cgcn_model_phase");
  const Ctx c = make_ctx(m);
  CGCN_TRY(prep_fwd_images(c));
  for (int l = 0; l < c.L; ++l) CGCN_TRY(fwd_layer(c, l, (l == 0) ? m->x_in : c.ws + c.lay.xo[l - 1]));
  return fwd_head(c);
}

// ---- backward stages.  Scratch panels: one dy per layer (never rewritten while the side stream's gram kernel reads
// it) and three rotating ones.  On the three-kernel path layer l reads the gradient entering its gate stage from
// src(l), writes dy_l and dxd (dC), overwrites src(l) with t_l = D^-1 (dy_l W_l^T), and the SpMM writes
// dx = dC + P t_l into the other rotating panel, which is src(l-1).
struct Fork {
  SideStream* side;
  cudaStream_t st, ss;
  bool serial;
  int id = 0;
  int fork() {                       // side stream waits for everything enqueued on `st` so far
    if (serial) return CGCN_OK;
    CGCN_CUDA(cudaEventRecord(side->fork[id], st));
    CGCN_CUDA(cudaStreamWaitEvent(ss, side->fork[id], 0));
    pdl_plain_next(ss);              // the next side-stream kernel depends on an event, not on its stream predecessor
    id = (id + 1) & 3;
    return CGCN_OK;
  }
  int join() {                       // the caller's stream owns every gradient again
    if (serial) return CGCN_OK;
    CGCN_CUDA(cudaEventRecord(side->join, ss));
    CGCN_CUDA(cudaStreamWaitEvent(st, side->join, 0));
    pdl_plain_next(st);
    return CGCN_OK;
  }
};

// serial: the side-stream work runs in order on the caller's stream
static int make_fork(const Ctx& c, bool serial, Fork* f) {
  static const bool no_side = getenv("CGCN_NO_SIDE_STREAM") != nullptr;   // developer aid
  f->serial = serial || no_side;
  f->st = c.st;
  f->side = nullptr;
  f->ss = c.st;
  if (!f->serial) {
    CGCN_TRY(side_stream(&f->side));
    f->ss = f->side->stream;
  }
  return CGCN_OK;
}

static float* bwd_src(const Ctx& c, int l) { return c.ws + ((((c.L - 1 - l) & 1) == 0) ? c.lay.dX : c.lay.dY); }
static float* bwd_other(const Ctx& c, int l) { return c.ws + ((((c.L - 1 - l) & 1) == 0) ? c.lay.dY : c.lay.dX); }

// head: side: d out.weight = dout^T hb ; d out.bias = colsum(dout).  main: d hb = dout Wout ; BatchNorm backward sums
static int bwd_head(const Ctx& c, Fork& f) {
  const cgcn_model* m = c.m;
  const WsLayout& lay = c.lay;
  float* ws = c.ws;
  float* dhb = bwd_src(c, c.L - 1);
  void* gram_ws = ws + lay.gram;               // used by the side stream only
  CGCN_TRY(prep_bwd_images(c));
  CGCN_TRY(f.fork());
  CGCN_TRY(gemm_gram_dispatch(m->out_grad, c.ldo, ws + lay.hb, c.d, m->grads.out_w, c.d, c.M, c.C, c.d, 0, m->gemm_impl, gram_ws,
                              lay.gram_bytes, f.ss));
  CGCN_TRY(colsum_launch(m->out_grad, c.M, c.C, c.ldo, m->grads.out_b, ws + lay.partial_side, f.ss));
  CGCN_TRY(gemm_rowpanel_dispatch(m->out_grad, c.ldo, m->params.out_w, 0, nullptr, dhb, c.d, c.M, c.d, c.C, nullptr, nullptr, 1,
                                  m->gemm_impl, c.tcws, lay.tc_bytes, c.st, bwd_image(c, 0)));
  BnBwdReduceArgs r{};
  r.dhb = dhb;
  r.h = ws + lay.xo[c.L - 1];
  r.mean = ws + lay.bn_mean;
  r.rstd = ws + lay.bn_rstd;
  r.partial = ws + lay.partial;
  r.n = c.n;
  r.drop = make_dropout(m->dropout_p, m->seed, m->step, 1, m->training, c.drop_off);
  int grid = 0;
  CGCN_TRY(bn_bwd_reduce_launch(r, c.d, c.S, &grid, c.st));
  // one GPU: c1, c2, d gamma, d beta.  Row-partitioned: local d gamma / d beta + this rank's sums into m->bn_sums
  return bn_bwd_finalize_launch(ws + lay.partial, grid, c.n_total, c.S, c.d, m->training, ws + lay.bn_c1, ws + lay.bn_c2,
                                m->grads.bn_w, m->grads.bn_b, nullptr, c.dist ? m->bn_sums : nullptr, c.st);
}

// Gradient entering layer l_from - 1 (or x_in_grad) from layer l_from; `gather` is the panel the next propagate reads
// (bwd_layer's *t_out, or its all-gathered copy).
// Three kernels: dx = dxd + P t, with t = D^-1 (dy W^T), into the other rotating panel.
// Fused: the gather comes first, A_hat^T G W^T = (P (D^-1 G)) W^T.  One kernel gathers u = P dys_{l_from}, contracts
// u W^T, adds (1-g) dh (dC) and, for l_from > 0, runs the whole gate / tanh backward of layer l_from - 1 in its epilogue
// (writes dys_{l_from-1}, dC, the column partials; *parts = partial rows written).  l_from == 0: d loss / d x_in.
// `parts` may be NULL.
static int bwd_propagate(const Ctx& c, int l_from, const float* gather, int* parts) {
  const cgcn_model* m = c.m;
  const WsLayout& lay = c.lay;
  float* ws = c.ws;
  if (!c.fused) {
    float* dx = (l_from == 0) ? m->x_in_grad : bwd_other(c, l_from);
    if (c.dist && m->peer != nullptr) return spmm_peer_launch(&m->graph, m->peer, dx, c.W, 0, ws + lay.dC, c.st);
    return spmm_launch(&m->graph, gather, dx, c.W, 0, ws + lay.dC, c.st);
  }
  fl::Args a{};
  a.rowptr = m->graph.rowptr;
  a.colidx = m->graph.colidx;
  a.n = c.n;
  a.gsrc = gather;
  if (c.dist && m->peer != nullptr) CGCN_TRY(peer_table(&a.peer, m->peer, c.n, "fused layer"));
  a.w = m->params.gc_w[l_from];
  a.w_transposed = 1;
  a.dxd_in = ws + lay.dC;
  a.gate_off = m->gate_off;
  if (l_from == 0) {
    a.dx_out = m->x_in_grad;
    a.drop = make_dropout(0.f, 0, 0, 0, false, 0);
    return fused_layer_launch(a, c.S, fl::BWD_INPUT, parts, c.st);
  }
  const int lp = l_from - 1;
  a.wg = m->params.gate_w[lp];
  a.z_prev = ws + lay.z[lp];
  a.x_prev = (lp == 0) ? m->x_in : ws + lay.xo[lp - 1];
  a.g_prev = m->gate[lp];
  a.dys_out = ws + lay.dy[lp];
  a.dxd_out = (lp > 0 || m->need_input_grad) ? ws + lay.dC : nullptr;
  a.partial = ws + lay.partial_l[lp];
  a.drop = make_dropout(m->dropout_p, m->seed, m->step, layer_drop_site(lp), m->training, c.drop_off);
  return fused_layer_launch(a, c.S, fl::BWD_MID, parts, c.st);
}

// Gate stage of layer l, its weight gradients (side stream) and the panel the next propagate gathers.
// The gate stage is a row-wise kernel for the head layer and on the three-kernel path; in fused mode it stores
// D^-1 dy, and the gate stage of every other layer already ran in the epilogue of bwd_propagate(l + 1) (`parts`
// partial rows).  *t_out = dy in fused mode, else t = D^-1 (dy W^T) in the panel that held src(l); NULL if the chain
// stops here.
static int bwd_layer(const Ctx& c, Fork& f, int l, int parts, const float** t_out) {
  const cgcn_model* m = c.m;
  const WsLayout& lay = c.lay;
  float* ws = c.ws;
  const bool head = (l == c.L - 1);
  const bool need_dx = (l > 0) || m->need_input_grad;
  float* src = bwd_src(c, l);
  float* dy = ws + lay.dy[l];
  *t_out = nullptr;
  if (head && c.dist)                // c1, c2 from the all-reduced BatchNorm backward sums
    CGCN_TRY(bn_bwd_finalize_launch(ws + lay.partial, 0, c.n_total, c.S, c.d, m->training, ws + lay.bn_c1, ws + lay.bn_c2, nullptr,
                                    nullptr, m->bn_sums, nullptr, c.st));
  if (head || !c.fused) {
    GateBwdArgs a{};
    a.dsrc = src;
    a.h = ws + lay.xo[l];
    a.mean = ws + lay.bn_mean;
    a.rstd = ws + lay.bn_rstd;
    a.gamma = m->params.bn_w;
    a.c1 = ws + lay.bn_c1;
    a.c2 = ws + lay.bn_c2;
    a.z = ws + lay.z[l];
    a.x = (l == 0) ? m->x_in : ws + lay.xo[l - 1];
    a.g = m->gate[l];
    a.wg = m->params.gate_w[l];
    a.dy = dy;
    a.dxd = need_dx ? ws + lay.dC : nullptr;
    a.partial = ws + lay.partial_l[l];
    a.n = c.n;
    a.drop = make_dropout(m->dropout_p, m->seed, m->step, head ? 1 : layer_drop_site(l), m->training, c.drop_off);
    a.scale_rowptr = c.fused ? m->graph.rowptr : nullptr;
    CGCN_TRY(gate_bwd_launch(a, c.d, c.S, head, &parts, c.st));
  }
  // side: bias / gate gradients from the partials, d W = (A_hat x)^T dy
  CGCN_TRY(f.fork());
  CGCN_TRY(gate_bwd_finalize_launch(ws + lay.partial_l[l], parts, c.d, m->grads.gc_b[l], m->grads.gate_w[l], m->grads.gate_b[l], f.ss));
  CGCN_TRY(gemm_gram_dispatch(ws + lay.ax[l], c.d, dy, c.d, m->grads.gc_w[l], c.d, c.M, c.d, c.d, 0, m->gemm_impl, ws + lay.gram,
                              lay.gram_bytes, f.ss));
  if (!need_dx) return CGCN_OK;
  if (c.fused) {
    *t_out = dy;
    return CGCN_OK;
  }
  // main: t = D^-1 (dy W^T) -> the panel that held `src`
  CGCN_TRY(gemm_rowpanel_dispatch(dy, c.d, m->params.gc_w[l], 1, nullptr, src, c.d, c.M, c.d, c.d, m->graph.rowptr,
                                  m->graph.row_inv, c.S, m->gemm_impl, c.tcws, lay.tc_bytes, c.st, bwd_image(c, 1 + l)));
  *t_out = src;
  return CGCN_OK;
}

static int model_backward(const cgcn_model* m) {
  CGCN_TRY(validate(m, true));
  CGCN_REQUIRE(m->n_total <= 0, "cgcn_model_backward: row-partitioned graphs (n_total > 0) run through cgcn_model_phase");
  const Ctx c = make_ctx(m);
  Fork f;
  CGCN_TRY(make_fork(c, false, &f));
  CGCN_TRY(bwd_head(c, f));
  int parts = 0;
  for (int l = c.L - 1; l >= 0; --l) {
    const float* t = nullptr;
    CGCN_TRY(bwd_layer(c, f, l, parts, &t));
    if (t == nullptr) break;
    CGCN_TRY(bwd_propagate(c, l, t, &parts));
  }
  return f.join();
}

// One stage of the row-partitioned model.  *publish (may be NULL) receives the local panel the host must
// all-gather into m->x_full before the next stage, or NULL when the next stage needs no gather.
static int model_phase(const cgcn_model* m, int kind, int layer, const float** publish) {
  if (publish) *publish = nullptr;
  CGCN_TRY(validate(m, kind >= CGCN_PHASE_BWD_HEAD));
  CGCN_REQUIRE(m->n_total >= m->graph.n && (m->x_full != nullptr || m->peer != nullptr) && m->bn_sums != nullptr && m->row_begin >= 0,
               "cgcn_model_phase: needs n_total, row_begin, x_full (or peer) and bn_sums");
  CGCN_REQUIRE(layer >= 0 && layer < m->layers, "cgcn_model_phase: layer %d", layer);
  const Ctx c = make_ctx(m);
  Fork f;
  CGCN_TRY(make_fork(c, true, &f));  // stage by stage: everything on the caller's stream
  const float* t = nullptr;
  int parts = 0;
  switch (kind) {
    case CGCN_PHASE_FWD_LAYER:       // x_full holds the gathered input of `layer`
      if (layer == 0) CGCN_TRY(prep_fwd_images(c));
      CGCN_TRY(fwd_layer(c, layer, m->x_full));
      if (publish && layer + 1 < c.L) *publish = c.ws + c.lay.xo[layer];
      return CGCN_OK;
    case CGCN_PHASE_FWD_HEAD:        // bn_sums all-reduced
      return fwd_head(c);
    case CGCN_PHASE_BWD_HEAD:
      return bwd_head(c, f);
    case CGCN_PHASE_BWD_LAYER:       // layer == L-1: bn_sums all-reduced ; else: x_full holds the gathered t of layer+1
      if (layer < c.L - 1) CGCN_TRY(bwd_propagate(c, layer + 1, m->x_full, &parts));
      CGCN_TRY(bwd_layer(c, f, layer, parts, &t));
      if (publish) *publish = t;
      return CGCN_OK;
    case CGCN_PHASE_BWD_INPUT:       // x_full holds the gathered t of layer 0
      CGCN_REQUIRE(m->need_input_grad && m->x_in_grad, "cgcn_model_phase: BWD_INPUT without need_input_grad");
      return bwd_propagate(c, 0, m->x_full, nullptr);
    default:
      set_error("cgcn_model_phase: unknown phase %d", kind);
      return CGCN_ERR_INVALID;
  }
}

}  // namespace cgcn

using namespace cgcn;

extern "C" int cgcn_abi_version(void) { return CGCN_ABI_VERSION; }
extern "C" const char* cgcn_last_error(void) { return tls_error; }
extern "C" int64_t cgcn_launch_count(void) { return g_launches.load(); }

extern "C" int cgcn_device_info(int32_t* sm, int32_t* major, int32_t* minor) {
  int dev = 0;
  CGCN_CUDA(cudaGetDevice(&dev));
  int a = 0, b = 0, c = 0;
  CGCN_CUDA(cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev));
  CGCN_CUDA(cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMajor, dev));
  CGCN_CUDA(cudaDeviceGetAttribute(&c, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm) *sm = a;
  if (major) *major = b;
  if (minor) *minor = c;
  return CGCN_OK;
}

extern "C" size_t cgcn_sizeof(int32_t which) {
  switch (which) {
    case 0: return sizeof(cgcn_graph);
    case 1: return sizeof(cgcn_params);
    case 2: return sizeof(cgcn_model);
    case 3: return sizeof(cgcn_peer_panel);
    default: return 0;
  }
}

extern "C" size_t cgcn_model_workspace_bytes(int32_t n, int32_t d, int32_t nclass, int32_t layers, int32_t strands) {
  if (n < 1 || d < 1 || layers < 1 || layers > CGCN_MAX_LAYERS || strands < 1 || strands > 2) return 0;
  return make_layout(n, d, nclass, layers, strands).total_floats * sizeof(float);
}

extern "C" int cgcn_model_forward(const cgcn_model* m) { return model_forward(m); }
extern "C" int cgcn_model_phase(const cgcn_model* m, int32_t kind, int32_t layer, const float** publish) {
  return model_phase(m, kind, layer, publish);
}
extern "C" int cgcn_model_backward(const cgcn_model* m) { return model_backward(m); }

extern "C" int cgcn_gcn_layer_fwd(const cgcn_graph* g, int32_t strands, const float* x_gather, const float* x_in,
                                  const float* W, const float* b, const float* wg, const float* bg, int32_t gate_off,
                                  float dropout_p, uint64_t seed, uint64_t step, int32_t site, float* sx, float* z,
                                  float* x_out, float* gate, float* stats_partial, int32_t* parts_host, cgcn_stream_t stream) {
  CGCN_REQUIRE(g && x_gather && x_in && W && b && sx && z && x_out && gate, "cgcn_gcn_layer_fwd: null argument");
  CGCN_REQUIRE(gate_off || (wg && bg), "cgcn_gcn_layer_fwd: null gate parameters");
  CGCN_REQUIRE(fused_layer_supported(128, g), "cgcn_gcn_layer_fwd: pattern graphs only (no value array)");
  CGCN_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "cgcn_gcn_layer_fwd: dropout_p=%f", dropout_p);
  fl::Args a{};
  a.rowptr = g->rowptr;
  a.colidx = g->colidx;
  a.n = g->n;
  a.gsrc = x_gather;
  a.w = W;
  a.w_transposed = 0;
  a.xin = x_in;
  a.bias = b;
  a.wg = wg;
  a.bg = bg;
  a.sx = sx;
  a.z = z;
  a.xo = x_out;
  a.g = gate;
  a.partial = stats_partial;
  a.gate_off = gate_off;
  a.drop = make_dropout(dropout_p, seed, step, site, dropout_p > 0.f, 0);
  int parts = 0;
  pdl_plain_next(static_cast<cudaStream_t>(stream));
  CGCN_TRY(fused_layer_launch(a, strands, stats_partial ? fl::FWD_STATS : fl::FWD, &parts, static_cast<cudaStream_t>(stream)));
  if (parts_host) *parts_host = parts;
  return CGCN_OK;
}

extern "C" int cgcn_gcn_layer_bwd(const cgcn_graph* g, int32_t strands, const float* dys_gather, const float* dxd, const float* W,
                                  const float* z_prev, const float* x_prev, const float* g_prev, const float* wg_prev,
                                  int32_t gate_off, float dropout_p, uint64_t seed, uint64_t step, int32_t site_prev,
                                  float* dys_out, float* dxd_out, float* dx_out, float* partial, int32_t* parts_host,
                                  cgcn_stream_t stream) {
  CGCN_REQUIRE(g && dys_gather && dxd && W, "cgcn_gcn_layer_bwd: null argument");
  CGCN_REQUIRE(fused_layer_supported(128, g), "cgcn_gcn_layer_bwd: pattern graphs only (no value array)");
  CGCN_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "cgcn_gcn_layer_bwd: dropout_p=%f", dropout_p);
  fl::Args a{};
  a.rowptr = g->rowptr;
  a.colidx = g->colidx;
  a.n = g->n;
  a.gsrc = dys_gather;
  a.w = W;
  a.w_transposed = 1;
  a.dxd_in = dxd;
  a.gate_off = gate_off;
  int parts = 0;
  pdl_plain_next(static_cast<cudaStream_t>(stream));
  if (z_prev == nullptr) {
    CGCN_REQUIRE(dx_out != nullptr, "cgcn_gcn_layer_bwd: null dx_out");
    a.dx_out = dx_out;
    a.drop = make_dropout(0.f, 0, 0, 0, false, 0);
    CGCN_TRY(fused_layer_launch(a, strands, fl::BWD_INPUT, &parts, static_cast<cudaStream_t>(stream)));
  } else {
    CGCN_REQUIRE(x_prev && g_prev && (gate_off || wg_prev) && dys_out && partial, "cgcn_gcn_layer_bwd: null layer-below argument");
    CGCN_REQUIRE(dys_out != dys_gather, "cgcn_gcn_layer_bwd: dys_out must not alias the gathered panel");
    a.wg = wg_prev;
    a.z_prev = z_prev;
    a.x_prev = x_prev;
    a.g_prev = g_prev;
    a.dys_out = dys_out;
    a.dxd_out = dxd_out;
    a.partial = partial;
    a.drop = make_dropout(dropout_p, seed, step, site_prev, dropout_p > 0.f, 0);
    CGCN_TRY(fused_layer_launch(a, strands, fl::BWD_MID, &parts, static_cast<cudaStream_t>(stream)));
  }
  if (parts_host) *parts_host = parts;
  return CGCN_OK;
}

static int train_step(const cgcn_model* m, const float* target, const uint32_t* target_bits, float* probs, float* loss_sum_out,
                      float* out_grad_scratch) {
  CGCN_REQUIRE(m && (target || target_bits) && loss_sum_out && out_grad_scratch, "cgcn_train_step: null argument");
  CGCN_TRY(model_forward(m));
  const Ctx c = make_ctx(m);
  CGCN_TRY(bce_launch(m->out, target, target_bits, c.n, c.C, c.S, c.ldo, probs, loss_sum_out, out_grad_scratch, c.ws + c.lay.partial, 0,
                      c.st));
  cgcn_model mb = *m;
  mb.out_grad = out_grad_scratch;
  return model_backward(&mb);
}

extern "C" int cgcn_train_step(const cgcn_model* m, const float* target, float* probs, float* loss_sum_out,
                               float* out_grad_scratch) {
  return train_step(m, target, nullptr, probs, loss_sum_out, out_grad_scratch);
}

extern "C" int cgcn_train_step_bits(const cgcn_model* m, const uint32_t* target_bits, float* probs, float* loss_sum_out,
                                    float* out_grad_scratch) {
  return train_step(m, nullptr, target_bits, probs, loss_sum_out, out_grad_scratch);
}

extern "C" int cgcn_gemm_rowpanel(const float* A, int64_t lda, const float* B, int32_t b_transposed, const float* bias,
                                  float* C, int64_t ldc, int64_t m, int32_t n, int32_t k,
                                  const int32_t* rowscale_rowptr, const float* rowscale_inv, int32_t rowscale_group, int32_t gemm_impl,
                                  void* workspace, size_t workspace_bytes, cgcn_stream_t stream) {
  return gemm_rowpanel_dispatch(A, lda, B, b_transposed, bias, C, ldc, m, n, k, rowscale_rowptr, rowscale_inv, rowscale_group,
                                gemm_impl, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" size_t cgcn_gemm_gram_workspace_bytes(int64_t m) { return gram_workspace_bytes(m); }

extern "C" int cgcn_gemm_gram(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t m,
                              int32_t ka, int32_t nb, int32_t accumulate, int32_t gemm_impl, void* workspace,
                              size_t workspace_bytes, cgcn_stream_t stream) {
  return gemm_gram_dispatch(A, lda, B, ldb, C, ldc, m, ka, nb, accumulate, gemm_impl, workspace, workspace_bytes,
                            static_cast<cudaStream_t>(stream));
}
