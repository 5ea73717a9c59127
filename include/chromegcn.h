/*
 * chromegcn.h -- C ABI of libchromegcn.so: the B200 (sm_100a) implementation of the
 * ChromeGCN chromosome-model hot path.
 *
 * The reference (QData/ChromeGCN) is pure Python/PyTorch and has no FFI of its own; its
 * hot path is nn.Module code.  This header is therefore the boundary a maintainer binds
 * (ctypes stub in INTEGRATION.md) to put the CUDA path behind the reference's Python
 * surface.  Each entry point names the reference code it replaces (paths relative to the
 * reference repository).
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless its name ends in _host;
 *   - every call enqueues work on the caller's stream (a cudaStream_t passed as void*) and
 *     neither allocates nor synchronises, except cgcn_adj_build / cgcn_coo_to_pattern, whose
 *     output size is data dependent (they synchronise `stream` before returning);
 *   - return value: 0 = ok, negative = error (cgcn_status); cgcn_last_error() returns a
 *     thread-local message for the last failing call of the calling thread;
 *   - thread-safe for distinct streams / buffers; no global mutable state but that string and, per host
 *     thread and device, one helper stream + events created on the first cgcn_model_backward (weight-gradient
 *     contractions run there, forked from and joined back to the caller's stream with events);
 *   - there is NO CPU fallback: on a machine without an sm_100 device every compute call
 *     returns CGCN_ERR_CUDA.
 *
 * Feature panels are row-major fp32 `[n][strands][d]` ("strand-interleaved": the forward
 * and reverse-complement feature rows of one window sit next to each other, so one column
 * index of the graph fetches strands*d*4 contiguous bytes).  strands = 1 is the layout of a
 * plain `[n][d]` tensor.  The SpMM takes any row width that is a multiple of 128 floats up to
 * 1024; the model entry points take d = 128 (the reference fixes it, main.py:62).
 */
#ifndef CHROMEGCN_H_
#define CHROMEGCN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGCN_ABI_VERSION 8
#define CGCN_MAX_LAYERS 4
#define CGCN_MAX_PEERS 8    /* GPUs of one NVSwitch box */

typedef void* cgcn_stream_t; /* cudaStream_t */

typedef enum cgcn_status {
  CGCN_OK = 0,
  CGCN_ERR_INVALID = -1,   /* bad argument (null pointer, unsupported d, ...) */
  CGCN_ERR_CUDA = -2,      /* CUDA runtime error, no device, wrong architecture */
  CGCN_ERR_WORKSPACE = -3, /* workspace too small */
  CGCN_ERR_DATA = -4,      /* input data violates the contract (NaN contact value, norm index out of range, ...) */
  CGCN_ERR_CAPACITY = -5   /* output buffer too small */
} cgcn_status;

/* ---------------------------------------------------------------- library ---- */
int cgcn_abi_version(void);
const char* cgcn_last_error(void);
/* SM count and compute capability of the current device. */
int cgcn_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
/* sizeof() of the structs below as compiled, for binding self-checks: which = 0 cgcn_graph,
 * 1 cgcn_params, 2 cgcn_model, 3 cgcn_peer_panel. */
size_t cgcn_sizeof(int32_t which);
/* Number of kernels this library has launched from the calling process (all threads). */
int64_t cgcn_launch_count(void);

/* ------------------------------------------------- piece 1: adjacency build ---- */
/*
 * Text ingest (host code, no CUDA call): the Juicer files data/7create_graph_new.py reads line by line with
 * csv.DictReader.  cgcn_contacts_parse: `RAWobserved` dump, "bin1 \t bin2 \t value" per line (:71-76; further
 * columns ignored, blank lines skipped) -> three arrays in file order.  cgcn_vector_parse: `*norm` vector, one
 * float per line (:56-59; "NaN" parses to NaN -- the build kernel applies the NaN / 0 -> inf rule of :60-63).
 * The file is memory-mapped and parsed by `threads` host threads (0 = all cores) over line-aligned byte ranges;
 * numbers convert like Python's int() / float() on the same token (correctly rounded).  Size the arrays with
 * cgcn_text_count_rows (non-blank lines).  A malformed line is CGCN_ERR_DATA with the row in cgcn_last_error().
 */
int cgcn_text_count_rows(const char* path, int32_t threads, int64_t* rows_out);
int cgcn_contacts_parse(const char* path, int64_t capacity, int64_t* bin1, int64_t* bin2, double* val,
                        int64_t* rows_out, int32_t threads);
int cgcn_vector_parse(const char* path, int64_t capacity, double* out, int64_t* rows_out, int32_t threads);
/* Windows bed file of create_bin_dict (data/7create_graph_new.py:24-37): for every row whose first column is one of
 * `chroms` ('\n'-separated names) the index of that name and the row's start position, in file order.  With
 * capacity too small returns CGCN_ERR_CAPACITY and the number of matching rows in *rows_out. */
int cgcn_bed_starts_parse(const char* path, const char* chroms, int64_t capacity, int32_t* chrom_index, int64_t* start,
                          int64_t* rows_out, int32_t threads);

/*
 * Hi-C contact list -> symmetric binary window adjacency in CSR (no self loops).
 * Replaces data/7create_graph_new.py:67-120 (get_contact_edge_pairs, get_top_contact_locs,
 * create_adj_mat) bit-exactly:
 *   keep rows with bin1 != bin2 and both bins in `window_starts` (sorted, unique);
 *   use_norm: v = val / (nv[bin1 / res_bp] * nv[bin2 / res_bp]) in IEEE double, nv = norm with
 *   NaN and 0.0 replaced by +inf (:51-65);  !use_norm: only the first k_pairs accepted rows (:88-89);
 *   duplicate (bin1,bin2) keys: rank position = first occurrence, value = last occurrence (:86);
 *   stable descending sort by v, first k_pairs entries (all if k_pairs == 0) (:93-104);
 *   emit (i,j) and (j,i), collapse duplicates, CSR with ascending columns (:108-120).
 * rowptr has n+1 entries; colidx capacity colidx_cap entries (2*k_pairs always suffices when
 * k_pairs > 0).  *nnz_host (host pointer) receives the number of stored entries.
 * A NaN contact value or a bin beyond norm_len is CGCN_ERR_DATA (the reference's behaviour there
 * is a Python exception / an undefined sort order).
 */
int cgcn_adj_build_workspace_bytes(int64_t m, int64_t n, int64_t k_pairs, size_t* bytes_host);
int cgcn_adj_build(const int64_t* bin1, const int64_t* bin2, const double* val, int64_t m,
                   const int64_t* window_starts, int64_t n,
                   const double* norm, int64_t norm_len, int64_t res_bp,
                   int64_t k_pairs, int32_t use_norm,
                   int32_t* rowptr, int32_t* colidx, int64_t colidx_cap, int64_t* nnz_host,
                   void* workspace, size_t workspace_bytes, cgcn_stream_t stream);

/*
 * Pattern of bin(A + I): merges the diagonal into every (column-sorted) CSR row.
 * Replaces the structural half of process_graph('hic') (utils/util_methods.py:152-165); the
 * numeric half, D^-1, is never materialised: every kernel derives 1/deg_i from rowptr.
 * rowptr_out: n+1 entries; colidx_out: nnz + n entries (an existing diagonal entry is merged:
 * the unused tail is left untouched and rowptr_out[n] is the true count).
 */
int cgcn_adj_add_selfloops_workspace_bytes(int32_t n, size_t* bytes_host);
int cgcn_adj_add_selfloops(const int32_t* rowptr, const int32_t* colidx, int32_t n,
                           int32_t* rowptr_out, int32_t* colidx_out,
                           void* workspace, size_t workspace_bytes, cgcn_stream_t stream);

/*
 * torch sparse COO (int64 rows/cols, fp32 values, any order) -> CSR pattern, for callers that
 * hand ChromeGCN.forward the tensor the reference's process_graph returns
 * (utils/util_methods.py:120-135).  flags_host bit 0: every value equals 1/deg(row) (mean
 * aggregation: pattern-only fast path is exact); bit 1: pattern is symmetric.
 * Workspace: cgcn_coo_to_pattern_workspace_bytes(nnz, n).  Synchronises `stream`.
 */
int cgcn_coo_to_pattern_workspace_bytes(int64_t nnz, int64_t n, size_t* bytes_host);
int cgcn_coo_to_pattern(const int64_t* rows, const int64_t* cols, const float* vals, int64_t nnz, int32_t n,
                        int32_t* rowptr, int32_t* colidx, int32_t* flags_host,
                        void* workspace, size_t workspace_bytes, cgcn_stream_t stream);

/* ------------------------------------------------------- piece 2: the SpMM ---- */
typedef struct cgcn_graph {
  int32_t n;             /* windows (rows) */
  int32_t nnz;           /* stored entries of bin(A+I) */
  const int32_t* rowptr; /* [n+1] */
  const int32_t* colidx; /* [nnz], ascending inside a row */
  /* Weighted graphs (adj_type 'both', utils/util_methods.py:166-169: hic + band + I is NOT binarised, so
   * values differ inside a row).  Both NULL = pattern-only mean aggregation (hic / constant / none).
   * vals: the raw SYMMETRIC weights a_ij of the un-normalised matrix; row_inv: 1 / sum_j a_ij.
   * Forward  A_hat x = row_inv_i * sum_j a_ij x_j ; backward  A_hat^T G = A (row_inv .* G). */
  const float* vals;     /* [nnz] or NULL */
  const float* row_inv;  /* [n] or NULL */
} cgcn_graph;

/*
 * out[i,:] = scale_i * sum_{j in row i} x[j,:]  (+ residual[i,:])
 *   scale_mode 0: scale_i = 1           (backward: A_hat^T G = P (D^-1 G), D^-1 folded upstream)
 *   scale_mode 1: scale_i = 1/deg_i     (forward mean aggregation, torch.spmm(adj, .) of
 *                                        models/SubLayers.py:46 with adj = D^-1 bin(A+I))
 * With g->vals the sum is weighted by a_ij and scale_i = g->row_inv[i].
 * width = floats per row (strands*d), a multiple of 128.  residual may be NULL.
 */
int cgcn_spmm(const cgcn_graph* g, const float* x, float* out, int32_t width, int32_t scale_mode,
              const float* residual, cgcn_stream_t stream);

/*
 * Gradient of Y = A X with respect to the stored VALUES of A:  out_vals[e] = <G[row(e), :], S[col(e), :]>  for every
 * stored entry e in CSR order (an SDDMM over the pattern).  With cgcn_spmm on a graph that carries `vals` (scale_mode 0,
 * row_inv all ones) this is the generic weighted aggregation + its adjacency gradient that the reference's A-saliency
 * analysis needs (scripts/visualize.py:30-45: dense `adj` with requires_grad, then |adj * adj.grad|; :103-111: re-normalised,
 * asymmetric sparse `adj2`).  width = floats per row of G and S (multiple of 128).
 */
int cgcn_sddmm(const cgcn_graph* g, const float* G, const float* S, int32_t width, float* out_vals, cgcn_stream_t stream);

/* ------------------------------------- piece 2b: peer-memory SpMM (one graph over several GPUs) ---- */
/*
 * One graph row-partitioned over the GPUs of one NVLink / NVSwitch box (BASELINE.json configs[3]; the reference
 * has no multi-GPU GCN path, SURVEY.md 2a).  Instead of all-gathering the feature panel before every SpMM, each
 * rank PUBLISHES its row block into an exchange buffer that the other ranks map into their address space (CUDA
 * IPC), and the SpMM kernel gathers neighbour rows straight from the owner's HBM with NVLink loads: only the rows
 * a rank's edges actually touch cross the fabric (Hi-C graphs are near-diagonal, so almost none do), the local
 * block is read at HBM / L2 speed, and no [n_total][width] copy of the panel exists anywhere.
 *
 * Protocol (host): cgcn_peer_alloc on every rank -> exchange the 64-byte handles (any transport) ->
 * cgcn_peer_open the others -> per exchange step: cgcn_peer_publish (device copy into the own buffer), a
 * cross-rank barrier ordered on the stream (e.g. a one-element NCCL all-reduce), then cgcn_spmm_peer.  Two
 * buffers used alternately make one barrier per exchange sufficient.
 */
int cgcn_peer_alloc(size_t bytes, void** ptr_host, unsigned char handle_host[64]);  /* cudaMalloc + IPC handle */
int cgcn_peer_open(const unsigned char handle_host[64], void** ptr_host);           /* map a peer's buffer */
int cgcn_peer_close(void* ptr);
int cgcn_peer_free(void* ptr);
int cgcn_peer_publish(void* exchange_buffer, const void* local_panel, size_t bytes, cgcn_stream_t stream);

typedef struct cgcn_peer_panel {
  int32_t world;                          /* ranks sharing the graph, <= CGCN_MAX_PEERS */
  int32_t rank;
  int32_t row_begin[CGCN_MAX_PEERS + 1];  /* rank r owns global rows [row_begin[r], row_begin[r+1]) */
  const float* base[CGCN_MAX_PEERS];      /* base[r]: rank r's exchange buffer, row row_begin[r] first */
} cgcn_peer_panel;

/* cgcn_spmm with the gathered panel spread over the ranks' exchange buffers: g holds the LOCAL rows with GLOBAL
 * column indices; out / residual are local [g->n][width]. */
int cgcn_spmm_peer(const cgcn_graph* g, const cgcn_peer_panel* panel, float* out, int32_t width, int32_t scale_mode,
                   const float* residual, cgcn_stream_t stream);

/* ------------------------------- piece 2c: one gated GCN layer as ONE kernel (d = 128) ---- */
/*
 * The layer of models/ChromeModels.py:37-40 (and its repeat :42-46) around GraphConvolution.forward
 * (models/SubLayers.py:42-52) for `strands` interleaved feature sets, as one persistent sm_100a kernel
 * (csrc/fused_layer.cu): CSR gather-reduce -> tcgen05 3xTF32 contraction with the weights stationary in tensor
 * memory -> epilogue.
 *   sx  = P x_gather                (un-normalised neighbour sums, saved: d W = sx^T (D^-1 dy))
 *   y   = (D^-1 sx) W + b ; z = tanh(y) ; g = sigmoid(z . wg + bg)   (g == 1 when gate_off)
 *   x_out = dropout((1-g) x_in + g z)   (keep-mask of cgcn_dropout_mask(seed, step, site); dropout_p == 0: none)
 * x_gather is the panel the column indices address ([*][strands][128]; x_in itself on one GPU, the all-gathered
 * copy for a row-partitioned graph); x_in / sx / z / x_out are the local rows [g->n][strands][128]; gate is
 * [g->n][strands].  stats_partial (may be NULL): [*parts_host][2*strands*128] per-CTA column sums of relu(x_out) and
 * relu(x_out)^2 (BatchNorm statistics of the head), *parts_host <= the device's SM count.
 * Pattern graphs only (g->vals == NULL); W is [128 in][128 out] row major.
 */
int cgcn_gcn_layer_fwd(const cgcn_graph* g, int32_t strands, const float* x_gather, const float* x_in,
                       const float* W, const float* b, const float* wg, const float* bg, int32_t gate_off,
                       float dropout_p, uint64_t seed, uint64_t step, int32_t site,
                       float* sx, float* z, float* x_out, float* gate,
                       float* stats_partial, int32_t* parts_host, cgcn_stream_t stream);
/*
 * Its autograd twin for the gradient entering the layer below:  with t = D^-1 dy of THIS layer (dys, gathered through
 * the symmetric pattern) and dxd = (1-g) dh of this layer,
 *   dx = (P dys) W^T + dxd                                         (A_hat^T G W^T re-associated so the gather comes first)
 * and, when z_prev != NULL, the gate / tanh backward of the layer below on dx in the same kernel:
 *   dh = dx * mask(site_prev) ; dgp = (sum_c dh (z_prev - x_prev)) g_prev (1 - g_prev) ;
 *   dz = g_prev dh + dgp wg_prev ; dy_prev = dz (1 - z_prev^2) ; dys_out = D^-1 dy_prev ; dxd_out = (1 - g_prev) dh
 *   partial[*parts_host][2*128+4]: per-CTA column sums of dy_prev | dgp z_prev | dgp   (d b, d w_g, d b_g)
 * With z_prev == NULL, dx is written to dx_out (d loss / d x_in) and nothing else.  dxd_out may be NULL or alias dxd.
 * dropout_p must lie in [0, 1) (0: no mask), as in cgcn_gcn_layer_fwd.
 */
int cgcn_gcn_layer_bwd(const cgcn_graph* g, int32_t strands, const float* dys_gather, const float* dxd, const float* W,
                       const float* z_prev, const float* x_prev, const float* g_prev, const float* wg_prev, int32_t gate_off,
                       float dropout_p, uint64_t seed, uint64_t step, int32_t site_prev,
                       float* dys_out, float* dxd_out, float* dx_out, float* partial, int32_t* parts_host,
                       cgcn_stream_t stream);

/* ------------------------------------------------ piece 3: dense contractions ---- */
/* gemm_impl: 0 = auto (tcgen05 when the shape allows), 1 = fp32 FFMA kernel, 2 = tcgen05 3xTF32. */
/*
 * C[m x n] = rowscale * (A[m x k] * op(B)) + bias.   A row-major (lda), C row-major (ldc).
 * b_transposed 0: B is [k][n] row-major (torch.mm(input, weight), models/SubLayers.py:43);
 * b_transposed 1: B is [n][k] row-major (nn.Linear weight, models/ChromeModels.py:51).
 * bias [n] or NULL.  rowscale_rowptr: NULL, or the graph's rowptr: row r is scaled by
 * 1/deg(r / rowscale_group) (the D^-1 of A_hat^T applied to the input of the backward SpMM);
 * rowscale_inv: NULL, or the graph's row_inv (weighted graphs; takes precedence over rowscale_rowptr).
 * Any k, n: weight operands wider than 128 are cut into <= 128 x 128 blocks whose k-blocks accumulate into C
 * (d_model 256 / 512); k, n <= 128 is the single-launch case.  The tcgen05 path needs lda, ldc multiples of 4 (rows
 * padded to round_up(k|n, 4) floats).
 */
int cgcn_gemm_rowpanel(const float* A, int64_t lda, const float* B, int32_t b_transposed, const float* bias,
                       float* C, int64_t ldc, int64_t m, int32_t n, int32_t k,
                       const int32_t* rowscale_rowptr, const float* rowscale_inv, int32_t rowscale_group,
                       int32_t gemm_impl, void* workspace, size_t workspace_bytes, cgcn_stream_t stream);
/*
 * C[ka x nb] (+)= sum_r A[r][0:ka] (x) B[r][0:nb]   (weight gradients X^T G: a reduction over
 * all m rows; autograd of models/SubLayers.py:43 and models/ChromeModels.py:51).
 * Deterministic: per-CTA partial tiles in the workspace, reduced in a fixed order in fp64.
 * accumulate != 0 adds to C.  Any ka, nb (one launch pair per <= 128 x 128 block of C).
 */
size_t cgcn_gemm_gram_workspace_bytes(int64_t m);
int cgcn_gemm_gram(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t m, int32_t ka, int32_t nb, int32_t accumulate,
                   int32_t gemm_impl, void* workspace, size_t workspace_bytes, cgcn_stream_t stream);

/* ----------------------------------- the model: forward / backward / train step ---- */
/* Parameters in the reference's state_dict order and shapes (models/ChromeModels.py:22-31):
 * GC{1,2}.weight [d][d] (in x out), GC{1,2}.bias [d], W{1,2}.weight [1][d], W{1,2}.bias [1],
 * batch_norm.weight/bias [d], out.weight [nclass][d], out.bias [nclass].  A second instance of
 * this struct holds the gradients.  Slots 2.. (GC3/W3, GC4/W4) belong to the variant-sweep extension
 * (layers > 2); the reference itself never builds more than two layers (models/ChromeModels.py:26-28). */
typedef struct cgcn_params {
  float* gc_w[CGCN_MAX_LAYERS];
  float* gc_b[CGCN_MAX_LAYERS];
  float* gate_w[CGCN_MAX_LAYERS];
  float* gate_b[CGCN_MAX_LAYERS];
  float* bn_w;
  float* bn_b;
  float* out_w;
  float* out_b;
} cgcn_params;

typedef struct cgcn_model {
  cgcn_graph graph;
  int32_t d;              /* feature width: 128 (main.py:62), 256 or 512 */
  int32_t nclass;         /* <= 128 */
  int32_t layers;         /* 1 or 2 (the reference builds 2 iff gcn_layers == 2); 3..CGCN_MAX_LAYERS = extension */
  int32_t strands;        /* 1 = one forward() call; 2 = x_f and x_r of finetune.py:41-42 batched */
  int32_t training;       /* BatchNorm batch statistics + dropout (ChromeModel.train()) */
  int32_t gemm_impl;      /* see above */
  int32_t need_input_grad;/* also produce d loss / d x_in (finetune.py:33-34 asks, nothing reads it) */
  int32_t out_ld;         /* floats per (row, strand) of `out` and `out_grad`, >= nclass; 0 = nclass.  A multiple of 4
                             (e.g. 104 for nclass 103) puts the head contractions on the tcgen05 path; padding columns of
                             `out` are zero-filled and those of `out_grad` must be finite */
  float dropout_p;        /* F.dropout p (models/ChromeModels.py:42,50) */
  float bn_momentum;      /* 0.1 */
  float bn_eps;           /* 1e-5 */
  int32_t row_begin;      /* row-partitioned graphs: global index of the first local row (dropout stream position) */
  int32_t gate_off;       /* extension (variant sweep "gate off"; the reference ignores its gate argument,
                             models/ChromeModels.py:22-31): 1 = every layer is x <- tanh(A_hat x W + b), g == 1 */
  int32_t reserved0;
  uint64_t seed;          /* dropout: keep-mask is a pure function of (seed, step, site, element) */
  uint64_t step;
  cgcn_params params;
  cgcn_params grads;      /* written (not accumulated) by backward */
  float* bn_running_mean; /* [d] */
  float* bn_running_var;  /* [d] */
  int64_t* bn_num_batches_tracked; /* [1] */
  const float* x_in;      /* [n][strands][d] */
  float* x_in_grad;       /* [n][strands][d] or NULL */
  float* out;             /* [n][strands][out_ld] logits in the first nclass columns (models/ChromeModels.py:51) */
  float* gate[CGCN_MAX_LAYERS]; /* [n][strands] g, g2 (models/ChromeModels.py:39,45) */
  const float* out_grad;  /* [n][strands][out_ld], input of backward */
  float* workspace;       /* cgcn_model_workspace_bytes() bytes, kept from forward to backward */
  size_t workspace_bytes;
  cgcn_stream_t stream;
  /* One graph row-partitioned over several GPUs (cgcn_model_phase): graph.n = local rows, colidx = GLOBAL columns.
   * n_total = global row count (0 = not partitioned), x_full = [n_total][strands][d] scratch the host all-gathers
   * panels into, bn_sums = [2*strands*d] doubles the host all-reduces (BatchNorm column sums). */
  int64_t n_total;
  float* x_full;
  double* bn_sums;
  /* Alternative to x_full: the panel the next SpMM stage gathers from lives in the ranks' exchange buffers
   * (cgcn_spmm_peer).  NULL = use x_full. */
  const cgcn_peer_panel* peer;
} cgcn_model;

size_t cgcn_model_workspace_bytes(int32_t n, int32_t d, int32_t nclass, int32_t layers, int32_t strands);
/* ChromeGCN.forward (models/ChromeModels.py:34-52) for `strands` feature sets at once. */
int cgcn_model_forward(const cgcn_model* m);
/* autograd of the same: fills m->grads (and x_in_grad) from m->out_grad and the workspace. */
int cgcn_model_backward(const cgcn_model* m);

/*
 * The same model stage by stage, for ONE graph row-partitioned over several GPUs (contiguous row blocks; the
 * pattern is symmetric, so the same partition serves forward and backward).  Between stages the host performs
 * the exchange step over NCCL:
 *   all-gather x_in -> x_full ; FWD_LAYER(0) ; [all-gather *publish -> x_full ; FWD_LAYER(1)] ;
 *   all-reduce bn_sums ; FWD_HEAD ; cgcn_bce_loss(n_total) ;
 *   BWD_HEAD ; all-reduce bn_sums ; BWD_LAYER(L-1) ; [all-gather *publish -> x_full ; BWD_LAYER(L-2)] ;
 *   [need_input_grad: all-gather *publish -> x_full ; BWD_INPUT] ; all-reduce the flat gradient buffer.
 * *publish is the local panel to gather before the next stage (NULL if none).
 * With m->peer set, "all-gather X -> x_full" becomes "cgcn_peer_publish X ; barrier" and the stage's SpMM reads
 * the peers' exchange buffers directly (no x_full).
 */
enum { CGCN_PHASE_FWD_LAYER = 0, CGCN_PHASE_FWD_HEAD = 1, CGCN_PHASE_BWD_HEAD = 2, CGCN_PHASE_BWD_LAYER = 3, CGCN_PHASE_BWD_INPUT = 4 };
int cgcn_model_phase(const cgcn_model* m, int32_t kind, int32_t layer, const float** publish);

/*
 * finetune.py:43-45,52: pred = mean over strands of the logits; loss = BCE-with-logits, mean over
 * n x nclass; probs = sigmoid(pred).  `out` and `out_grad` rows are out_ld floats apart (>= nclass).
 * Writes loss_sum_out[0] += loss (a device accumulator, like `total_loss += loss.item()` without the
 * sync), probs [n][nclass] (may be NULL), and, if out_grad != NULL, d loss / d out (padding columns 0).
 */
size_t cgcn_bce_workspace_bytes(int32_t n, int32_t nclass);
int cgcn_bce_loss(const float* out, const float* target, int32_t n, int32_t nclass, int32_t strands, int32_t out_ld,
                  int64_t n_total /* rows the mean runs over; 0 = n (row-partitioned graphs pass the global count) */,
                  float* probs, float* loss_sum_out, float* out_grad,
                  void* workspace, size_t workspace_bytes, cgcn_stream_t stream);
/* Same with bit-packed labels: target_bits [n][(nclass+31)/32] uint32, bit (c & 31) of word c >> 5 of a row
 * = label c (numpy packbits, bitorder 'little').  The label matrix of finetune.py:32 is 0/1 and is the one
 * input that does not change between epochs, so the host packs it once and each pass moves 1/26 of the
 * float matrix over PCIe. */
int cgcn_bce_loss_bits(const float* out, const uint32_t* target_bits, int32_t n, int32_t nclass, int32_t strands,
                       int32_t out_ld, int64_t n_total, float* probs, float* loss_sum_out, float* out_grad,
                       void* workspace, size_t workspace_bytes, cgcn_stream_t stream);

/* One iteration of the chromosome loop of finetune.py:39-53 for split == 'train':
 * forward (both strands), loss, backward.  The optimiser step is cgcn_sgd_step / cgcn_adam_step. */
int cgcn_train_step(const cgcn_model* m, const float* target, float* probs, float* loss_sum_out,
                    float* out_grad_scratch);
int cgcn_train_step_bits(const cgcn_model* m, const uint32_t* target_bits, float* probs, float* loss_sum_out,
                         float* out_grad_scratch);

/* ------------------------------------------------------- split metrics ---- */
/*
 * Per-label ranking metrics of one split, replacing the sklearn calls of utils/metrics.py that
 * utils/evals.py:86-90 makes once per split per epoch (runner.py:41,45,51) on the [n][nclass] probability
 * matrix: roc_auc_score (utils/metrics.py:238-253), precision_recall_curve + auc (:168-183), the recall at
 * the lowest threshold whose 1 - precision <= fdr_cutoff (:148-165) and average_precision_score (:25-26).
 * preds [n][pred_ld] fp32 (device); labels either as floats targets [n][target_ld] (non-zero = positive) or as
 * bit rows target_bits [n][(nclass+31)/32] (exactly one of the two non-NULL).
 * out (device, double) [5][nclass]: AUROC (NaN for a label with a single class: roc_auc_score raises and the
 * reference skips it), AUPR, recall at the cutoff, average precision, number of positives.
 * Equal scores form one threshold, exactly like sklearn's distinct-threshold curves; results agree with
 * sklearn to fp64 rounding (tests: 1e-9).  Enqueues on `stream`; no allocation, no synchronisation.
 */
size_t cgcn_label_metrics_workspace_bytes(int64_t n, int32_t nclass);
int cgcn_label_metrics(const float* preds, int64_t pred_ld, const float* targets, int64_t target_ld,
                       const uint32_t* target_bits, int64_t n, int32_t nclass, double fdr_cutoff, double* out,
                       void* workspace, size_t workspace_bytes, cgcn_stream_t stream);

/* ------------------------------------------------------------- optimiser ---- */
/* torch.optim.SGD(lr, momentum, weight_decay) as built by utils/util_methods.py:18-19, over one flat
 * buffer: g += wd*p ; buf = momentum*buf + g ; p -= lr*buf.  grad_scale multiplies g first (1/world
 * for data-parallel averaging, else 1). */
int cgcn_sgd_step(float* params, const float* grads, float* momentum_buf, int64_t count,
                  float lr, float momentum, float weight_decay, float grad_scale, cgcn_stream_t stream);
/* torch.optim.Adam(lr, betas) as built by utils/util_methods.py:16-17 (eps 1e-8, no weight decay);
 * step_index counts from 1. */
int cgcn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t count,
                   float lr, float beta1, float beta2, float eps, int64_t step_index, float grad_scale,
                   cgcn_stream_t stream);

/* ------------------------------------------ collectives for a non-Python host ---- */
/* The multi-GPU paths need three exchanges and nothing else: the flat-gradient sum of the chromosome-sharded pass
 * (the reference has ONE model and steps it once per chromosome, finetune.py:46-49; N replicas must sum their
 * gradients before the shared step), the BatchNorm column sums of the row-partitioned graph (models/ChromeModels.py:49
 * normalises over ALL windows of the chromosome), and -- only for the copy-based exchange -- the all-gather of a
 * panel's row blocks.  The Python host uses torch.distributed for them (chromegcn_b200/dist.py); these entry points
 * give a C / C++ / Go host the same three calls over NCCL without any Python.  NCCL is loaded at first use with
 * dlopen("libnccl.so.2") (the copy already mapped into the process if there is one): the library itself carries no
 * link-time NCCL dependency, and every call returns CGCN_ERR_INVALID with a message when NCCL cannot be loaded.
 * One communicator per process, bound to the device that is current at cgcn_comm_init. */
typedef struct cgcn_comm* cgcn_comm_t;
#define CGCN_COMM_ID_BYTES 128
/* rank 0: fill 128 bytes; the host ships them to the other ranks by its own means (file, socket, MPI) */
int cgcn_comm_unique_id(unsigned char id_host[CGCN_COMM_ID_BYTES]);
/* collective over all ranks of the job */
int cgcn_comm_init(cgcn_comm_t* comm_host, const unsigned char id_host[CGCN_COMM_ID_BYTES], int32_t world, int32_t rank);
int cgcn_comm_destroy(cgcn_comm_t comm);
/* buf (device, fp32) <- sum over ranks, in place; enqueued on `stream` */
int cgcn_comm_allreduce_sum(cgcn_comm_t comm, float* buf, size_t count, cgcn_stream_t stream);
/* recv[r * bytes_per_rank ...] <- rank r's `send` (device buffers; recv holds world * bytes_per_rank bytes) */
int cgcn_comm_allgather(cgcn_comm_t comm, const void* send, void* recv, size_t bytes_per_rank, cgcn_stream_t stream);

/* --------------------------------------------------------------- utilities ---- */
/* Read-bandwidth probe (measurement aid, tools/l2_bw.py): streams `bytes` of `buf` `reps` times with L2-only loads.  A
 * buffer that fits L2 gives the L2 -> SM read rate, one of several GB the HBM read rate.  sink: one float. */
int cgcn_membw_read(const float* buf, size_t bytes, int32_t reps, float* sink, cgcn_stream_t stream);
/* [n][d] x strands  <->  [n][strands][d].  src/dst arrays of `strands` pointers are HOST arrays. */
int cgcn_interleave_strands(const float* const* src_host, int32_t strands, int32_t n, int32_t d, float* dst,
                            cgcn_stream_t stream);
int cgcn_deinterleave_strands(const float* src, int32_t strands, int32_t n, int32_t width, float* const* dst_host,
                              cgcn_stream_t stream);
/* The keep-mask (0 or 1/(1-p)) the model draws at dropout site `site` (0: between the layers,
 * 1: after BatchNorm) for (seed, step): lets a test inject the same mask into the oracle. */
int cgcn_dropout_mask(float* mask, int32_t n, int32_t strands, int32_t d, float p, uint64_t seed, uint64_t step,
                      int32_t site, cgcn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CHROMEGCN_H_ */
