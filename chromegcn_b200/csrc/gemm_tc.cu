// tcgen05 / TMEM dense contractions for the GCN path (sm_100a), fp32-faithful via 3xTF32.
//
// The two contraction shapes of the model (see gemm_ffma.cu) on the 5th-generation tensor cores:
//
//   row panel  C[m x 128] = rowscale * (A[m x 128] * Bw) + bias       (A_hat x) W ,  G W^T
//   gram       C[128x128] = sum_r A[r,:]^T (x) B[r,:]                 weight gradients X^T G
//
// fp32 parity (<= 1e-5, BASELINE.md) rules out a single TF32 pass (8.8e-5).  Every fp32 operand v is
// split in registers into hi = rna_tf32(v) and lo = rna_tf32(v - hi) (the subtraction is exact in
// fp32), and each tile accumulates hi*hi + lo*hi + hi*lo in the fp32 TMEM
// accumulator: three kind::tf32 MMAs per k-step.  Because the split needs the operands in registers
// anyway, tiles are staged global -> registers -> shared memory by producer warps that write the
// UMMA canonical SWIZZLE_128B layout directly (no TMA descriptor): 16-byte chunk c of 128-byte row r
// lands at  (r/8)*1024 + (r%8)*128 + ((c ^ (r%8)) * 16).
//
// Warp roles (416 threads, one CTA per SM, persistent over tiles):
//   warps 0-3   epilogue: tcgen05.ld the accumulator (lane = tile row), scale/bias, 128-bit stores
//   warp  4     TMEM alloc/dealloc + the single-thread tcgen05.mma issuer
//   warps 5-12  producers: coalesced 128-bit global loads, hi/lo split, swizzled st.shared,
//               fence.proxy.async, mbarrier arrive
// Pipelines: smem stage full/empty mbarriers (producers <-> MMA, freed by tcgen05.commit) and, in
// the row-panel kernel, a double-buffered TMEM accumulator (MMA <-> epilogue).
#include <cstdlib>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace cgcn {

void gram_finalize_launch(const float* partial, int parts, int part_stride, int pld, int ka, int nb, float* C,
                          int64_t ldc, int accumulate, cudaStream_t stream);
int64_t gram_rows_per_cta(int64_t m);
size_t gram_workspace_bytes(int64_t m);

namespace tc {

constexpr int TILE = 128;
constexpr int KCH = 32;                               // floats per 128-byte swizzle row
constexpr int ATOM_BYTES = 1024;                      // 8 rows x 128 B
constexpr int CHUNK_BYTES = TILE * KCH * 4;           // 128 rows x 128 B = 16 KB
constexpr int STAGES = 3;                             // gram kernel
constexpr int RP_STAGES = 2;                          // row-panel kernel (B image + epilogue staging need the room)
constexpr int STG_PITCH = 36;                         // floats per staged row: 128-bit accesses stay bank-conflict free
constexpr int STG_BYTES = 4 * 32 * STG_PITCH * 4;     // 4 epilogue warps x 32 rows x 36 floats = 18 KB
constexpr int NUM_EPI_WARPS = 4, NUM_PROD_WARPS = 8;
constexpr int MMA_WARP = NUM_EPI_WARPS;
constexpr int THREADS = (NUM_EPI_WARPS + 1 + NUM_PROD_WARPS) * 32;      // 416
constexpr int PROD_THREADS = NUM_PROD_WARPS * 32;

// Epilogue write-out of one 32-row x 32-column accumulator block held "thread = row" (tcgen05.ld 32x32b):
// a row-per-thread global store would touch 32 different 128-byte lines per instruction (measured: 15 k
// cycles per tile).  Stage through a padded per-warp shared-memory block instead and let 8 lanes write
// one contiguous 128-byte row segment: 4 full lines per warp instruction.
__device__ __forceinline__ void store_block_coalesced(uint32_t stg, const uint4 (&o)[8], int lane, float* __restrict__ dst_base,
                                                      int64_t ld, int64_t row_first, int64_t row_limit, int col0,
                                                      int col_limit, bool accumulate = false) {
#pragma unroll
  for (int j = 0; j < 8; ++j) sts128(stg + (lane * STG_PITCH + 4 * j) * 4, o[j]);
  __syncwarp();
  const int q = lane & 7, rsub = lane >> 3;
  uint4 v[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) v[it] = lds128(stg + ((it * 4 + rsub) * STG_PITCH + 4 * q) * 4);
  const int col = col0 + 4 * q;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int64_t grow = row_first + it * 4 + rsub;
    if (grow < row_limit && col < col_limit) {
      if (accumulate) {
        const float4 o = *reinterpret_cast<const float4*>(dst_base + grow * ld + col);
        v[it] = make_uint4(__float_as_uint(__uint_as_float(v[it].x) + o.x), __float_as_uint(__uint_as_float(v[it].y) + o.y),
                           __float_as_uint(__uint_as_float(v[it].z) + o.z), __float_as_uint(__uint_as_float(v[it].w) + o.w));
      }
      *reinterpret_cast<uint4*>(dst_base + grow * ld + col) = v[it];
    }
  }
  __syncwarp();
}

// ------------------------------------------------------------------ B image (weights) preparation
// img[(hi|lo)][kchunk 4][n 128][32 floats] in the K-major SWIZZLE_128B layout; Bw(n,k) is the weight
// that multiplies A[:,k] into C[:,n].
__global__ void tc_prep_b_kernel(const float* __restrict__ B, int b_transposed, int n_valid, int k_valid, int64_t ldb,
                                 uint32_t* __restrict__ img) {
  pdl_grid_sync();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= TILE * TILE) return;
  const int n = idx >> 7, k = idx & 127;
  float v = 0.f;                                               // zero padding up to 128 x 128
  if (n < n_valid && k < k_valid) v = b_transposed ? __ldg(B + n * ldb + k) : __ldg(B + k * ldb + n);
  uint32_t hi, lo;
  split_tf32(v, hi, lo);
  const int kc = k >> 5, kk = k & 31;
  const int off = (kc * CHUNK_BYTES + (n >> 3) * ATOM_BYTES + (n & 7) * 128 + (((kk >> 2) ^ (n & 7)) << 4) + (kk & 3) * 4) >> 2;
  img[off] = hi;
  img[(4 * CHUNK_BYTES >> 2) + off] = lo;
}

// All weight images one model pass needs, in ONE launch (blockIdx.y = image): the weights only change at the
// optimiser step, so the forward (and the backward) pass prepares its images up front instead of once per
// contraction on the critical path.
constexpr int PREP_MAX = 8;
struct PrepBatchArgs {
  const float* B[PREP_MAX];
  uint32_t* img[PREP_MAX];
  int b_transposed[PREP_MAX], n_valid[PREP_MAX], k_valid[PREP_MAX];
};
__global__ void tc_prep_b_batch_kernel(const PrepBatchArgs a) {
  pdl_grid_sync();
  const int w = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= TILE * TILE) return;
  const int n = idx >> 7, k = idx & 127;
  const int n_valid = a.n_valid[w], k_valid = a.k_valid[w];
  const float* __restrict__ B = a.B[w];
  float v = 0.f;
  if (n < n_valid && k < k_valid) v = a.b_transposed[w] ? __ldg(B + n * k_valid + k) : __ldg(B + k * n_valid + n);
  uint32_t hi, lo;
  split_tf32(v, hi, lo);
  const int kc = k >> 5, kk = k & 31;
  const int off = (kc * CHUNK_BYTES + (n >> 3) * ATOM_BYTES + (n & 7) * 128 + (((kk >> 2) ^ (n & 7)) << 4) + (kk & 3) * 4) >> 2;
  a.img[w][off] = hi;
  a.img[w][(4 * CHUNK_BYTES >> 2) + off] = lo;
}

// ------------------------------------------------------------------ row-panel kernel
struct RowPanelTcArgs {
  const float* A;
  int64_t lda;
  const uint32_t* b_img;       // 128 KB prepared image
  const float* bias;
  float* C;
  int64_t ldc;
  int64_t m;
  int64_t rows_per_cta;        // each CTA owns one contiguous row range (its last tile may be partial)
  const int32_t* rowscale_rowptr;
  const float* rowscale_inv;
  int rowscale_group;
  int n_valid, k_valid;        // <= 128; A rows hold round_up(k_valid, 4) readable floats, C rows round_up(n_valid, 4) writable
  long long* trace;            // developer aid (CGCN_TC_TRACE=1): per-role clock64() stamps of CTA 0, else NULL
  int accumulate;              // C += ... (k-blocked contractions wider than 128)
};

#define TC_TRACE(slot, idx)                                                                   \
  do {                                                                                        \
    if (p.trace != nullptr && blockIdx.x == 0 && lane == 0 && (idx) < 64) p.trace[(slot) * 64 + (idx)] = clock64(); \
  } while (0)

constexpr int RP_B_BYTES = 2 * 4 * CHUNK_BYTES;                 // hi + lo, 4 k-chunks: 128 KB
constexpr int RP_STAGE_BYTES = 2 * CHUNK_BYTES;                 // A hi + lo of one k-chunk: 32 KB
constexpr int RP_SMEM = RP_B_BYTES + RP_STAGES * RP_STAGE_BYTES + STG_BYTES + 256 + 512 + 1024;   // + barriers + bias

__global__ void __launch_bounds__(THREADS, 1) gemm_rowpanel_tc_kernel(const RowPanelTcArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sB = base;
  const uint32_t sA = base + RP_B_BYTES;
  const uint32_t sStg = sA + RP_STAGES * RP_STAGE_BYTES;        // epilogue staging, 4 warps x 4.5 KB
  const uint32_t sBar = sStg + STG_BYTES;                       // full[S] empty[S] tfull[2] tempty[2] | tmem ptr
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * RP_STAGES, bar_tfull = sBar + 16 * RP_STAGES, bar_tempty = bar_tfull + 16;
  const uint32_t s_tmem_ptr = bar_tempty + 16, bar_b = bar_tempty + 24;
  const uint32_t sBias = sBar + 256;                            // 128 floats (zero padded): the L1 is all shared memory here
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));        // generic pointer to the aligned base
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Contiguous, equally sized row range per CTA instead of round-robin whole tiles: the kernel is bound by
  // the bytes it moves, and a partial last tile moves only its valid rows, so every SM carries the same
  // traffic (m / grid rows) even when m / 128 is not a multiple of the grid.
  const int64_t r_begin = static_cast<int64_t>(blockIdx.x) * p.rows_per_cta;
  const int64_t r_end = r_begin + p.rows_per_cta < p.m ? r_begin + p.rows_per_cta : p.m;
  const int ntile = r_end > r_begin ? static_cast<int>((r_end - r_begin + TILE - 1) / TILE) : 0;

  // Set-up that touches no global memory (barriers, TMEM allocation) runs before the grid dependency resolves, i.e.
  // while the previous kernel of the stream is still draining (programmatic dependent launch).
  if (threadIdx.x == 0) {
    for (int s = 0; s < RP_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, NUM_PROD_WARPS);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, NUM_EPI_WARPS);
    }
    mbar_init(bar_b, 1);
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(s_tmem_ptr, 256);
  pdl_grid_sync();

  if (threadIdx.x < TILE)
    reinterpret_cast<float*>(gen + (sBias - base))[threadIdx.x] =
        (p.bias != nullptr && static_cast<int>(threadIdx.x) < p.n_valid) ? __ldg(p.bias + threadIdx.x) : 0.f;

  // Producers put their first tile's loads in flight first: the B image copy below then overlaps with the DRAM
  // latency of the first A tile.
  const int pt = static_cast<int>(threadIdx.x) - (MMA_WARP + 1) * 32;      // 0..255 for producer threads
  float4 v[4][4];      // register ring: one whole tile (4 k-chunks x 4 float4) of look-ahead = 64 KB in flight per SM
  auto issue = [&](int t, int kc) {
    const int64_t row0 = r_begin + static_cast<int64_t>(t) * TILE;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int u = pt + PROD_THREADS * i;
      const int r = u >> 3, c = u & 7;
      const int64_t grow = row0 + r;
      const int col = kc * KCH + c * 4;
      v[kc][i] = (grow < r_end && col < p.k_valid) ? ldg4(p.A + grow * p.lda + col) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  if (warp > MMA_WARP) {
#pragma unroll
    for (int kc = 0; kc < 4; ++kc) issue(0, kc);
  }

  // The B image (already swizzled by tc_prep_b_kernel) as 8 x 16 KB bulk copies that complete on bar_b: nothing but
  // the first MMA waits for them.
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar_b, RP_B_BYTES);
#pragma unroll 1
    for (int i = 0; i < RP_B_BYTES / CHUNK_BYTES; ++i)
      bulk_g2s(sB + i * CHUNK_BYTES, reinterpret_cast<const uint8_t*>(p.b_img) + i * CHUNK_BYTES, CHUNK_BYTES, bar_b);
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + (s_tmem_ptr - base));

  if (warp > MMA_WARP) {
    // ===================== producers =====================
    uint32_t stage = 0, phase = 0;
    for (int t = 0; t < ntile; ++t) {
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        if (warp == MMA_WARP + 1) TC_TRACE(0, t * 4 + kc);
        const uint32_t sHi = sA + stage * RP_STAGE_BYTES, sLo = sHi + CHUNK_BYTES;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int u = pt + PROD_THREADS * i;
          const int r = u >> 3, c = u & 7;
          const uint32_t off = (r >> 3) * ATOM_BYTES + (r & 7) * 128 + ((c ^ (r & 7)) << 4);
          uint4 hi, lo;
          split4(v[kc][i], hi, lo);
          sts128(sHi + off, hi);
          sts128(sLo + off, lo);
        }
        if (warp == MMA_WARP + 1) TC_TRACE(1, t * 4 + kc);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * stage);
        if (warp == MMA_WARP + 1) TC_TRACE(2, t * 4 + kc);
        if (t + 1 < ntile) issue(t + 1, kc);                    // refill this slot for the next tile
        if (++stage == RP_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc(false, false);
    uint32_t stage = 0, phase = 0;
    if (ntile > 0) mbar_wait(bar_b, 0);                         // weights image landed
    for (uint32_t it = 0; it < static_cast<uint32_t>(ntile); ++it) {
      const uint32_t acc = it & 1;
      mbar_wait(bar_tempty + 8 * acc, ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * TILE;
      for (int kc = 0; kc < 4; ++kc) {
        mbar_wait(bar_full + 8 * stage, phase);
        tc_fence_after();
        TC_TRACE(3, static_cast<int>(it) * 4 + kc);
        if (lane == 0) {
          const uint32_t aHi = sA + stage * RP_STAGE_BYTES, aLo = aHi + CHUNK_BYTES;
          const uint32_t bHi = sB + kc * CHUNK_BYTES, bLo = bHi + 4 * CHUNK_BYTES;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t dah = make_desc(aHi + ks * 32, 16, ATOM_BYTES), dal = make_desc(aLo + ks * 32, 16, ATOM_BYTES);
            const uint64_t dbh = make_desc(bHi + ks * 32, 16, ATOM_BYTES), dbl = make_desc(bLo + ks * 32, 16, ATOM_BYTES);
            umma_tf32(d_tmem, dal, dbh, idesc, (kc | ks) != 0);      // small terms first
            umma_tf32(d_tmem, dah, dbl, idesc, 1);
            umma_tf32(d_tmem, dah, dbh, idesc, 1);
          }
          umma_commit(bar_empty + 8 * stage);                     // frees the stage when these MMAs retire
          if (kc == 3) umma_commit(bar_tfull + 8 * acc);          // accumulator complete
        }
        TC_TRACE(4, static_cast<int>(it) * 4 + kc);
        __syncwarp();
        if (++stage == RP_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    // ===================== epilogue =====================
    for (uint32_t it = 0; it < static_cast<uint32_t>(ntile); ++it) {
      const uint32_t acc = it & 1;
      mbar_wait(bar_tfull + 8 * acc, (it >> 1) & 1);
      tc_fence_after();
      const int64_t tile_row0 = r_begin + static_cast<int64_t>(it) * TILE;
      const int64_t grow = tile_row0 + warp * 32 + lane;
      float scale = 1.0f;
      if ((p.rowscale_rowptr != nullptr || p.rowscale_inv != nullptr) && grow < r_end)
        scale = row_scale(p.rowscale_rowptr, p.rowscale_inv, static_cast<int>(grow / p.rowscale_group));
      const uint32_t stg = sStg + warp * (32 * STG_PITCH * 4);
      const int n_store = (p.n_valid + 3) & ~3;
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        if (cc * 32 >= n_store) break;                          // warp-uniform
        uint32_t r[32];
        if (warp == 0) TC_TRACE(5, static_cast<int>(it) * 8 + cc * 2);
        tmem_ld32(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + acc * TILE + cc * 32, r);
        if (warp == 0) TC_TRACE(5, static_cast<int>(it) * 8 + cc * 2 + 1);
        uint4 o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int col = cc * 32 + 4 * j;
          const uint4 bq = lds128(sBias + col * 4);             // broadcast read, zero beyond n_valid
          const float4 f = make_float4(fmaf(__uint_as_float(r[4 * j]), scale, __uint_as_float(bq.x)),
                                       fmaf(__uint_as_float(r[4 * j + 1]), scale, __uint_as_float(bq.y)),
                                       fmaf(__uint_as_float(r[4 * j + 2]), scale, __uint_as_float(bq.z)),
                                       fmaf(__uint_as_float(r[4 * j + 3]), scale, __uint_as_float(bq.w)));
          o[j] = make_uint4(__float_as_uint(f.x), __float_as_uint(f.y), __float_as_uint(f.z), __float_as_uint(f.w));
        }
        if (warp == 0) TC_TRACE(6, static_cast<int>(it) * 8 + cc * 2);
        store_block_coalesced(stg, o, lane, p.C, p.ldc, tile_row0 + warp * 32, r_end, cc * 32, n_store, p.accumulate != 0);
        if (warp == 0) TC_TRACE(6, static_cast<int>(it) * 8 + cc * 2 + 1);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ------------------------------------------------------------------ gram kernel
struct GramTcArgs {
  const float* A;
  int64_t lda;
  const float* B;
  int64_t ldb;
  int64_t m;
  int64_t rows_per_cta;        // multiple of 32
  float* partial;              // [gridDim.x][128][128]
  int ka_valid, nb_valid;      // <= 128; rows hold round_up(valid, 4) readable floats
};

constexpr int GR_OP_BYTES = 2 * CHUNK_BYTES;                     // one operand, hi + lo, 32 rows x 128 cols: 32 KB
constexpr int GR_STAGE_BYTES = 2 * GR_OP_BYTES;                  // A + B: 64 KB
constexpr int GR_SMEM = STAGES * GR_STAGE_BYTES + STG_BYTES + 256 + 1024;
constexpr int GR_SLOTS = 2;                                      // register look-ahead of the producers, in 32-row chunks

__global__ void __launch_bounds__(THREADS, 1) gemm_gram_tc_kernel(const GramTcArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sS = base;
  const uint32_t sStg = base + STAGES * GR_STAGE_BYTES;
  const uint32_t sBar = sStg + STG_BYTES;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * STAGES, bar_tfull = sBar + 16 * STAGES;
  const uint32_t s_tmem_ptr = bar_tfull + 8;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int64_t r_begin = static_cast<int64_t>(blockIdx.x) * p.rows_per_cta;
  const int64_t r_end = min(r_begin + p.rows_per_cta, p.m);
  const int chunks = static_cast<int>((r_end - r_begin + KCH - 1) / KCH);       // >= 1 by construction

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, NUM_PROD_WARPS);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_tfull, 1);
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(s_tmem_ptr, 128);
  pdl_grid_sync();                   // nothing above touches global memory
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + (s_tmem_ptr - base));

  if (warp > MMA_WARP) {
    // producers: 32 rows x 128 floats of A and of B per stage; one warp moves one 512-byte row per
    // instruction.  MN-major 32-bit operands must use SWIZZLE_128B_BASE32B (the only MN-major layout
    // kind::tf32 accepts): 128-byte rows (32 MN elements of one k), atoms of 4 k-rows, 32-byte chunks
    // XOR-ed with (k % 4).  16-byte chunk c (floats 4c..4c+3) of row r goes to
    // (c/8)*4096 + r*128 + ((((c%8)/2) ^ (r%4)) * 32) + (c%2)*16      [LBO = 4096, SBO = 512].
    const int pt = threadIdx.x - (MMA_WARP + 1) * 32;
    uint32_t stage = 0, phase = 0;
    // GR_SLOTS chunks of look-ahead in registers (8 float4 per thread and chunk: 32 KB per chunk in flight per SM)
    float4 va[GR_SLOTS][4], vb[GR_SLOTS][4];
    auto issue = [&](int ch, int slot) {
      const int64_t row0 = r_begin + static_cast<int64_t>(ch) * KCH;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int u = pt + PROD_THREADS * i;
        const int r = u >> 5, c = u & 31;
        const int64_t grow = row0 + r;
        const bool ok = ch < chunks && grow < r_end;
        va[slot][i] = (ok && c * 4 < p.ka_valid) ? ldg4(p.A + grow * p.lda + c * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        vb[slot][i] = (ok && c * 4 < p.nb_valid) ? ldg4(p.B + grow * p.ldb + c * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
#pragma unroll
    for (int slot = 0; slot < GR_SLOTS; ++slot) issue(slot, slot);
    for (int ch0 = 0; ch0 < chunks; ch0 += GR_SLOTS) {
#pragma unroll
      for (int slot = 0; slot < GR_SLOTS; ++slot) {
        const int ch = ch0 + slot;
        if (ch >= chunks) break;
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        const uint32_t sAh = sS + stage * GR_STAGE_BYTES, sAl = sAh + CHUNK_BYTES;
        const uint32_t sBh = sAh + GR_OP_BYTES, sBl = sBh + CHUNK_BYTES;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int u = pt + PROD_THREADS * i;
          const int r = u >> 5, c = u & 31;
          const uint32_t off = (c >> 3) * 4096 + r * 128 + ((((c & 7) >> 1) ^ (r & 3)) << 5) + ((c & 1) << 4);
          uint4 hi, lo;
          split4(va[slot][i], hi, lo);
          sts128(sAh + off, hi);
          sts128(sAl + off, lo);
          split4(vb[slot][i], hi, lo);
          sts128(sBh + off, hi);
          sts128(sBl + off, lo);
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * stage);
        issue(ch + GR_SLOTS, slot);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    constexpr uint32_t idesc = make_idesc(true, true);
    uint32_t stage = 0, phase = 0;
    for (int ch = 0; ch < chunks; ++ch) {
      mbar_wait(bar_full + 8 * stage, phase);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t aHi = sS + stage * GR_STAGE_BYTES, aLo = aHi + CHUNK_BYTES;
        const uint32_t bHi = aHi + GR_OP_BYTES, bLo = bHi + CHUNK_BYTES;
#pragma unroll
        for (int kg = 0; kg < 4; ++kg) {
          const uint64_t dah = make_desc(aHi + kg * 1024, 4096, 512, 1), dal = make_desc(aLo + kg * 1024, 4096, 512, 1);
          const uint64_t dbh = make_desc(bHi + kg * 1024, 4096, 512, 1), dbl = make_desc(bLo + kg * 1024, 4096, 512, 1);
          umma_tf32(tmem_base, dal, dbh, idesc, (ch | kg) != 0);
          umma_tf32(tmem_base, dah, dbl, idesc, 1);
          umma_tf32(tmem_base, dah, dbh, idesc, 1);
        }
        umma_commit(bar_empty + 8 * stage);
        if (ch == chunks - 1) umma_commit(bar_tfull);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else {
    mbar_wait(bar_tfull, 0);
    tc_fence_after();
    float* dst = p.partial + static_cast<size_t>(blockIdx.x) * TILE * TILE;      // row of C = column of A
    const uint32_t stg = sStg + warp * (32 * STG_PITCH * 4);
#pragma unroll 1
    for (int cc = 0; cc < 4; ++cc) {
      uint32_t r[32];
      tmem_ld32(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + cc * 32, r);
      uint4 o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
      store_block_coalesced(stg, o, lane, dst, TILE, warp * 32, TILE, cc * 32, TILE);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

}  // namespace tc

// ------------------------------------------------------------------ host side
static bool aligned16(const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; }

static int up4(int v) { return (v + 3) / 4 * 4; }
bool tc_rowpanel_supported(int64_t lda, int64_t ldc, int n, int k, const void* A, const void* C) {
  return n >= 1 && n <= 128 && k >= 1 && k <= 128 && lda % 4 == 0 && ldc % 4 == 0 && lda >= up4(k) && ldc >= up4(n) &&
         aligned16(A) && aligned16(C);
}
bool tc_gram_supported(int64_t lda, int64_t ldb, int ka, int nb, const void* A, const void* B) {
  return ka >= 1 && ka <= 128 && nb >= 1 && nb <= 128 && lda % 4 == 0 && ldb % 4 == 0 && lda >= up4(ka) && ldb >= up4(nb) &&
         aligned16(A) && aligned16(B);
}
size_t tc_workspace_bytes() { return tc::RP_B_BYTES + 256; }

// Prepare up to 8 weight images with one launch.  specs[i].img: tc_workspace_bytes() bytes, 16-byte aligned.
int tc_prep_images(const TcImageSpec* specs, int count, cudaStream_t stream) {
  CGCN_REQUIRE(count >= 0 && count <= tc::PREP_MAX, "tc_prep_images: count=%d", count);
  if (count == 0) return CGCN_OK;
  tc::PrepBatchArgs a{};
  for (int i = 0; i < count; ++i) {
    CGCN_REQUIRE(specs[i].B && specs[i].img && aligned16(specs[i].img) && specs[i].n >= 1 && specs[i].n <= 128 && specs[i].k >= 1 &&
                     specs[i].k <= 128,
                 "tc_prep_images: bad spec %d", i);
    a.B[i] = specs[i].B;
    a.img[i] = static_cast<uint32_t*>(specs[i].img);
    a.b_transposed[i] = specs[i].b_transposed;
    a.n_valid[i] = specs[i].n;
    a.k_valid[i] = specs[i].k;
  }
  CGCN_CUDA(launch_k(tc::tc_prep_b_batch_kernel, dim3((tc::TILE * tc::TILE + 255) / 256, count), dim3(256), 0, stream, a));
  return check_launch("tc_prep_b_batch_kernel");
}

int gemm_rowpanel_tc(const float* A, int64_t lda, const float* B, int b_transposed, const float* bias, float* C,
                     int64_t ldc, int64_t m, int n, int k, const int32_t* rowscale_rowptr, const float* rowscale_inv, int rowscale_group,
                     void* workspace, size_t workspace_bytes, const void* ready_image, cudaStream_t stream, int64_t ldb,
                     int accumulate) {
  CGCN_REQUIRE(A && B && C, "cgcn_gemm_rowpanel: null operand");
  if (ldb <= 0) ldb = b_transposed ? k : n;
  CGCN_REQUIRE(tc_rowpanel_supported(lda, ldc, n, k, A, C),
               "cgcn_gemm_rowpanel(tcgen05): needs n, k <= 128 and 16-byte aligned rows padded to a multiple of 4 floats");
  CGCN_REQUIRE(bias == nullptr || aligned16(bias), "cgcn_gemm_rowpanel(tcgen05): bias must be 16-byte aligned");
  if (ready_image == nullptr && (workspace == nullptr || workspace_bytes < tc_workspace_bytes() || !aligned16(workspace))) {
    set_error("cgcn_gemm_rowpanel(tcgen05): needs a %zu-byte, 16-byte aligned workspace", tc_workspace_bytes());
    return CGCN_ERR_WORKSPACE;
  }
  if (m <= 0) return CGCN_OK;
  static bool attr_set[64] = {};
  if (first_use_on_device(attr_set)) {
    CGCN_CUDA(cudaFuncSetAttribute(tc::gemm_rowpanel_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::RP_SMEM));
  }
  const uint32_t* img = static_cast<const uint32_t*>(ready_image);      // prepared by tc_prep_images for this (B, n, k)
  if (img == nullptr) {
    uint32_t* fresh = static_cast<uint32_t*>(workspace);
    CGCN_CUDA(launch_k(tc::tc_prep_b_kernel, dim3((tc::TILE * tc::TILE + 255) / 256), dim3(256), 0, stream, B, b_transposed, n, k, ldb, fresh));
    CGCN_TRY(check_launch("tc_prep_b_kernel"));
    img = fresh;
  }
  const int64_t tiles = (m + tc::TILE - 1) / tc::TILE;
  int grid = static_cast<int>(tiles < sm_count() ? tiles : sm_count());
  const int64_t rows_per_cta = ((m + grid - 1) / grid + 7) / 8 * 8;
  grid = static_cast<int>((m + rows_per_cta - 1) / rows_per_cta);
  tc::RowPanelTcArgs p{A, lda, img, bias, C, ldc, m, rows_per_cta, rowscale_rowptr, rowscale_inv, rowscale_group, n, k, nullptr, accumulate};
  static const bool trace = getenv("CGCN_TC_TRACE") != nullptr;
  if (trace) {                                                  // developer aid: synchronous, prints CTA 0's timeline
    long long* d = nullptr;
    CGCN_CUDA(cudaMalloc(&d, 7 * 64 * sizeof(long long)));
    CGCN_CUDA(cudaMemset(d, 0, 7 * 64 * sizeof(long long)));
    p.trace = d;
    tc::gemm_rowpanel_tc_kernel<<<grid, tc::THREADS, tc::RP_SMEM, stream>>>(p);
    CGCN_CUDA(cudaStreamSynchronize(stream));
    long long h[7 * 64];
    CGCN_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
    cudaFree(d);
    static const char* names[7] = {"prod empty-wait done", "prod stores done", "prod arrived", "mma full-wait done",
                                   "mma issued+commit", "epi tfull-wait done", "epi stores done"};
    long long t0 = 0;
    for (int i = 0; i < 7 * 64; ++i) if (h[i] && (t0 == 0 || h[i] < t0)) t0 = h[i];
    fprintf(stderr, "[tc trace] m=%lld tiles=%lld grid=%d\n", (long long)m, (long long)tiles, grid);
    for (int r = 0; r < 7; ++r) {
      fprintf(stderr, "  %-22s", names[r]);
      for (int i = 0; i < 32; ++i) if (h[r * 64 + i]) fprintf(stderr, " %6lld", h[r * 64 + i] - t0);
      fprintf(stderr, "\n");
    }
    return check_launch("gemm_rowpanel_tc_kernel");
  }
  CGCN_CUDA(launch_k(tc::gemm_rowpanel_tc_kernel, dim3(grid), dim3(tc::THREADS), tc::RP_SMEM, stream, p));
  return check_launch("gemm_rowpanel_tc_kernel");
}

int gemm_gram_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t m, int ka,
                 int nb, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CGCN_REQUIRE(A && B && C && m >= 1, "cgcn_gemm_gram: bad operand");
  CGCN_REQUIRE(tc_gram_supported(lda, ldb, ka, nb, A, B),
               "cgcn_gemm_gram(tcgen05): needs ka, nb <= 128 and 16-byte aligned rows padded to a multiple of 4 floats");
  if (workspace == nullptr || workspace_bytes < gram_workspace_bytes(m) || !aligned16(workspace)) {
    set_error("cgcn_gemm_gram(tcgen05): workspace %zu < %zu bytes", workspace_bytes, gram_workspace_bytes(m));
    return CGCN_ERR_WORKSPACE;
  }
  static bool attr_set[64] = {};
  if (first_use_on_device(attr_set)) {
    CGCN_CUDA(cudaFuncSetAttribute(tc::gemm_gram_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::GR_SMEM));
  }
  // one CTA per SM (the kernel owns the whole shared memory): a single wave, <= #SM partial tiles
  int64_t rows = (m + sm_count() - 1) / sm_count();
  if (rows < 256) rows = 256;
  rows = (rows + tc::KCH - 1) / tc::KCH * tc::KCH;
  const int parts = static_cast<int>((m + rows - 1) / rows);
  tc::GramTcArgs p{A, lda, B, ldb, m, rows, static_cast<float*>(workspace), ka, nb};
  CGCN_CUDA(launch_k(tc::gemm_gram_tc_kernel, dim3(parts), dim3(tc::THREADS), tc::GR_SMEM, stream, p));
  CGCN_TRY(check_launch("gemm_gram_tc_kernel"));
  gram_finalize_launch(p.partial, parts, tc::TILE * tc::TILE, tc::TILE, ka, nb, C, ldc, accumulate, stream);
  return check_launch("gram_finalize_kernel");
}

}  // namespace cgcn
