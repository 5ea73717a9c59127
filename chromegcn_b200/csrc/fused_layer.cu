// One gated GCN layer as ONE persistent sm_100a kernel: CSR gather-reduce -> tcgen05 3xTF32 contraction -> gate epilogue.
//
// Forward (models/SubLayers.py:43-50 + models/ChromeModels.py:37-42 / 43-46), per 64-row tile of the strand-
// interleaved panel:
//   gather warps   sx_i = sum_{j in row i of bin(A+I)} x_j       (warp per window row, both strands per column index,
//                  software-pipelined: the next row's rowptr / colidx are in flight while this row's neighbours load)
//                  -> global (saved for d W = sx^T (D^-1 dy)), and  A_hat x = sx / deg  split into hi / lo TF32 straight
//                  into the UMMA SWIZZLE_128B K-major shared-memory layout
//   MMA warp       tcgen05.mma kind::tf32, M = 64, N = 128, K = 8: (A_hat x) W as lo*hi + hi*lo + hi*hi against the
//                  resident 128 KB weight image, fp32 accumulator in TMEM (double buffered)
//   epilogue warps TMEM -> shared (thread = row), then 8 lanes per row: + b, tanh, gate dot (3 shuffles), sigmoid,
//                  blend with x, dropout, BatchNorm column partials; z, x', g written once, coalesced
// so the panel is read once (gather) and written three times (sx, z, x') per layer; the unfused path of model.cu
// moves it eight times (SpMM out, GEMM in / out, gate in x2 / out x2).
//
// Backward twin, with the contraction re-associated as  A_hat^T G W^T = (P (D^-1 G)) W^T  so that the gather comes
// first: gather u = P t over t = D^-1 dy_l (written pre-scaled by the previous gate stage), u W_l^T on the tensor
// cores, epilogue dx = u W_l^T + (1-g_l) dh_l, then the whole gate / tanh backward of layer l-1 (dropout mask, gate
// dot, dz, dy, D^-1 scale, column partials for d b, d w_g, d b_g) -- replaces the row-panel contraction, the SpMM and
// gate_bwd_kernel<MID> of the unfused path.
//
// Weight-stationary operand roles.  The contraction is issued TRANSPOSED:  y^T [128 features x 64 rows] = W^T (A_hat x)^T,
// with the 128 x 128 weight matrix (hi and lo TF32 images, 256 TMEM columns, written once per CTA with tcgen05.st) as
// the A operand FROM TENSOR MEMORY and the gathered 64-row tile as the shared-memory B operand (N = 64).  Shared memory
// is then just the tile (hi + lo, 64 KB) + the epilogue's transposition buffer (32 KB): ~97 KB, which leaves the SM
// ~156 KB of L1.  That matters more than anything else in this kernel: every in-flight gather load holds an L1 line,
// and the first version (weight image resident in shared memory, 225 KB, ~28 KB of L1) ran the gather at 0.4 of the
// standalone SpMM's rate for exactly that reason (profiles/r02_fused_v1_*).
#include "common.cuh"
#include "tc_ptx.cuh"
#include "fused_layer.cuh"

namespace cgcn {

namespace fl {
using namespace tc;

constexpr int TM = 64;                         // panel rows per tile = UMMA N
// The E = 4 epilogue warps (warp w <-> TMEM lane quarter w) come first, then the 16 gather warps; the first of those also
// issues the MMAs (no dedicated warp).  20 warps = 5 per scheduler -> 96 registers per thread.
constexpr int E = 4, G_WARPS = 16, THREADS = (E + G_WARPS) * 32;
constexpr int A_CHUNK = TM * 128;              // one k-chunk (32 floats) of the tile: 64 rows x 128 B = 8 KB
constexpr int A_BYTES = 2 * 4 * A_CHUNK;       // hi + lo: 64 KB
constexpr int Y_BYTES = TM * 512;              // fp32 y tile, row major [64 rows][128 features]: 32 KB
constexpr int OFF_Y = A_BYTES, OFF_MISC = OFF_Y + Y_BYTES;
constexpr int OFF_VEC1 = OFF_MISC + 128;       // gate weights (128 floats)
constexpr int SMEM = OFF_VEC1 + 512;           // 98 944 bytes: the 100 KB carve-out, ~156 KB of L1 left
static_assert(SMEM + 1024 <= 100 * 1024, "must fit the 100 KB shared-memory carve-out");
// TMEM columns: W hi 0..127 | W lo 128..255 | accumulator 0: 256..319 | accumulator 1: 320..383
constexpr uint32_t TM_WHI = 0, TM_WLO = 128, TM_ACC = 256, TM_COLS = 512;

// D = F32, A = B = TF32, both K-major, M = 128 (weight rows = output features), N = 64 (tile rows)
__host__ __device__ constexpr uint32_t idesc_m128_n64() {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
}
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// acc += v as two packed fp32x2 adds (FADD2, sm_100): same rounding as four FADDs, half the issue slots
__device__ __forceinline__ void add4_packed(float4& acc, const float4 v) {
  asm("{\n\t"
      ".reg .b64 ra, rb, va, vb;\n\t"
      "mov.b64 ra, {%0, %1};\n\t"
      "mov.b64 rb, {%2, %3};\n\t"
      "mov.b64 va, {%4, %5};\n\t"
      "mov.b64 vb, {%6, %7};\n\t"
      "add.rn.f32x2 ra, ra, va;\n\t"
      "add.rn.f32x2 rb, rb, vb;\n\t"
      "mov.b64 {%0, %1}, ra;\n\t"
      "mov.b64 {%2, %3}, rb;\n\t"
      "}"
      : "+f"(acc.x), "+f"(acc.y), "+f"(acc.z), "+f"(acc.w)
      : "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
}

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
  const uint4 v = lds128(saddr);
  return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

template <int S, int MODE, bool PEER>
__global__ void __launch_bounds__(THREADS, 1) fused_layer_kernel(const Args a) {
  constexpr int EPI_WARPS = E, ISSUE_WARP = E;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = smem_u32(smem_raw);
  const uint32_t sA = base, sY = base + OFF_Y;
  const uint32_t bar_a_full = base + OFF_MISC, bar_a_empty = bar_a_full + 8, bar_tfull = bar_a_full + 16,
                 bar_tempty = bar_a_full + 32, s_tmem_ptr = bar_a_full + 56;
  const uint32_t sVec1 = base + OFF_VEC1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr bool FORWARD = (MODE == FWD || MODE == FWD_STATS);
  constexpr int TG = TM / S;                       // window rows per tile
  constexpr int RPW = TG / G_WARPS;                // window rows per gather warp per tile
  static_assert(RPW >= 1 && 2 * RPW <= 32, "tile / warp split");

  const int r_begin = blockIdx.x * a.rows_per_cta;
  const int r_end = min(r_begin + a.rows_per_cta, a.n);
  const int ntile = r_end > r_begin ? (r_end - r_begin + TG - 1) / TG : 0;

  // ---- set-up that touches no global memory (runs under the previous kernel's tail: programmatic dependent launch)
  if ((base & 1023u) != 0u) __trap();              // SWIZZLE_128B operands need the 1024-byte aligned window start
  if (threadIdx.x == 0) {
    mbar_init(bar_a_full, G_WARPS);
    mbar_init(bar_a_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, 1);
    }
    fence_barrier_init();
  }
  if (warp == ISSUE_WARP) tmem_alloc(s_tmem_ptr, TM_COLS);
  pdl_grid_sync();

  if (threadIdx.x < 128)
    *reinterpret_cast<float*>(smem_raw + OFF_VEC1 + threadIdx.x * 4) =
        ((FORWARD || MODE == BWD_MID) && !a.gate_off) ? __ldg(a.wg + threadIdx.x) : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_raw + OFF_MISC + 56);

  if (warp < 4 && ntile > 0) {
    // The weight operand into tensor memory: thread f of the epilogue warps owns TMEM lane f = output feature f and
    // writes A[f][k] = Bw(f, k) (the weight that multiplies input column k into output column f) for k = 0..127,
    // as hi and lo TF32 images.  W is 64 KB and L2 resident; this runs once per CTA while the gather warps already
    // work on the first tile.  Barrier 3 (epilogue warps + the issuing warp, which joins right before its first MMA)
    // publishes the images.
    const int f = threadIdx.x;
#pragma unroll 1
    for (int kb = 0; kb < 4; ++kb) {
      uint32_t hi[32], lo[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int k = kb * 32 + j;
        const float v = a.w_transposed ? __ldg(a.w + f * 128 + k) : __ldg(a.w + k * 128 + f);
        split_tf32(v, hi[j], lo[j]);
      }
      const uint32_t t = tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + kb * 32;
      tmem_st32(t + TM_WHI, hi);
      tmem_st32(t + TM_WLO, lo);
    }
    tmem_wait_st();
    tc_fence_before();
    named_bar_sync(3, 5 * 32);
    tc_fence_after();
  }

  if (warp >= EPI_WARPS) {
    // =========================================================== gather warps
    // Each warp owns RPW window rows of every tile and walks their neighbour lists as ONE stream of "segments" (<= 32
    // column indices of one row, held one per lane) cut into batches of U neighbours.  Two register sets alternate:
    // while batch i is being summed, batch i+1 -- of the same segment, or the first of the next row / tile -- is already
    // in flight, so the load queue never drains at a row or tile boundary.  Column indices are fetched two segments
    // ahead, row pointers two tiles ahead.  Sums run in CSR order (deterministic).
    const int gw = warp - EPI_WARPS;
    // ---- MMA issue (first gather warp, after it has delivered its own rows of the tile)
    constexpr uint32_t idesc = idesc_m128_n64();
    auto issue_mma = [&](int t) {
      const uint32_t accb = t & 1;
      if (t == 0) {                                // the weight images are in tensor memory (see above)
        named_bar_sync(3, 5 * 32);
        tc_fence_after();
      }
      mbar_wait(bar_tempty + 8 * accb, ((t >> 1) & 1) ^ 1);
      mbar_wait(bar_a_full, t & 1);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t d_tmem = tmem_base + TM_ACC + accb * 64;
#pragma unroll
        for (int kc = 0; kc < 4; ++kc) {
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t k0 = kc * 32 + ks * 8;                 // TMEM column of this k-step inside a weight image
            const uint64_t dxh = make_desc(sA + kc * A_CHUNK + ks * 32, 16, 1024);
            const uint64_t dxl = make_desc(sA + 4 * A_CHUNK + kc * A_CHUNK + ks * 32, 16, 1024);
            umma_tf32_ts(d_tmem, tmem_base + TM_WLO + k0, dxh, idesc, (kc | ks) != 0);      // small terms first
            umma_tf32_ts(d_tmem, tmem_base + TM_WHI + k0, dxl, idesc, 1);
            umma_tf32_ts(d_tmem, tmem_base + TM_WHI + k0, dxh, idesc, 1);
          }
        }
        umma_commit(bar_a_empty);                  // tile buffer free once these MMAs retire
        umma_commit(bar_tfull + 8 * accb);         // accumulator complete
      }
      __syncwarp();
    };
    // one finished panel row (lane owns columns 4 lane .. 4 lane + 3) into the tile buffer as hi / lo TF32
    auto put_row = [&](int pr, const float4 v) {
      uint4 hi, lo;
      split4(v, hi, lo);
      const uint32_t off = (lane >> 3) * A_CHUNK + (pr >> 3) * 1024 + (pr & 7) * 128 + (((lane & 7) ^ (pr & 7)) << 4);
      sts128(sA + off, hi);
      sts128(sA + 4 * A_CHUNK + off, lo);
    };
    auto deliver = [&](int t) {                    // this warp's rows of tile t are in the buffer
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a_full);
      if (warp == ISSUE_WARP) issue_mma(t);
    };

    constexpr int U = (S == 2) ? 3 : 6;
    const int nrow = ntile * RPW;                  // rows this warp visits; rows beyond r_end read as empty
    auto load_ptrs = [&](int t) -> int {           // lane 2h + e holds rowptr[row_h + e] of tile t
      int v = 0;
      if (lane < 2 * RPW && t < ntile) {
        const int row = r_begin + t * TG + gw + G_WARPS * (lane >> 1);
        if (row < r_end) v = __ldg(a.rowptr + row + (lane & 1));
      }
      return v;
    };
    // ---- segment iterator (producer side of the descriptors)
    int p0 = load_ptrs(0), p1 = load_ptrs(1), p2 = load_ptrs(2);
    int it_q = -1, it_off = 0, it_end = 0;
    auto next_seg = [&](int& cols, int& cnt_last) {        // cnt_last = cnt | (last segment of its row ? 64 : 0)
      if (it_off >= it_end) {                              // next row
        ++it_q;
        if (it_q > 0 && (it_q % RPW) == 0) {               // next tile: shift the row-pointer registers
          p0 = p1;
          p1 = p2;
          p2 = load_ptrs(it_q / RPW + 2);
        }
        const int h = it_q % RPW;
        it_off = __shfl_sync(0xffffffffu, p0, 2 * h);
        it_end = __shfl_sync(0xffffffffu, p0, 2 * h + 1);
        if (it_q >= nrow) it_off = it_end = 0;
      }
      int cnt = it_end - it_off;
      cnt = cnt < 0 ? 0 : (cnt > 32 ? 32 : cnt);
      cols = (lane < cnt) ? __ldg(a.colidx + it_off + lane) : 0;
      it_off += 32;
      cnt_last = cnt | ((it_off >= it_end) ? 64 : 0);
    };
    // Loads are unconditional: slots past the end of the segment re-read its last neighbour (an L1 hit) and are simply
    // not summed -- a predicated load would have to preserve the register set's previous contents (moves per load).
    const float* const gbase = a.gsrc + lane * 4;
    auto issue = [&](float4 (&v)[U][S], int cols, int k0, int cnt) {
      const int last = cnt > 0 ? cnt - 1 : 0;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = __shfl_sync(0xffffffffu, cols, min(k0 + u, last));
        const float* p;
        if constexpr (PEER) {                      // owner of global row c: NVLink load from its exchange buffer
          p = peer_row(a.peer, c, S * 128) + lane * 4;
        } else {
          p = gbase + static_cast<size_t>(c) * (S * 128);
        }
#pragma unroll
        for (int s = 0; s < S; ++s) v[u][s] = ldg4(p + s * 128);
      }
    };
    auto consume = [&](const float4 (&v)[U][S], int k0, int cnt, float4 (&acc)[S]) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (k0 + u < cnt) {
#pragma unroll
          for (int s = 0; s < S; ++s) add4_packed(acc[s], v[u][s]);
        }
      }
    };
    float4 X[U][S], Y[U][S];
    int c_cols, c_cl, n_cols, n_cl, nn_cols, nn_cl;        // current / next / next-next segment
    next_seg(c_cols, c_cl);
    next_seg(n_cols, n_cl);
    next_seg(nn_cols, nn_cl);
    issue(X, c_cols, 0, c_cl & 63);
    int parity = 0, deg = 0;
    float4 acc[S];
#pragma unroll
    for (int s = 0; s < S; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q = 0; q < nrow;) {
      const int cnt = c_cl & 63;
      const int nb = cnt > 0 ? (cnt + U - 1) / U : 1;
      for (int b = 0; b < nb; ++b) {
        const int k0 = b * U;
        const bool same = (b + 1 < nb);
        const int i_cols = same ? c_cols : n_cols, i_k0 = same ? k0 + U : 0, i_cnt = same ? cnt : (n_cl & 63);
        if (parity == 0) {
          issue(Y, i_cols, i_k0, i_cnt);
          consume(X, k0, cnt, acc);
        } else {
          issue(X, i_cols, i_k0, i_cnt);
          consume(Y, k0, cnt, acc);
        }
        parity ^= 1;
      }
      deg += cnt;
      if (c_cl & 64) {                             // the row is complete: scale, save, split, deliver
        const int t = q / RPW, h = q % RPW;
        const int lr = gw + G_WARPS * h;           // window row inside the tile
        const int row = r_begin + t * TG + lr;
        float scale = 1.0f;
        if (FORWARD) {
          scale = deg > 0 ? __fdiv_rn(1.0f, static_cast<float>(deg)) : 1.0f;
          if (row < r_end) {
#pragma unroll
            for (int s = 0; s < S; ++s) st4(a.sx + (static_cast<size_t>(row) * S + s) * 128 + lane * 4, acc[s]);
          }
        }
        if (h == 0) mbar_wait(bar_a_empty, (t & 1) ^ 1);        // the MMAs of the previous tile have read the tile buffer
#pragma unroll
        for (int s = 0; s < S; ++s) {
          put_row(lr * S + s, make_float4(acc[s].x * scale, acc[s].y * scale, acc[s].z * scale, acc[s].w * scale));
          acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        deg = 0;
        if (h == RPW - 1) deliver(t);
        ++q;
      }
      c_cols = n_cols;
      c_cl = n_cl;
      n_cols = nn_cols;
      n_cl = nn_cl;
      next_seg(nn_cols, nn_cl);
    }
  } else {
    // =========================================================== epilogue warps
    // Phase A (thread = output feature: the accumulator is y^T, TMEM lane f = feature f, column r = tile row r):
    // TMEM -> + bias -> row-major shared y tile (one conflict-free 128-byte store per row per warp).
    // Phase B (LPR lanes per row, RPI rows per warp step; lane q owns the float4 column groups cc * CSTRIDE + 4 q):
    // everything else, on TM / E rows per epilogue warp: 8 lanes per row, 16 values per lane per step.
    constexpr int LPR = 8, RPI = 32 / LPR, CPL = 32 / LPR, CSTRIDE = LPR * 4;
    constexpr int ROWS_W = TM / E, ITERS = ROWS_W / RPI;
    static_assert(CPL * CSTRIDE == 128 && ITERS >= 1 && ROWS_W % 2 == 0 && E * RPI == 16, "epilogue split");
    const int sub = lane / LPR, q = lane % LPR;
    constexpr int NST = (MODE == FWD_STATS || MODE == BWD_MID) ? CPL : 1;
    float4 st0[NST], st1[NST];                     // FWD_STATS: sum / sum of squares of relu(x') ; BWD_MID: d b / d w_g
    float st2 = 0.f;                               // BWD_MID: d b_g
#pragma unroll
    for (int i = 0; i < NST; ++i) st0[i] = st1[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float bg = (FORWARD && !a.gate_off) ? __ldg(a.bg) : 0.f;
    float bias_f = 0.f;                            // threadIdx.x = this thread's feature
    if (FORWARD && threadIdx.x < 128) bias_f = __ldg(a.bias + threadIdx.x);
    const int64_t prow_end = static_cast<int64_t>(r_end) * S;

    for (int t = 0; t < ntile; ++t) {
      const uint32_t accb = t & 1;
      if (warp < 4) {
        mbar_wait(bar_tfull + 8 * accb, (t >> 1) & 1);
        tc_fence_after();
      }
      if (warp < 4) {                              // the four warps that can read the accumulator's 128 lanes
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          uint32_t r[32];
          tmem_ld32(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + TM_ACC + accb * 64 + half * 32, r);
          float* yrow = reinterpret_cast<float*>(smem_raw + OFF_Y) + (half * 32) * 128 + threadIdx.x;
#pragma unroll
          for (int j = 0; j < 32; ++j) yrow[j * 128] = __uint_as_float(r[j]) + bias_f;
        }
        tc_fence_before();
      }
      named_bar_sync(2, E * 32);                   // the y tile is complete (every warp wrote 32 features of every row)
      if (threadIdx.x == 0) mbar_arrive(bar_tempty + 8 * accb);            // accumulator released before the heavy phase

      const int64_t tile_prow0 = (static_cast<int64_t>(r_begin) + static_cast<int64_t>(t) * TG) * S;
#pragma unroll 1
      for (int it = 0; it < ITERS; ++it) {
        const int pr = ROWS_W * warp + it * RPI + sub;
        const int64_t grow = tile_prow0 + pr;      // panel row (local)
        const bool valid = grow < prow_end;
        const size_t gofs = static_cast<size_t>(grow) * 128 + 4 * q;
        {
          // L1 prefetch of the NEXT step's streamed operands (next 4 rows of this warp; the first 4 of the next tile
          // after the last step): the epilogue warps have no registers to spare for a software pipeline, and without
          // this every step starts with a full L2 / DRAM round trip (3 panels in the backward mode).
          const int64_t nrow_p = (it < ITERS - 1) ? grow + RPI : grow + (TM - (ITERS - 1) * RPI);
          if (nrow_p < prow_end) {
            const size_t nofs = static_cast<size_t>(nrow_p) * 128 + 4 * q;
#pragma unroll
            for (int cc = 0; cc < CPL; ++cc) {
              if constexpr (FORWARD) {
                prefetch_l1(a.xin + nofs + cc * CSTRIDE);
              } else {
                prefetch_l1(a.dxd_in + nofs + cc * CSTRIDE);
                if constexpr (MODE == BWD_MID) {
                  prefetch_l1(a.z_prev + nofs + cc * CSTRIDE);
                  prefetch_l1(a.x_prev + nofs + cc * CSTRIDE);
                }
              }
            }
          }
        }
        float4 y[CPL];
#pragma unroll
        for (int cc = 0; cc < CPL; ++cc) y[cc] = lds_f4(sY + pr * 512 + (cc * CSTRIDE + 4 * q) * 4);

        if constexpr (FORWARD) {
          float4 xv[CPL];
#pragma unroll
          for (int cc = 0; cc < CPL; ++cc) xv[cc] = valid ? ldg4(a.xin + gofs + cc * CSTRIDE) : make_float4(0.f, 0.f, 0.f, 0.f);
          float dot = 0.f;
#pragma unroll
          for (int cc = 0; cc < CPL; ++cc) {
            const float4 w = lds_f4(sVec1 + (cc * CSTRIDE + 4 * q) * 4);
            y[cc] = make_float4(tanhf(y[cc].x), tanhf(y[cc].y), tanhf(y[cc].z), tanhf(y[cc].w));
            dot += y[cc].x * w.x + y[cc].y * w.y + y[cc].z * w.z + y[cc].w * w.w;
          }
          dot += __shfl_xor_sync(0xffffffffu, dot, 1);
          dot += __shfl_xor_sync(0xffffffffu, dot, 2);
          dot += __shfl_xor_sync(0xffffffffu, dot, 4);
          const float g = a.gate_off ? 1.0f : sigmoidf_(dot + bg);
          const float omg = 1.0f - g;
          if (valid) {
            if (q == 0) a.g[grow] = g;
#pragma unroll
            for (int cc = 0; cc < CPL; ++cc) {
              float4 h = make_float4(omg * xv[cc].x + g * y[cc].x, omg * xv[cc].y + g * y[cc].y, omg * xv[cc].z + g * y[cc].z,
                                     omg * xv[cc].w + g * y[cc].w);
              if (a.drop.enabled) {
                const float4 m = dropout_mult4(a.drop, (gofs + cc * CSTRIDE) >> 2);
                h = make_float4(h.x * m.x, h.y * m.y, h.z * m.z, h.w * m.w);
              }
              st4(a.z + gofs + cc * CSTRIDE, y[cc]);
              st4(a.xo + gofs + cc * CSTRIDE, h);
              if constexpr (MODE == FWD_STATS) {
                const float4 rl = make_float4(fmaxf(h.x, 0.f), fmaxf(h.y, 0.f), fmaxf(h.z, 0.f), fmaxf(h.w, 0.f));
                st0[cc].x += rl.x; st0[cc].y += rl.y; st0[cc].z += rl.z; st0[cc].w += rl.w;
                st1[cc].x += rl.x * rl.x; st1[cc].y += rl.y * rl.y; st1[cc].z += rl.z * rl.z; st1[cc].w += rl.w * rl.w;
              }
            }
          }
        } else if constexpr (MODE == BWD_INPUT) {
          if (valid) {
#pragma unroll
            for (int cc = 0; cc < CPL; ++cc) {
              const float4 e = ldg4(a.dxd_in + gofs + cc * CSTRIDE);
              st4(a.dx_out + gofs + cc * CSTRIDE, make_float4(y[cc].x + e.x, y[cc].y + e.y, y[cc].z + e.z, y[cc].w + e.w));
            }
          }
        } else {                                   // BWD_MID: gate / tanh backward of layer l-1 on dx = u W^T + (1-g_l) dh_l
          float4 zv[CPL];
          float part = 0.f;
          // scalar operands of the row first: their latency overlaps the panel loads instead of following the reduction
          float g = 1.0f;
          int deg = 1;
          if (valid) {
            if (!a.gate_off) g = __ldg(a.g_prev + grow);
            const int wr = static_cast<int>(grow / S);
            deg = __ldg(a.rowptr + wr + 1) - __ldg(a.rowptr + wr);
          }
#pragma unroll
          for (int cc = 0; cc < CPL; ++cc) {
            float4 e = make_float4(0.f, 0.f, 0.f, 0.f), xv = e;
            zv[cc] = e;
            if (valid) {
              e = ld4(a.dxd_in + gofs + cc * CSTRIDE);  // may alias dxd_out: plain load, same lane reads then writes
              zv[cc] = ldg4(a.z_prev + gofs + cc * CSTRIDE);
              xv = ldg4(a.x_prev + gofs + cc * CSTRIDE);
            }
            float4 d = make_float4(y[cc].x + e.x, y[cc].y + e.y, y[cc].z + e.z, y[cc].w + e.w);
            if (a.drop.enabled) {
              const float4 m = dropout_mult4(a.drop, (gofs + cc * CSTRIDE) >> 2);
              d = make_float4(d.x * m.x, d.y * m.y, d.z * m.z, d.w * m.w);
            }
            y[cc] = d;
            part += d.x * (zv[cc].x - xv.x) + d.y * (zv[cc].y - xv.y) + d.z * (zv[cc].z - xv.z) + d.w * (zv[cc].w - xv.w);
          }
          part += __shfl_xor_sync(0xffffffffu, part, 1);
          part += __shfl_xor_sync(0xffffffffu, part, 2);
          part += __shfl_xor_sync(0xffffffffu, part, 4);
          if (valid) {
            const float dgp = a.gate_off ? 0.0f : part * g * (1.0f - g);
            const float omg = 1.0f - g;
            const float inv = deg > 0 ? __fdiv_rn(1.0f, static_cast<float>(deg)) : 0.0f;
#pragma unroll
            for (int cc = 0; cc < CPL; ++cc) {
              const float4 w = lds_f4(sVec1 + (cc * CSTRIDE + 4 * q) * 4);
              const float4 dz = make_float4(g * y[cc].x + dgp * w.x, g * y[cc].y + dgp * w.y, g * y[cc].z + dgp * w.z,
                                            g * y[cc].w + dgp * w.w);
              const float4 dy = make_float4(dz.x * (1.0f - zv[cc].x * zv[cc].x), dz.y * (1.0f - zv[cc].y * zv[cc].y),
                                            dz.z * (1.0f - zv[cc].z * zv[cc].z), dz.w * (1.0f - zv[cc].w * zv[cc].w));
              st4(a.dys_out + gofs + cc * CSTRIDE, make_float4(dy.x * inv, dy.y * inv, dy.z * inv, dy.w * inv));
              if (a.dxd_out != nullptr)
                st4(a.dxd_out + gofs + cc * CSTRIDE, make_float4(omg * y[cc].x, omg * y[cc].y, omg * y[cc].z, omg * y[cc].w));
              st0[cc].x += dy.x; st0[cc].y += dy.y; st0[cc].z += dy.z; st0[cc].w += dy.w;
              st1[cc].x += dgp * zv[cc].x; st1[cc].y += dgp * zv[cc].y; st1[cc].z += dgp * zv[cc].z; st1[cc].w += dgp * zv[cc].w;
            }
            if (q == 0) st2 += dgp;
          }
        }
      }
      named_bar_sync(2, E * 32);                   // everybody is done reading the y tile
    }

    // ---- column partials of this CTA, fixed order: (warp, row slot) pairs summed per column by 128 threads
    if constexpr (MODE == FWD_STATS || MODE == BWD_MID) {
      float* red = reinterpret_cast<float*>(smem_raw + OFF_Y);      // [2][16 slots][128 cols] (+ 16 floats)
      const int slot = warp * RPI + sub;           // 16 slots; a slot always sees the same strand (slot & 1)
#pragma unroll
      for (int cc = 0; cc < CPL; ++cc) {
        *reinterpret_cast<float4*>(red + (0 * 16 + slot) * 128 + cc * CSTRIDE + 4 * q) = st0[cc];
        *reinterpret_cast<float4*>(red + (1 * 16 + slot) * 128 + cc * CSTRIDE + 4 * q) = st1[cc];
      }
      if (MODE == BWD_MID && q == 0) red[2 * 16 * 128 + slot] = st2;
      named_bar_sync(1, E * 32);
      const int c = threadIdx.x;                   // 0..127: one column each (the other epilogue threads are done)
      if (c < 128) {
      if constexpr (MODE == FWD_STATS) {
        // slot's strand: panel rows alternate strands and a slot always sees the same parity (S == 2: sub & 1)
        float* dst = a.partial + static_cast<size_t>(blockIdx.x) * (2 * S * 128);
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float t0 = 0.f, t1 = 0.f;
          for (int sl = 0; sl < 16; ++sl) {
            if (S == 1 || (sl & 1) == s) {
              t0 += red[(0 * 16 + sl) * 128 + c];
              t1 += red[(1 * 16 + sl) * 128 + c];
            }
          }
          dst[(0 * S + s) * 128 + c] = t0;
          dst[(1 * S + s) * 128 + c] = t1;
        }
      } else {
        float* dst = a.partial + static_cast<size_t>(blockIdx.x) * (2 * 128 + 4);
        float t0 = 0.f, t1 = 0.f;
        for (int sl = 0; sl < 16; ++sl) {
          t0 += red[(0 * 16 + sl) * 128 + c];
          t1 += red[(1 * 16 + sl) * 128 + c];
        }
        dst[c] = t0;
        dst[128 + c] = t1;
        if (c < 4) {
          float t2 = 0.f;
          if (c == 0)
            for (int sl = 0; sl < 16; ++sl) t2 += red[2 * 16 * 128 + sl];
          dst[256 + c] = t2;
        }
      }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == ISSUE_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TM_COLS);
  }
}

}  // namespace fl

// ------------------------------------------------------------------ host side
int fused_layer_grid(int n, int S, int* rows_per_cta_out) {
  const int tg = fl::TM / S;
  const int tiles = (n + tg - 1) / tg;
  int grid = tiles < sm_count() ? tiles : sm_count();
  if (grid < 1) grid = 1;
  int rows = (n + grid - 1) / grid;
  rows = (rows + 3) / 4 * 4;
  if (rows < 4) rows = 4;
  grid = (n + rows - 1) / rows;
  if (grid < 1) grid = 1;
  if (rows_per_cta_out) *rows_per_cta_out = rows;
  return grid;
}

bool fused_layer_supported(int d, const cgcn_graph* g) { return d == 128 && g != nullptr && g->vals == nullptr; }

template <int S, int MODE, bool PEER>
static int launch_kernel(const fl::Args& a, int grid, cudaStream_t stream) {
  static bool attr_set[64] = {};
  if (first_use_on_device(attr_set))
    CGCN_CUDA(cudaFuncSetAttribute(fl::fused_layer_kernel<S, MODE, PEER>, cudaFuncAttributeMaxDynamicSharedMemorySize, fl::SMEM));
  CGCN_CUDA(launch_k(fl::fused_layer_kernel<S, MODE, PEER>, dim3(grid), dim3(fl::THREADS), fl::SMEM, stream, a));
  return check_launch("fused_layer_kernel");
}

template <int S, bool PEER>
static int launch_mode(const fl::Args& a, int mode, int grid, cudaStream_t stream) {
  switch (mode) {
    case fl::FWD: return launch_kernel<S, fl::FWD, PEER>(a, grid, stream);
    case fl::FWD_STATS: return launch_kernel<S, fl::FWD_STATS, PEER>(a, grid, stream);
    case fl::BWD_MID: return launch_kernel<S, fl::BWD_MID, PEER>(a, grid, stream);
    case fl::BWD_INPUT: return launch_kernel<S, fl::BWD_INPUT, PEER>(a, grid, stream);
  }
  set_error("fused layer: unsupported strands=%d mode=%d", S, mode);
  return CGCN_ERR_INVALID;
}

int fused_layer_launch(fl::Args a, int S, int mode, int* grid_out, cudaStream_t stream) {
  CGCN_REQUIRE(a.rowptr && a.colidx && (a.gsrc || a.peer.world > 0) && a.w, "fused layer: null graph / panel / weight");
  CGCN_REQUIRE(S == 1 || S == 2, "fused layer: strands=%d", S);
  int rows = 0;
  const int grid = fused_layer_grid(a.n, S, &rows);
  a.rows_per_cta = rows;
  if (grid_out) *grid_out = grid;
  if (a.n <= 0) return CGCN_OK;
  const bool peer = a.peer.world > 0;
  if (peer) a.gsrc = a.peer.base[0];
  if (S == 1) return peer ? launch_mode<1, true>(a, mode, grid, stream) : launch_mode<1, false>(a, mode, grid, stream);
  return peer ? launch_mode<2, true>(a, mode, grid, stream) : launch_mode<2, false>(a, mode, grid, stream);
}

}  // namespace cgcn
