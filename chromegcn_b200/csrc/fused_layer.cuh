// Argument block and launcher of the fused GCN layer kernels (fused_layer.cu), shared with model.cu.
#pragma once
#include "common.cuh"

namespace cgcn {
namespace fl {

enum Mode { FWD = 0, FWD_STATS = 1, BWD_MID = 2, BWD_INPUT = 3 };

struct Args {
  const int32_t* rowptr;
  const int32_t* colidx;
  int n;                       // local window rows
  int rows_per_cta;            // window rows per CTA (contiguous range)
  const float* gsrc;           // panel the gather reads, indexed by column index: [*][S][128]
  const float* w;              // the 128 x 128 weight matrix (row major) ...
  int w_transposed;            // 0: y = u W (W is [k][n]) ; 1: y = u W^T (W is [n][k])
  // ---- forward
  const float* xin;            // layer input, local rows [n][S][128]
  const float* bias;           // [128]
  const float* wg;             // [128]  gate weights (forward: this layer; backward: layer l-1)
  const float* bg;             // [1]
  float* sx;                   // [n][S][128] un-normalised neighbour sums (saved for the weight gradient)
  float* z;                    // [n][S][128] tanh
  float* xo;                   // [n][S][128] layer output
  float* g;                    // [n][S]
  float* partial;              // FWD_STATS: [grid][2*S*128] ; BWD_MID: [grid][2*128+4]
  int gate_off;
  DropoutCfg drop;             // forward: this layer's output site ; backward: layer l-1's output site
  // ---- backward
  const float* dxd_in;         // (1-g_l) dh_l, local rows
  const float* z_prev;         // layer l-1: tanh output
  const float* x_prev;         // layer l-1: input
  const float* g_prev;         // layer l-1: gate [n][S]
  float* dys_out;              // D^-1 dy_{l-1}
  float* dxd_out;              // (1-g_{l-1}) dh_{l-1} or NULL (may alias dxd_in)
  float* dx_out;               // BWD_INPUT: d loss / d x_in
  // ---- peer gather (one graph row-partitioned over the GPUs of an NVLink box): the gathered panel lives in the ranks'
  // exchange buffers (cgcn_peer_panel); rank r owns global rows [peer_begin[r], peer_begin[r+1]) at peer_base[r].
  // peer_world == 0: plain gather from gsrc.
  int peer_world;
  int peer_begin[CGCN_MAX_PEERS + 1];
  const float* peer_base[CGCN_MAX_PEERS];
};

}  // namespace fl

bool fused_layer_supported(int d, const cgcn_graph* g);
int fused_layer_grid(int n, int S, int* rows_per_cta_out);
int fused_layer_launch(fl::Args a, int S, int mode, int* grid_out, cudaStream_t stream);
int fused_layer_set_peer(fl::Args* a, const cgcn_peer_panel* pp, int n_local);

}  // namespace cgcn
