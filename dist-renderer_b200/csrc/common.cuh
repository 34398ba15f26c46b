// Shared device/host helpers for libdist_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/dist_b200.h"

namespace dist {

void set_error(const char* fmt, ...);
int num_sms();
void count_launch();   // every kernel launch of the library is counted (dist_launch_count)

#define DIST_CHECK_CUDA(expr)                                                                   \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      ::dist::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DIST_E_CUDA;                                                                       \
    }                                                                                           \
  } while (0)

#define DIST_REQUIRE(cond, ...)                 \
  do {                                          \
    if (!(cond)) {                              \
      ::dist::set_error(__VA_ARGS__);           \
      return DIST_E_INVALID;                    \
    }                                           \
  } while (0)

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Device copy of the network description (passed by value as a kernel parameter).
struct NetDev {
  int n_layers, latent_in, use_tanh;
  int K[DIST_MAX_LAYERS], N[DIST_MAX_LAYERS];
  const float* Wt[DIST_MAX_LAYERS];
  const float* W[DIST_MAX_LAYERS];
  const float* bias[DIST_MAX_LAYERS];
  int n_codes;   // > 1: bias[0] / bias[latent_in] are per-code tables [n_codes][Np4] (dist_net_t.n_codes)
};

int make_netdev(const dist_net_t* net, NetDev* out);

// engines (mlp_simt.cu / mlp_tc.cu).  mode: 0 forward, 1 input-gradient, 2 backward replay
struct MlpArgs {
  const float* points;      // [n][3]
  int64_t n_host;
  const int32_t* n_dev;
  float clamp_dist;         // <= 0: no clamp
  float* sdf;               // [n] or null
  float* grad;              // [n][3] or null (modes 1,2: coef * dsdf/dxyz)
  const float* coef;        // [n] or null (=1)
  const uint8_t* use_clamp; // [n] or null (= clamp_dist > 0 for every row)
  float* acc0;              // [N0] or null
  float* accl;              // [Nl] or null
  int64_t* rows_evaluated;  // optional counter (+= n)
  // optional second row segment: rows [seg2_offset, seg2_offset + n2) of the same arrays (n2 from *n2_dev when set, else
  // n2_host, which is then the capacity); seg2_offset is a multiple of 128 and >= the capacity of the first segment
  int64_t n2_host;
  const int32_t* n2_dev;
  int64_t seg2_offset;
  // two-tier precision of forward launches on the tensor-core engine (mlp_tc.cu); 0 / null: full precision everywhere
  int screen_seg1;          // tiles of the first segment are evaluated with one fp16 pass first, the second with three
  float screen_thresh;      // one-pass values stand where every row of the 64-row half-tile has |sdf| > screen_thresh
  uint8_t* seg_approx;      // [rows / 64] out: 1 = this half-tile's sdf are one-pass values
  unsigned long long* tile_counters;  // optional [2]: tile programs evaluated with one / with three passes
  // ReLU-mask cache of the tensor-core engine (mlp_tc.cu): a forward launch (mode 0) records the sign bits of every hidden
  // layer for the rows it evaluates at full precision in its first sweep, at slots mask_base + row index (of segment 2
  // when segment 1 is screened, of the only segment otherwise); mode 3 replays the transposed chain from them.
  uint32_t* mask_buf;       // [16 * (n_layers - 1)][mask_cap] (one word per hidden layer and 32-feature block) or null
  int64_t mask_cap;
  int64_t mask_base_host;   // used when mask_base_dev is null
  const int32_t* mask_base_dev;
  const int32_t* slots;     // mode 3: [n] mask slot per row (-1: row contributes nothing)
  const float* sdf_in;      // mode 3: [n] recorded decoder output per row
  // several latent codes (NetDev.n_codes > 1): row r uses code row_code[r] / code_div.  The launch sites pass an array they
  // already have, aligned with the rows (an active list of pixels, pixel * DIST_MAX_BUFFER + record, ...), and the divisor
  // that maps its entries to the view; accumulators acc0 / accl are then [n_codes][N].  Unused with one code.
  const int32_t* row_code;
  int32_t code_div;
};
int mlp_simt_launch(const NetDev& net, int mode, const MlpArgs& a, cudaStream_t stream);
int mlp_tc_launch(const dist_net_t* net, const NetDev& nd, int mode, const MlpArgs& a, cudaStream_t stream);

// engine dispatch; brackets the launch with CUDA events while dist_profile_begin() is active (abi.cu)
int mlp_launch(const dist_net_t* net, const NetDev& nd, int engine, int mode, const MlpArgs& a, cudaStream_t stream);

}  // namespace dist
