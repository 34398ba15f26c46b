// fp32 FFMA engine for the folded DeepSDF decoder (DIST_ENGINE_SIMT).
//
// One CTA owns a tile of TM=64 decoder rows and carries it through every layer with the activations resident in
// shared memory (never written to HBM); weights stream L2 -> smem through a 3-stage cp.async ring.  The same tile
// code runs the transposed chain for input-gradients / backward replay, with the ReLU sign bits of the forward pass
// kept as bitmasks in shared memory.  This engine is exact fp32 (sequential FFMA accumulation): it is the numerical
// anchor the tensor-core engine (mlp_tc.cu) is checked against at sizes the CPU oracle cannot reach, and the engine
// used for network shapes the tensor path does not cover.
//
// Replaces: Decoder.inference (core/graph/deep_sdf_decoder.py:80-111), decode_sdf / decode_sdf_gradient
// (core/utils/decoder_utils.py:53-92) and the autograd backward through them.
#include <cuda_runtime.h>
#include "common.cuh"

namespace dist {
namespace {

constexpr int TM = 64;       // rows per tile
constexpr int NT = 256;      // threads per CTA
constexpr int HMAX = DIST_MAX_WIDTH;
constexpr int KC = 8;        // weight rows per pipeline stage
constexpr int NSTAGE = 3;
constexpr int MAXH_GRAD = 10;  // hidden layers whose ReLU masks fit in smem for the gradient modes

struct Smem {
  float act[HMAX * TM];               // act[k][row]
  float wst[NSTAGE][KC * HMAX];
  float xyz[TM * 3];
  float dxyz[TM * 3];
  float rowt[TM];                     // tanh output per row
  float rowt1[TM];                    // inner tanh (use_tanh) per row
  float rowd[TM];                     // d loss / d last pre-activation per row
};
constexpr size_t kSmemFwd = sizeof(Smem);
constexpr size_t kSmemGrad = sizeof(Smem) + size_t(MAXH_GRAD) * TM * 64;
constexpr size_t kSmemCodes = TM * sizeof(int);   // several latent codes: the tile's row codes, behind everything else

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// acc[r][j*4+e] += sum_k act[k][rg*16+r] * Wg[k][half*256 + j*128 + lane*4 + e],  k < Kp8
__device__ __forceinline__ void gemm_tile(Smem& sm, const float* __restrict__ Wg, int Kp8, int ldw,
                                          float (&acc)[16][8], int tid) {
  const int rg = tid >> 6, half = (tid >> 5) & 1, lane = tid & 31;
  const int c0 = half * 256 + lane * 4, c1 = c0 + 128;
  const bool has0 = c0 < ldw, has1 = c1 < ldw;
#pragma unroll
  for (int r = 0; r < 16; ++r)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
  const int nst = Kp8 / KC;
  const int f4_per_stage = KC * ldw / 4;
  auto issue = [&](int s) {
    if (s < nst) {
      const float4* src = reinterpret_cast<const float4*>(Wg + (size_t)s * KC * ldw);
      float4* dst = reinterpret_cast<float4*>(sm.wst[s % NSTAGE]);
      for (int i = tid; i < f4_per_stage; i += NT) cp_async16(dst + i, src + i);
    }
    cp_async_commit();
  };
  for (int s = 0; s < NSTAGE - 1; ++s) issue(s);
  for (int s = 0; s < nst; ++s) {
    cp_async_wait<NSTAGE - 2>();
    __syncthreads();
    issue(s + NSTAGE - 1);
    const float* w = sm.wst[s % NSTAGE];
    const float* a = sm.act + (size_t)s * KC * TM + rg * 16;
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) {
      float av[16];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float4 t = *reinterpret_cast<const float4*>(a + kk * TM + q * 4);
        av[q * 4 + 0] = t.x; av[q * 4 + 1] = t.y; av[q * 4 + 2] = t.z; av[q * 4 + 3] = t.w;
      }
      if (has0) {
        float4 t = *reinterpret_cast<const float4*>(w + kk * ldw + c0);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          acc[r][0] = fmaf(av[r], t.x, acc[r][0]); acc[r][1] = fmaf(av[r], t.y, acc[r][1]);
          acc[r][2] = fmaf(av[r], t.z, acc[r][2]); acc[r][3] = fmaf(av[r], t.w, acc[r][3]);
        }
      }
      if (has1) {
        float4 t = *reinterpret_cast<const float4*>(w + kk * ldw + c1);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          acc[r][4] = fmaf(av[r], t.x, acc[r][4]); acc[r][5] = fmaf(av[r], t.y, acc[r][5]);
          acc[r][6] = fmaf(av[r], t.z, acc[r][6]); acc[r][7] = fmaf(av[r], t.w, acc[r][7]);
        }
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();  // every thread is done reading act / wst
}

__device__ __forceinline__ int col_of(int tid, int c) {
  const int half = (tid >> 5) & 1, lane = tid & 31;
  return half * 256 + (c >> 2) * 128 + lane * 4 + (c & 3);
}

// store the thread's 16x8 values as act[col][rg*16 + r]
__device__ __forceinline__ void store_cols(Smem& sm, const float (&v)[16][8], int tid, int ncols_store) {
  const int rg = tid >> 6;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int col = col_of(tid, c);
    if (col < ncols_store) {
      float* dst = sm.act + (size_t)col * TM + rg * 16;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        *reinterpret_cast<float4*>(dst + q * 4) = make_float4(v[q * 4][c], v[q * 4 + 1][c], v[q * 4 + 2][c], v[q * 4 + 3][c]);
    }
  }
}

__device__ __forceinline__ void zero_rows(Smem& sm, int k_begin, int k_end, int tid) {
  for (int i = k_begin * TM + tid; i < k_end * TM; i += NT) sm.act[i] = 0.f;
}

// MODE: 0 forward, 1 input gradient, 2 backward replay (adds coef / accumulators).
// MC: several latent codes (net.n_codes > 1): per-row folded biases of layer 0 and the latent_in layer, per-code row sums.
template <int MODE, bool MC>
__global__ void __launch_bounds__(NT, 1) mlp_simt_kernel(NetDev net, MlpArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  unsigned char* masks = smem_raw + sizeof(Smem);  // [layer][row][64] (gradient modes)
  int* codes = reinterpret_cast<int*>(smem_raw + (MODE == 0 ? kSmemFwd : kSmemGrad));   // [TM] (MC)
  const int tid = threadIdx.x;
  const int rg = tid >> 6;
  const int64_t n = a.n_dev ? (int64_t)*a.n_dev : a.n_host;
  if (blockIdx.x == 0 && tid == 0 && a.rows_evaluated && n > 0)
    atomicAdd(reinterpret_cast<unsigned long long*>(a.rows_evaluated), (unsigned long long)n);
  const int L = net.n_layers;
  const int last = L - 1;
  const bool clampd = a.clamp_dist > 0.f;
  float acc[16][8];

  for (int64_t tile = blockIdx.x; tile * TM < n; tile += gridDim.x) {
    const int64_t row0 = tile * TM;
    const int nvalid = (int)min((int64_t)TM, n - row0);
    __syncthreads();
    // ---- stage inputs
    if (tid < TM * 3) {
      const int r = tid / 3;
      float v = (r < nvalid) ? a.points[(row0 + r) * 3 + (tid % 3)] : 0.f;
      sm.xyz[tid] = v;
      sm.dxyz[tid] = 0.f;
      sm.act[(tid % 3) * TM + r] = v;
    }
    // rows past the end take the last row's code: their contributions are zero, and they do not split a run of codes
    if (MC && tid < TM) codes[tid] = a.row_code[row0 + min(tid, nvalid - 1)] / a.code_div;
    zero_rows(sm, 3, 8, tid);
    __syncthreads();

    // ---- forward through the hidden layers
    for (int l = 0; l < last; ++l) {
      const int N = net.N[l], Np4 = round_up(N, 4);
      gemm_tile(sm, net.Wt[l], round_up(net.K[l], 8), Np4, acc, tid);
      const float* bias = net.bias[l];
      const bool per_code = MC && (l == 0 || l == net.latent_in);     // folded bias: [n_codes][Np4]
      unsigned mbits[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) mbits[r] = 0u;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int col = col_of(tid, c);
        const float b = (col < Np4) ? __ldg(bias + col) : 0.f;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          float bb = b;
          if (per_code) bb = (col < Np4) ? __ldg(bias + (size_t)codes[rg * 16 + r] * Np4 + col) : 0.f;
          float v = acc[r][c] + bb;
          if (v > 0.f) mbits[r] |= (1u << c); else v = 0.f;
          acc[r][c] = v;
        }
      }
      store_cols(sm, acc, tid, Np4);
      if (MODE != 0) {
        unsigned char* mrow = masks + ((size_t)l * TM + rg * 16) * 64 + (tid & 63);
#pragma unroll
        for (int r = 0; r < 16; ++r) mrow[r * 64] = (unsigned char)mbits[r];
      }
      const int Knext = net.K[l + 1];
      zero_rows(sm, Np4, round_up(Knext, 8), tid);
      __syncthreads();
      if (l + 1 == net.latent_in) {  // next layer takes [h | xyz]  (deep_sdf_decoder.py:92-93 after folding)
        if (tid < TM * 3) sm.act[(size_t)(N + tid % 3) * TM + tid / 3] = sm.xyz[tid];
        __syncthreads();
      }
    }

    // ---- last layer: dot product + tanh (deep_sdf_decoder.py:96-110)
    {
      const int K = net.K[last];
      const float* wl = net.W[last];  // row 0 of [Np8][Kp4]
      const int r = tid >> 2, part = tid & 3;
      float s = 0.f;
      for (int k = part; k < K; k += 4) s = fmaf(sm.act[(size_t)k * TM + r], __ldg(wl + k), s);
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      if (part == 0) {
        float x = s + __ldg(net.bias[last]);
        float t1 = x, t;
        if (net.use_tanh) { t1 = tanhf(x); t = tanhf(t1); } else { t = tanhf(x); }
        sm.rowt[r] = t;
        sm.rowt1[r] = t1;
        if (r < nvalid && a.sdf) {
          float o = t;
          if (clampd) o = fminf(fmaxf(o, -a.clamp_dist), a.clamp_dist);
          a.sdf[row0 + r] = o;
        }
        if (MODE != 0) {
          float d = 1.f - t * t;
          if (net.use_tanh) d *= (1.f - t1 * t1);
          bool uc = clampd;
          if (MODE == 2 && a.use_clamp) uc = (r < nvalid) ? (a.use_clamp[row0 + r] != 0) : false;
          if (uc && !(t >= -a.clamp_dist && t <= a.clamp_dist)) d = 0.f;
          float cf = 1.f;
          if (MODE == 2 && a.coef) cf = (r < nvalid) ? a.coef[row0 + r] : 0.f;
          if (r >= nvalid) cf = 0.f;
          sm.rowd[r] = d * cf;
        }
      }
    }
    if (MODE == 0) continue;
    __syncthreads();

    // ---- backward chain: delta wrt pre-activation of the last hidden layer
    {
      const int hl = last - 1;  // last hidden layer
      const int N = net.N[hl], Np4 = round_up(N, 4);
      const float* wl = net.W[last];
      const unsigned char* mrow = masks + ((size_t)hl * TM + rg * 16) * 64 + (tid & 63);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int col = col_of(tid, c);
        const float w = (col < N) ? __ldg(wl + col) : 0.f;
#pragma unroll
        for (int r = 0; r < 16; ++r)
          acc[r][c] = ((mrow[r * 64] >> c) & 1) ? sm.rowd[rg * 16 + r] * w : 0.f;
      }
      store_cols(sm, acc, tid, Np4);
      zero_rows(sm, Np4, round_up(N, 8), tid);
      __syncthreads();
    }
    for (int l = last - 1; l >= 0; --l) {
      // act holds delta_pre[l] as [n][row], n < N[l].  Accumulate its row-sum for the latent gradient.
      if (MODE == 2) {
        float* accp = (l == 0) ? a.acc0 : ((l == net.latent_in) ? a.accl : nullptr);
        if (accp && MC) {
          // per-code row sums: runs of equal codes, flushed to accp[code][nn] when the code changes (rotated start as below)
          const int Nl = net.N[l];
          for (int nn = tid; nn < Nl; nn += NT) {
            int cur = codes[tid & (TM - 1)];
            float s = 0.f;
            for (int k = 0; k < TM; ++k) {
              const int r = (k + tid) & (TM - 1);
              const int cr = codes[r];
              if (cr != cur) {
                if (s != 0.f) atomicAdd(accp + (size_t)cur * Nl + nn, s);
                s = 0.f; cur = cr;
              }
              s += sm.act[(size_t)nn * TM + r];
            }
            if (s != 0.f) atomicAdd(accp + (size_t)cur * Nl + nn, s);
          }
        } else if (accp) {
          for (int nn = tid; nn < net.N[l]; nn += NT) {
            float s = 0.f;
#pragma unroll 8
            for (int r = 0; r < TM; ++r) s += sm.act[(size_t)nn * TM + ((r + tid) & (TM - 1))];
            atomicAdd(accp + nn, s);
          }
        }
      }
      // gradient wrt the input of layer l:  g[row][k] = sum_n delta_pre[l][row][n] * W[l][n][k]
      const int K = net.K[l], Kp4 = round_up(K, 4);
      gemm_tile(sm, net.W[l], round_up(net.N[l], 8), Kp4, acc, tid);
      const int h = (l == 0) ? 0 : net.N[l - 1];  // width of the previous hidden activation
      if (l == 0 || l == net.latent_in) {          // xyz columns: h .. h+2
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int col = col_of(tid, c);
          if (col >= h && col < h + 3) {
#pragma unroll
            for (int r = 0; r < 16; ++r) sm.dxyz[(rg * 16 + r) * 3 + (col - h)] += acc[r][c];
          }
        }
      }
      if (l > 0) {
        const unsigned char* mrow = masks + ((size_t)(l - 1) * TM + rg * 16) * 64 + (tid & 63);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int col = col_of(tid, c);
#pragma unroll
          for (int r = 0; r < 16; ++r)
            if (!((mrow[r * 64] >> c) & 1) || col >= h) acc[r][c] = 0.f;
        }
        const int hp4 = round_up(h, 4);
        store_cols(sm, acc, tid, hp4);
        zero_rows(sm, hp4, round_up(h, 8), tid);
      }
      __syncthreads();
    }
    if (tid < TM * 3 && tid / 3 < nvalid && a.grad) a.grad[(row0 + tid / 3) * 3 + tid % 3] = sm.dxyz[tid];
  }
}

}  // namespace

int mlp_simt_launch(const NetDev& net, int mode, const MlpArgs& a, cudaStream_t stream) {
  DIST_REQUIRE(mode >= 0 && mode <= 2, "mlp_simt: bad mode %d", mode);
  DIST_REQUIRE(net.n_layers >= 2 && net.n_layers <= DIST_MAX_LAYERS, "mlp_simt: n_layers %d unsupported", net.n_layers);
  if (mode != 0) DIST_REQUIRE(net.n_layers - 1 <= MAXH_GRAD, "mlp_simt: at most %d hidden layers in gradient modes", MAXH_GRAD);
  if (a.n_host <= 0 && !a.n_dev) return DIST_OK;
  const bool mc = net.n_codes > 1;
  if (mc) DIST_REQUIRE(a.row_code && a.code_div > 0, "mlp_simt: %d latent codes need per-row codes", net.n_codes);
  static bool attr_done_dev[64] = {false};
  int cur_dev = 0;
  cudaGetDevice(&cur_dev);
  bool& attr_done = attr_done_dev[cur_dev & 63];
  if (!attr_done) {
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_simt_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemFwd));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_simt_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemGrad));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_simt_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemGrad));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_simt_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemFwd + kSmemCodes)));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_simt_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemGrad + kSmemCodes)));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_simt_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemGrad + kSmemCodes)));
    attr_done = true;
  }
  int64_t tiles = (a.n_host + TM - 1) / TM;
  int grid = (int)((tiles < (int64_t)num_sms()) ? tiles : (int64_t)num_sms());
  if (grid < 1) grid = 1;
  if (!mc) {
    if (mode == 0) { mlp_simt_kernel<0, false><<<grid, NT, kSmemFwd, stream>>>(net, a); }
    else if (mode == 1) { mlp_simt_kernel<1, false><<<grid, NT, kSmemGrad, stream>>>(net, a); }
    else { mlp_simt_kernel<2, false><<<grid, NT, kSmemGrad, stream>>>(net, a); }
  } else {
    if (mode == 0) { mlp_simt_kernel<0, true><<<grid, NT, kSmemFwd + kSmemCodes, stream>>>(net, a); }
    else if (mode == 1) { mlp_simt_kernel<1, true><<<grid, NT, kSmemGrad + kSmemCodes, stream>>>(net, a); }
    else { mlp_simt_kernel<2, true><<<grid, NT, kSmemGrad + kSmemCodes, stream>>>(net, a); }
  }
  count_launch();
  DIST_CHECK_CUDA(cudaGetLastError());
  return DIST_OK;
}

}  // namespace dist
