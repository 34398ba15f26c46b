// extern "C" surface of libdist_b200.so (see include/dist_b200.h) + small shared helpers.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <atomic>
#include <stdio.h>
#include <string.h>
#include <vector>
#include "common.cuh"

namespace dist {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int num_sms() {
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int& n = cache[dev & 63];
  if (n == 0 && (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)) n = 148;
  return n;
}

// ---- optional event timing of the decoder-row kernels (dist_profile_begin / dist_profile_end)
static bool g_prof_on = false;
static std::vector<cudaEvent_t> g_prof_pool;   // events are created once and reused across windows
static size_t g_prof_used = 0;
static const size_t kProfMaxEvents = 2 * 65536;

int mlp_launch(const dist_net_t* net, const NetDev& nd, int engine, int mode, const MlpArgs& a, cudaStream_t stream) {
  const bool timed = g_prof_on && g_prof_used + 2 <= kProfMaxEvents;
  if (timed) {
    while (g_prof_pool.size() < g_prof_used + 2) {
      cudaEvent_t e;
      DIST_CHECK_CUDA(cudaEventCreate(&e));
      g_prof_pool.push_back(e);
    }
    DIST_CHECK_CUDA(cudaEventRecord(g_prof_pool[g_prof_used], stream));
  }
  int rc;
  if (engine == DIST_ENGINE_TC) {
    rc = mlp_tc_launch(net, nd, mode, a, stream);
  } else if (mode == 3) {
    set_error("the mask-cache replay (mode 3) exists on the tensor-core engine only");
    rc = DIST_E_UNSUPPORTED;
  } else {
    // the fp32 engine knows one row range: a second segment is a second launch on the shifted arrays
    MlpArgs a1 = a;
    a1.n2_host = 0; a1.n2_dev = nullptr; a1.seg2_offset = 0; a1.screen_seg1 = 0; a1.seg_approx = nullptr;
    rc = mlp_simt_launch(nd, mode, a1, stream);
    if (rc == DIST_OK && (a.n2_dev || a.n2_host > 0)) {
      MlpArgs a2 = a1;
      const int64_t o = a.seg2_offset;
      a2.points = a.points + 3 * o; a2.n_host = a.n2_host; a2.n_dev = a.n2_dev;
      if (a.sdf) a2.sdf = a.sdf + o;
      if (a.grad) a2.grad = a.grad + 3 * o;
      if (a.coef) a2.coef = a.coef + o;
      if (a.use_clamp) a2.use_clamp = a.use_clamp + o;
      if (a.row_code) a2.row_code = a.row_code + o;
      rc = mlp_simt_launch(nd, mode, a2, stream);
    }
  }
  if (timed) {
    DIST_CHECK_CUDA(cudaEventRecord(g_prof_pool[g_prof_used + 1], stream));
    g_prof_used += 2;
  }
  return rc;
}

int make_netdev(const dist_net_t* net, NetDev* out) {
  DIST_REQUIRE(net != nullptr, "net: null descriptor");
  DIST_REQUIRE(net->n_layers >= 2 && net->n_layers <= DIST_MAX_LAYERS, "net: n_layers %d not in [2,%d]", net->n_layers, DIST_MAX_LAYERS);
  DIST_REQUIRE(net->latent_in == -1 || (net->latent_in >= 1 && net->latent_in < net->n_layers - 1),
               "net: latent_in %d must be a hidden layer >= 1", net->latent_in);
  out->n_layers = net->n_layers; out->latent_in = net->latent_in; out->use_tanh = net->use_tanh;
  for (int l = 0; l < net->n_layers; ++l) {
    DIST_REQUIRE(net->K[l] >= 1 && net->K[l] <= DIST_MAX_WIDTH && net->N[l] >= 1 && net->N[l] <= DIST_MAX_WIDTH,
                 "net: layer %d shape %dx%d exceeds max width %d", l, net->N[l], net->K[l], DIST_MAX_WIDTH);
    DIST_REQUIRE(net->Wt[l] && net->W[l] && net->bias[l], "net: layer %d has a null buffer", l);
    const int expectK = (l == 0) ? 3 : net->N[l - 1] + (l == net->latent_in ? 3 : 0);
    DIST_REQUIRE(net->K[l] == expectK, "net: layer %d has K=%d, expected %d", l, net->K[l], expectK);
    out->K[l] = net->K[l]; out->N[l] = net->N[l];
    out->Wt[l] = net->Wt[l]; out->W[l] = net->W[l]; out->bias[l] = net->bias[l];
  }
  DIST_REQUIRE(net->n_codes >= 0, "net: n_codes %d < 0", net->n_codes);
  out->n_codes = net->n_codes > 1 ? net->n_codes : 1;
  DIST_REQUIRE(net->N[net->n_layers - 1] == 1, "net: last layer must have one output (got %d)", net->N[net->n_layers - 1]);
  return DIST_OK;
}

namespace {
// out[n] = b[n] + Wz[n,:] . latent     one warp per output row; code c = blockIdx.y reads latent[c][:], writes out[c][:]
__global__ void k_fold(const float* __restrict__ Wz, const float* __restrict__ b, const float* __restrict__ latent,
                       int N, int Lz, float* __restrict__ out, int Npad) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= Npad) return;
  latent += (size_t)blockIdx.y * Lz;
  out += (size_t)blockIdx.y * Npad;
  float s = 0.f;
  if (warp < N) {
    for (int k = lane; k < Lz; k += 32) s = fmaf(Wz[(size_t)warp * Lz + k], latent[k], s);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    s += b[warp];
  }
  if (lane == 0) out[warp] = s;
}
// dist_decoder_*: the per-row codes come from net->row_code
int decoder_codes(const dist_net_t* net, MlpArgs* a) {
  if (net->n_codes <= 1) return DIST_OK;
  DIST_REQUIRE(net->row_code != nullptr, "net: n_codes = %d needs row_code", net->n_codes);
  a->row_code = net->row_code; a->code_div = 1;
  return DIST_OK;
}
}  // namespace

int render_depth_fwd(const dist_net_t*, int, const dist_camera_t*, const dist_march_t*, const dist_workspace_t*, float*,
                     uint8_t*, float*, int64_t*, cudaStream_t);
int render_normal_fwd(const dist_net_t*, int, const dist_camera_t*, const float*, const uint8_t*, float, int, float*,
                      int32_t*, float*, float*, int32_t*, int64_t*, cudaStream_t);
int render_depth_bwd(const dist_net_t*, int, const dist_camera_t*, const dist_march_t*, const dist_workspace_t*,
                     const float*, const float*, float*, float*, float*, float*, float*, int32_t*, float*, float*, uint8_t*,
                     float*, int32_t*, int64_t*, cudaStream_t);

}  // namespace dist

using namespace dist;

extern "C" {

int dist_abi_version(void) { return DIST_ABI_VERSION; }
const char* dist_last_error(void) { return g_err; }
long long dist_launch_count(void) { return g_launches.load(); }

int dist_profile_begin(void) {
  g_prof_used = 0;
  g_prof_on = true;
  return DIST_OK;
}

int dist_profile_end(double* total_ms, long long* launches) {
  g_prof_on = false;
  double sum = 0.0;
  for (size_t i = 0; i + 1 < g_prof_used; i += 2) {
    DIST_CHECK_CUDA(cudaEventSynchronize(g_prof_pool[i + 1]));
    float ms = 0.f;
    DIST_CHECK_CUDA(cudaEventElapsedTime(&ms, g_prof_pool[i], g_prof_pool[i + 1]));
    sum += ms;
  }
  if (total_ms) *total_ms = sum;
  if (launches) *launches = (long long)(g_prof_used / 2);
  g_prof_used = 0;
  return DIST_OK;
}

int dist_device_supports_tc(int device) {
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

int dist_fold_latent(const dist_net_t* net, const float* latent, float* out0, float* outl, void* stream) {
  DIST_REQUIRE(net && out0, "fold_latent: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int Lz = net->latent_size;
  DIST_REQUIRE(net->n_codes >= 0 && net->n_codes <= 65535, "fold_latent: n_codes %d outside [0, 65535]", net->n_codes);
  const unsigned C = net->n_codes > 1 ? (unsigned)net->n_codes : 1u;      // one grid row per code
  {
    const int N = net->N[0], Np = round_up(N, 4);
    if (Lz > 0) {
      DIST_REQUIRE(latent && net->Wz0 && net->b0, "fold_latent: null latent buffers");
      k_fold<<<dim3((Np * 32 + 255) / 256, C), 256, 0, st>>>(net->Wz0, net->b0, latent, N, Lz, out0, Np); count_launch();
    } else {
      k_fold<<<dim3((Np * 32 + 255) / 256, C), 256, 0, st>>>(net->b0, net->b0, net->b0, N, 0, out0, Np); count_launch();
    }
  }
  if (net->latent_in >= 0 && Lz > 0) {
    DIST_REQUIRE(outl && net->Wzl && net->bl, "fold_latent: null latent_in buffers");
    const int N = net->N[net->latent_in], Np = round_up(N, 4);
    k_fold<<<dim3((Np * 32 + 255) / 256, C), 256, 0, st>>>(net->Wzl, net->bl, latent, N, Lz, outl, Np); count_launch();
  }
  DIST_CHECK_CUDA(cudaGetLastError());
  return DIST_OK;
}

int dist_decoder_forward(const dist_net_t* net, int engine, const float* points, int64_t n_host, const int32_t* n_dev,
                         float clamp_dist, float* sdf, void* stream) {
  NetDev nd;
  int rc = make_netdev(net, &nd);
  if (rc) return rc;
  MlpArgs a{};
  a.points = points; a.n_host = n_host; a.n_dev = n_dev; a.clamp_dist = clamp_dist; a.sdf = sdf;
  rc = decoder_codes(net, &a);
  if (rc) return rc;
  return mlp_launch(net, nd, engine, 0, a, (cudaStream_t)stream);
}

int dist_decoder_forward_tiers(const dist_net_t* net, const float* points, int64_t n_screen, int64_t n_exact,
                               int64_t exact_offset, float screen_thresh, float* sdf, uint8_t* seg_approx,
                               unsigned long long* tile_counters, void* stream) {
  NetDev nd;
  int rc = make_netdev(net, &nd);
  if (rc) return rc;
  DIST_REQUIRE(seg_approx, "decoder_forward_tiers: seg_approx is required");
  MlpArgs a{};
  a.points = points; a.n_host = n_screen; a.n2_host = n_exact; a.seg2_offset = exact_offset; a.clamp_dist = 0.f; a.sdf = sdf;
  a.screen_seg1 = 1; a.screen_thresh = screen_thresh; a.seg_approx = seg_approx; a.tile_counters = tile_counters;
  rc = decoder_codes(net, &a);
  if (rc) return rc;
  return mlp_launch(net, nd, DIST_ENGINE_TC, 0, a, (cudaStream_t)stream);
}

int dist_decoder_forward_masks(const dist_net_t* net, const float* points, int64_t n, float* sdf, uint32_t* mask_buf,
                               int64_t mask_cap, int64_t mask_base, void* stream) {
  NetDev nd;
  int rc = make_netdev(net, &nd);
  if (rc) return rc;
  DIST_REQUIRE(mask_buf && mask_cap > 0 && mask_base >= 0, "decoder_forward_masks: mask buffer required");
  MlpArgs a{};
  a.points = points; a.n_host = n; a.clamp_dist = 0.f; a.sdf = sdf;
  a.mask_buf = mask_buf; a.mask_cap = mask_cap; a.mask_base_host = mask_base;
  rc = decoder_codes(net, &a);
  if (rc) return rc;
  return mlp_launch(net, nd, DIST_ENGINE_TC, 0, a, (cudaStream_t)stream);
}

int dist_decoder_backward_masked(const dist_net_t* net, const int32_t* slots, const float* sdf_in, const float* coef, int64_t n,
                                 float clamp_dist, const uint32_t* mask_buf, int64_t mask_cap, float* dpoints, float* acc0,
                                 float* accl, void* stream) {
  NetDev nd;
  int rc = make_netdev(net, &nd);
  if (rc) return rc;
  MlpArgs a{};
  a.n_host = n; a.clamp_dist = clamp_dist; a.grad = dpoints; a.coef = coef; a.acc0 = acc0; a.accl = accl;
  a.mask_buf = const_cast<uint32_t*>(mask_buf); a.mask_cap = mask_cap; a.slots = slots; a.sdf_in = sdf_in;
  rc = decoder_codes(net, &a);
  if (rc) return rc;
  return mlp_launch(net, nd, DIST_ENGINE_TC, 3, a, (cudaStream_t)stream);
}

int dist_decoder_input_grad(const dist_net_t* net, int engine, const float* points, int64_t n_host,
                            const int32_t* n_dev, float clamp_dist, float* grad, float* sdf, void* stream) {
  NetDev nd;
  int rc = make_netdev(net, &nd);
  if (rc) return rc;
  MlpArgs a{};
  a.points = points; a.n_host = n_host; a.n_dev = n_dev; a.clamp_dist = clamp_dist; a.sdf = sdf; a.grad = grad;
  rc = decoder_codes(net, &a);
  if (rc) return rc;
  return mlp_launch(net, nd, engine, 1, a, (cudaStream_t)stream);
}

int dist_decoder_backward(const dist_net_t* net, int engine, const float* points, const float* coef,
                          const uint8_t* use_clamp, int64_t n_host, const int32_t* n_dev, float clamp_dist,
                          float* dpoints, float* acc0, float* accl, void* stream) {
  NetDev nd;
  int rc = make_netdev(net, &nd);
  if (rc) return rc;
  MlpArgs a{};
  a.points = points; a.n_host = n_host; a.n_dev = n_dev; a.clamp_dist = clamp_dist; a.grad = dpoints;
  a.coef = coef; a.use_clamp = use_clamp; a.acc0 = acc0; a.accl = accl;
  rc = decoder_codes(net, &a);
  if (rc) return rc;
  return mlp_launch(net, nd, engine, 2, a, (cudaStream_t)stream);
}

int dist_render_depth_fwd(const dist_net_t* net, int engine, const dist_camera_t* cam, const dist_march_t* mp,
                          const dist_workspace_t* ws, float* Zdepth, uint8_t* mask, float* min_sdf,
                          int64_t* rows_evaluated, void* stream) {
  DIST_REQUIRE(net && cam && mp && ws && Zdepth && mask && min_sdf, "render_depth_fwd: null argument");
  return render_depth_fwd(net, engine, cam, mp, ws, Zdepth, mask, min_sdf, rows_evaluated, (cudaStream_t)stream);
}

int dist_render_normal_fwd(const dist_net_t* net, int engine, const dist_camera_t* cam, const float* Zdepth,
                           const uint8_t* mask, float clamp_dist, int normalize, float* Znormal, int32_t* scratch_idx,
                           float* scratch_pts, float* scratch_grad, int32_t* scratch_count, int64_t* rows_evaluated,
                           void* stream) {
  DIST_REQUIRE(net && cam && Zdepth && mask && Znormal && scratch_idx && scratch_pts && scratch_grad && scratch_count,
               "render_normal_fwd: null argument");
  return render_normal_fwd(net, engine, cam, Zdepth, mask, clamp_dist, normalize, Znormal, scratch_idx, scratch_pts,
                           scratch_grad, scratch_count, rows_evaluated, (cudaStream_t)stream);
}

int dist_render_depth_bwd(const dist_net_t* net, int engine, const dist_camera_t* cam, const dist_march_t* mp,
                          const dist_workspace_t* ws, const float* gZ, const float* gM, float* acc0, float* accl,
                          float* d_cam_pos, float* d_ray, float* d_ray_coarse, int32_t* scratch_row_pix, float* scratch_pts,
                          float* scratch_coef, uint8_t* scratch_clamp, float* scratch_dpts, int32_t* scratch_count,
                          int64_t* rows_evaluated, void* stream) {
  DIST_REQUIRE(net && cam && mp && ws && acc0 && scratch_row_pix && scratch_pts && scratch_coef && scratch_dpts &&
                   scratch_count, "render_depth_bwd: null argument");
  return render_depth_bwd(net, engine, cam, mp, ws, gZ, gM, acc0, accl, d_cam_pos, d_ray, d_ray_coarse, scratch_row_pix, scratch_pts,
                          scratch_coef, scratch_clamp, scratch_dpts, scratch_count, rows_evaluated,
                          (cudaStream_t)stream);
}

}  // extern "C"
