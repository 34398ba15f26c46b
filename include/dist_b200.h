/*
 * dist_b200.h -- C ABI of the B200-native sphere-tracing library (libdist_b200.so).
 *
 * The reference (B1ueber2y/DIST-Renderer) has no FFI/plugin interface: its boundary is the Python class
 * `SDFRenderer` (core/sdfrenderer/renderer.py:12) plus `decode_sdf` / `decode_sdf_gradient`
 * (core/utils/decoder_utils.py:53,76) and `Decoder.inference` (core/graph/deep_sdf_decoder.py:80).
 * Each entry point below names the reference code it replaces.  Conventions:
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates; the library never allocates,
 *     never synchronises the device and never touches the host copy of any buffer), except `dist_net_t*`
 *     / `dist_camera_t*` descriptors, which are small host structs passed by pointer and copied at launch;
 *   - all work is enqueued on the `stream` argument (a cudaStream_t passed as void*);
 *   - return value 0 = success, otherwise a DIST_E_* code; dist_last_error() gives the message;
 *   - all floating-point data is fp32, row-major.
 */
#ifndef DIST_B200_H_
#define DIST_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIST_ABI_VERSION 3
#define DIST_MAX_LAYERS 16
#define DIST_MAX_WIDTH 512
#define DIST_MAX_BUFFER 8      /* max buffer_size (samples kept per ray) */

enum {
  DIST_OK = 0,
  DIST_E_INVALID = 1,    /* bad argument / unsupported network shape */
  DIST_E_CUDA = 2,       /* a CUDA runtime call failed */
  DIST_E_UNSUPPORTED = 3 /* feature not available in this build (e.g. tensor path on a non-sm_100 device) */
};

enum { DIST_MARCH_TRIVIAL = 0, DIST_MARCH_RECURSIVE = 1, DIST_MARCH_PYRAMID = 2 };

/* Evaluation engines for the decoder rows. */
enum {
  DIST_ENGINE_SIMT = 0,   /* fp32 FFMA reference engine (exact fp32 arithmetic, CUDA cores) */
  DIST_ENGINE_TC = 1      /* tcgen05 tensor-core engine, split-fp16 operands with fp32 accumulation */
};

/*
 * The decoder network in "folded" form (deep_sdf_decoder.py:80-111 with weight-norm applied and the latent code
 * folded into per-render biases -- SURVEY.md section 7 step 2):
 *   layer 0 takes xyz (K=3); the layer listed in `latent_in` takes [h | xyz] (K = width of h + 3);
 *   every other layer takes the previous activation.  ReLU after all but the last layer, tanh at the end
 *   (twice when `use_tanh`).  The last layer must have N = 1.
 * Wt[l] : [Kp8][Np4] fp32, transposed weights (input-major), zero padded: Kp8 = roundup(K,8), Np4 = roundup(N,4).
 * W [l] : [Np8][Kp4] fp32, weights (output-major), zero padded.
 * bias[l]: [Np4] fp32.  For layer 0 and the latent_in layer this is the per-render folded bias written by
 *          dist_fold_latent(); for the others the plain bias.
 * Wz0 / Wzl : latent columns of layer 0 / the latent_in layer, [N][latent_size], used by dist_fold_latent().
 */
typedef struct dist_net {
  int32_t n_layers;
  int32_t latent_size;
  int32_t latent_in;          /* layer index, or -1 */
  int32_t use_tanh;
  int32_t K[DIST_MAX_LAYERS];
  int32_t N[DIST_MAX_LAYERS];
  const float* Wt[DIST_MAX_LAYERS];
  const float* W[DIST_MAX_LAYERS];
  const float* bias[DIST_MAX_LAYERS];
  const float* Wz0;
  const float* b0;            /* unfolded bias of layer 0, [N0] */
  const float* Wzl;
  const float* bl;            /* unfolded bias of the latent_in layer */
  /* tensor-core engine operands (NULL when only the SIMT engine is prepared) */
  const void* tc_blob;        /* split-fp16 weight tiles, see csrc/mlp_tc.cu */
  const float* tc_scale;      /* HOST array: 1/sW per tensor-core layer (forward layers, then the transposed chain) */
  int64_t tc_blob_bytes;
  const float* tc_bias[DIST_MAX_LAYERS]; /* biases in the engine's scaled activation units (bias * 32), per net layer */
  /* Several latent codes in one call (0 or 1: one code, the layout above).  No counterpart in the reference, which decodes
   * one code per call.  With n_codes > 1, bias[0], bias[latent_in] and tc_bias[latent_in] point to per-code tables
   * [n_codes][Np4] (written by dist_fold_latent from latent [n_codes][latent_size]), and the acc0 / accl accumulators of the
   * backward entry points are [n_codes][N] (N = N[0] / N[latent_in]).  Which code a decoder row uses: */
  int32_t n_codes;
  const int32_t* row_code;    /* dist_decoder_*: device [n] code of row i, in [0, n_codes).  Ignored by dist_render_*, where
                                 the code of a row is the view of its pixel: n_codes must then equal dist_camera_t.n_views
                                 (DIST_E_INVALID otherwise), view v being rendered with code v */
} dist_net_t;

/* Camera + image description for one render (renderer.py:13-59,180-200). */
typedef struct dist_camera {
  float Kinv[9];              /* inverse intrinsic, row-major (renderer.py:161-164) */
  float M[9];                 /* matrix whose transpose maps world points into the decoder frame: transform_matrix
                                 (renderer.py:44-48, :119), or identity when use_transform=False; only 3x3 supported */
  float Mn[9];                /* transform_matrix applied to the normals (renderer.py:902) -- always the real one */
  const float* R;             /* device, [n_views][9] row-major world->camera rotations */
  const float* cam_pos;       /* device, [n_views][3]  = -R^T T  (renderer.py:180-188) */
  int32_t width;              /* full image width */
  int32_t height;             /* full image height */
  int32_t row0;               /* first image row rendered by this call (ray-tile sharding, SURVEY 8e) */
  int32_t row_step;           /* image rows between the starts of consecutive row groups (interleaved bands) */
  int32_t n_rows;             /* number of rows rendered; local pixel lp = lrow*width + x */
  float radius;               /* unit-sphere radius (renderer.py:23) */
  int32_t n_views;            /* views of the same shape marched by ONE call (0 or 1: a single view).  All per-pixel
                                 arrays then hold n_views * n_rows * width entries, view-major: the multi-view loops of
                                 optimize_multi.py:62-80 / renderer_warp.py:108-109 become one march, one compaction
                                 list, one tail.  Each view keeps the per-render semantics of the reference (its own
                                 early break, 'No valid depth' test, pyramid levels). */
  int32_t row_group;          /* rows per interleaved group (0 or 1: single rows): local row l is image row
                                 row0 + (l / row_group) * row_step + l % row_group.  DIST_MARCH_PYRAMID on a band needs
                                 row_group % 4 == 0, which keeps the 1/2- and 1/4-resolution levels band-local
                                 (SURVEY 8e); the last group of a band may be shorter (image height not a multiple). */
} dist_camera_t;

/* March parameters (renderer.py:13 ctor arguments + render_depth arguments). */
typedef struct dist_march {
  int32_t march_step;
  int32_t buffer_size;
  int32_t marching_type;      /* DIST_MARCH_* */
  int32_t first_query_check;  /* renderer.py:580-582 */
  float ratio;                /* ray_marching_ratio */
  float threshold;
  float clamp_dist;
  int32_t replay_grad_rounding; /* reproduce the value-neutral (z - a) + a roundings of renderer.py:414-417 (a render with depth
                                   gradients adds and subtracts each selected sample; no_grad_depth skips it, renderer.py:413).
                                   Bit mask: bit 31 = every view, else bit v = view v of a multi-view call (v < 31) */
  int32_t coarse_steps[2];    /* DIST_MARCH_PYRAMID: trivial steps at 1/4 and 1/2 resolution (renderer.py:13 march_step_list) */
  int32_t screen;             /* two-tier precision of the march on DIST_ENGINE_TC (0 = every row at full precision): a row
                                 whose sdf is safely beyond the clamp, |sdf| > clamp_dist + screen_margin, steps by exactly
                                 ratio * clamp_dist whatever its last bits are (renderer.py:548-551), so 128-row tiles are
                                 first evaluated with ONE fp16 tensor-core pass and only tiles with a nearer row are
                                 re-evaluated with the three split-precision passes; the value of a one-pass sample is
                                 only ever used where the reference's result does not depend on it, except a ray's
                                 smallest |sdf|, which is re-queried at full precision before the maps are written */
  float screen_margin;        /* one-pass values must be accurate to screen_margin / 2 (checked at prepare time) */
  float screen_tpred;         /* a ray whose last |sdf| exceeds screen_tpred is predicted "far" for its next sample ... */
  float screen_ext_margin;    /* ... as is one whose last two samples extrapolate linearly to beyond clamp_dist +
                                 screen_margin + screen_ext_margin; rays predicted far are compacted into the first row
                                 segment of the next step (one-pass tiles), all others into the second (three passes) */
  int32_t cam_grad_levels;    /* dist_render_depth_bwd: which samples carry a camera gradient -- bit 0: samples of the
                                 full-resolution march, bit 1: samples inherited from the coarse pyramid levels
                                 (0 = both).  no_grad_camera detaches only the points of ray_marching_recursive
                                 (renderer.py:536-537); ray_marching_trivial never detaches (renderer.py:481-484) */
} dist_march_t;

/*
 * Per-render device workspace, all arrays sized by the number of local pixels P = n_views*n_rows*width
 * (B = buffer_size).  The top-B sample records double as the tensors saved for backward.
 */
typedef struct dist_workspace {
  float* ray;        /* [3][P] unit ray directions, world frame */
  float* entry;      /* [P] ray depth of the unit-sphere entry (renderer.py:254-273) */
  float* exit_;      /* [P] entry + chord (renderer.py:275-282) */
  float* dist;       /* [P] distance of the ray to the origin */
  float* z;          /* [P] marching depth relative to entry */
  uint8_t* flags;    /* [P] bit0 sphere hit, bit1 first query > threshold */
  int32_t* nreal;    /* [P] number of real samples recorded */
  float* top_sdf;    /* [B][P] samples with the smallest |sdf|, sorted ascending */
  float* top_pt;     /* [B][3][P] their points (decoder frame) */
  float* top_zafter; /* [B][P] marching depth after the step that produced the sample */
  float* top_zgen;   /* [B][P] absolute ray depth the sample point was generated at (NaN: not on this ray) */
  int32_t* list_a;   /* [2*SEG] active ray list (ping), two row segments -- see below */
  int32_t* list_b;   /* [2*SEG] active ray list (pong) */
  float* pts;        /* [2][2*SEG][3] query points, ping-pong by step parity */
  float* sdf;        /* [2*SEG] decoder outputs of the current step */
  int32_t* counts;   /* [2*(march_step + 2)] active rays per step and segment (8-byte aligned: a step's pair advances with one 64-bit atomic); zeroed by dist_render_depth_fwd */
  float* sdf_origin; /* [1] sdf at the origin (filler samples, renderer.py:539-540); [n_views] when dist_net_t.n_codes > 1
                        (one origin query per view, with that view's code) */
  float* entry0;     /* [P] true unit-sphere entry depth; == entry except in DIST_MARCH_PYRAMID, where `entry` holds the
                        depth the full-resolution march starts from (inherited from the 1/2-resolution parent ray) */
  uint8_t* top_lvl;  /* [B][P] bits 0-1: pyramid level the sample was taken at (0 = this ray; 1, 2 = parent / grandparent
                        ray); bit 7: the recorded sdf is a one-pass value; bit 6: it was re-queried at full precision */
  /* DIST_MARCH_PYRAMID only (renderer.py:713-805).  With (w1,h1) = ceil((w,h)/2), (w2,h2) = ceil((w1,h1)/2),
   * P1 = w1*h1, P2 = w2*h2:  pyr_f: 23*(P1+P2) floats, pyr_i: 4*(P1+P2)+8 int32, pyr_b: (P1+P2) bytes. */
  float* pyr_f;      /* (all three scale with n_views) */
  int32_t* pyr_i;
  uint8_t* pyr_b;
  /* Row segments of the march's query arrays: SEG = round_up(P + 1, 128); `list_a`, `list_b`, `sdf` hold 2*SEG entries,
   * `pts` 2 x 2*SEG x 3, `counts` 2*(march_step + 2): counts[2s] / counts[2s+1] = rows of step s in segment 1 (rows
   * [0, n1): rays predicted far from the surface) / segment 2 (rows [SEG, SEG + n2): the rest, and the origin at step 0).
   * two-tier precision (dist_march_t.screen; NULL otherwise): */
  uint8_t* seg_approx;  /* [2*SEG/64] per 64-row half-tile of the current step: 1 = one-pass values */
  float* sprev;         /* [P] the ray's previous sdf (far / near prediction) */
  int32_t* rq_idx;      /* [P*B] re-query rows: local pixel * DIST_MAX_BUFFER + record slot */
  float* rq_pts;        /* [P*B][3] */
  float* rq_sdf;        /* [P*B] */
  int32_t* rq_cnt;      /* [1] */
  /* ReLU-mask cache (NULL: off; needs dist_march_t.screen): the forward records, for every march / re-query row evaluated at
   * full precision, the sign bits of all hidden layers (one 32-bit word per layer and 32-feature block) in
   * mask_buf[16 * (n_layers - 1)][mask_cap]; a selected sample remembers its slot in top_slot[B][P] (-1: none), and
   * dist_render_depth_bwd replays such samples with the transposed chain alone (no forward recomputation).  A slot is
   * mask_base[s] + (row index in segment 2 of step s); mask_base ([march_step + 3] int32) is maintained on the device. */
  uint32_t* mask_buf;
  int32_t* mask_base;
  int32_t* top_slot;
  int32_t* bm_row;      /* [P*B] backward scratch of the rows replayed from the mask cache: pixel * DIST_MAX_BUFFER + slot ... */
  int32_t* bm_slot;     /* [P*B] ... their mask slots */
  float* bm_sdf;        /* [P*B] ... their recorded decoder outputs */
  float* bm_coef;       /* [P*B] ... their upstream coefficients */
  float* bm_dpts;       /* [P*B][3] ... d/d point out */
  int32_t* bm_cnt;      /* [1] */
  unsigned long long* tile_counters; /* optional [2], accumulated: 128-row tile programs evaluated with one fp16 pass /
                           with three (a gradient tile counts two programs: forward + transposed chain) */
  int64_t mask_cap;   /* row slots of mask_buf */
  int32_t* view_stat; /* [n_views][4] per-view bookkeeping, zeroed by dist_render_depth_fwd: [0] rays alive at step 0
                         (0 <=> the reference raises 'No valid depth', renderer.py:214), [1] march steps the view
                         executed before its early break (renderer.py:562), [2] float bits of the largest coarse-level
                         sphere entry (renderer.py:270-272), [3] != 0: a decoder output of the march was not in
                         [-1, 1] (NaN / inf: operand overflow of the fp16 tensor-core engine) */
} dist_workspace_t;

/* ---- library ---- */
int dist_abi_version(void);
const char* dist_last_error(void);
/* number of CUDA kernels this library has launched in this process so far */
long long dist_launch_count(void);
/* Kernel timing for roofline accounting (off by default, no cost when off).  While enabled, every decoder-row kernel
 * launch (the dominant kernel: dist_decoder_* and the launches inside dist_render_*) is bracketed by a pair of CUDA
 * events on its own stream.  dist_profile_end synchronises those events, returns the number of bracketed launches and
 * their summed duration in milliseconds, and switches timing off.  Not thread-safe; at most 65536 launches per window. */
int dist_profile_begin(void);
int dist_profile_end(double* total_ms, long long* launches);
/* 1 if the device has the tcgen05 path (compute capability 10.x) */
int dist_device_supports_tc(int device);

/* ---- decoder (decoder_utils.py:53-92, deep_sdf_decoder.py:80-111) ---- */

/* Per-render folded biases: out0[n] = b0[n] + Wz0[n,:].latent ; outl likewise for the latent_in layer.
 * Replaces the latent.expand + torch.cat of decoder_utils.py:61-62 and deep_sdf_decoder.py:92-93.
 * net->n_codes > 1: latent is [n_codes][latent_size], out0 / outl are [n_codes][Np4], row c computed exactly as a
 * single-code call on latent[c] computes it. */
int dist_fold_latent(const dist_net_t* net, const float* latent, float* out0, float* outl, void* stream);

/* sdf[i] = decoder(latent, points[i]) for i < n (n read from *n_dev when n_dev != NULL, else n_host).
 * clamp_dist <= 0 means no clamp.  Replaces decode_sdf (decoder_utils.py:53-74). */
int dist_decoder_forward(const dist_net_t* net, int engine, const float* points, int64_t n_host,
                         const int32_t* n_dev, float clamp_dist, float* sdf, void* stream);

/* dist_decoder_forward on the tensor-core engine with the two-tier precision the march uses (dist_march_t.screen), exposed
 * for the prepare-time accuracy check of the one-pass values and for tests.  Rows [0, n_screen) are evaluated in 128-row
 * tiles with ONE fp16 pass first; a 64-row half-tile keeps those values when all of its rows have |sdf| > screen_thresh
 * and is flagged in seg_approx[row / 64] = 1; a tile with a nearer row in either half is re-evaluated with the three
 * split-precision passes.  Rows [exact_offset, exact_offset + n_exact) (exact_offset a multiple of 128, >= n_screen) get the
 * three passes directly.  Every row not flagged is bit-identical to dist_decoder_forward.  tile_counters (optional, [2])
 * += tile programs evaluated with one / three passes.
 * No counterpart in the reference: its decoder (deep_sdf_decoder.py:80-111) is fp32 throughout. */
int dist_decoder_forward_tiers(const dist_net_t* net, const float* points, int64_t n_screen, int64_t n_exact,
                               int64_t exact_offset, float screen_thresh, float* sdf, uint8_t* seg_approx,
                               unsigned long long* tile_counters, void* stream);

/* Mask cache of the tensor-core engine, exposed for tests (the renderer uses it through dist_workspace_t.mask_buf):
 * dist_decoder_forward_masks = dist_decoder_forward (three passes, no clamp) that also records the ReLU sign bits of every
 * hidden layer of row i at slot mask_base + i of mask_buf[16 * (n_layers - 1)][mask_cap];
 * dist_decoder_backward_masked = dist_decoder_backward for rows given by (mask slot, recorded decoder output, coefficient)
 * instead of points: the transposed chain alone, no forward recomputation (what the autograd backward of the reference
 * does with its saved activations, renderer.py:386,415). */
int dist_decoder_forward_masks(const dist_net_t* net, const float* points, int64_t n, float* sdf, uint32_t* mask_buf,
                               int64_t mask_cap, int64_t mask_base, void* stream);
int dist_decoder_backward_masked(const dist_net_t* net, const int32_t* slots, const float* sdf_in, const float* coef, int64_t n,
                                 float clamp_dist, const uint32_t* mask_buf, int64_t mask_cap, float* dpoints, float* acc0,
                                 float* accl, void* stream);

/* grad[i] = d clamp(sdf)/d xyz at points[i]; sdf (optional) receives the clamped value.
 * Replaces decode_sdf_gradient (decoder_utils.py:76-92). */
int dist_decoder_input_grad(const dist_net_t* net, int engine, const float* points, int64_t n_host,
                            const int32_t* n_dev, float clamp_dist, float* grad, float* sdf, void* stream);

/* Backward replay: for row i with upstream coefficient coef[i] on its (optionally clamped) sdf,
 *   dpoints[i] = coef[i] * d sdf/d xyz,   acc0 += sum_i coef[i] * d sdf/d preact0,  accl += ... latent_in layer.
 * use_clamp[i] != 0 applies the clamp mask.  acc0/accl ([N0]/[Nl] fp32) are accumulated atomically (caller zeroes).
 * Replaces the autograd backward of the re-query decoder calls (renderer.py:386,415; optimize_single.py:83). */
int dist_decoder_backward(const dist_net_t* net, int engine, const float* points, const float* coef,
                          const uint8_t* use_clamp, int64_t n_host, const int32_t* n_dev, float clamp_dist,
                          float* dpoints, float* acc0, float* accl, void* stream);

/* ---- renderer (renderer.py:836-910) ---- */

/* Ray setup + sphere clip + march + sample selection + depth/mask/min-sdf maps for the rows of `cam`.
 * Outputs (local pixel order): Zdepth[P] (1e11 where the ray misses the unit sphere), mask[P] (uint8),
 * min_sdf[P] (dist + threshold - radius where the ray misses the unit sphere), rows_evaluated[1] (int64 counter of
 * decoder rows pushed through the network, for roofline accounting).  Replaces render_depth forward
 * (renderer.py:836-878) with ray_marching_trivial / ray_marching_recursive (renderer.py:472-583). */
int dist_render_depth_fwd(const dist_net_t* net, int engine, const dist_camera_t* cam, const dist_march_t* mp,
                          const dist_workspace_t* ws, float* Zdepth, uint8_t* mask, float* min_sdf,
                          int64_t* rows_evaluated, void* stream);

/* Surface normals at Zdepth on `mask` pixels: Znormal[3][P], zeros elsewhere.  Replaces render_normal
 * (renderer.py:880-910) with the analytic decoder input-gradient (decoder_utils.py:76-92).
 * scratch_idx[P] int32, scratch_pts[P][3], scratch_grad[P][3], scratch_count[1] int32 are caller workspaces. */
int dist_render_normal_fwd(const dist_net_t* net, int engine, const dist_camera_t* cam, const float* Zdepth,
                           const uint8_t* mask, float clamp_dist, int normalize, float* Znormal,
                           int32_t* scratch_idx, float* scratch_pts, float* scratch_grad, int32_t* scratch_count,
                           int64_t* rows_evaluated, void* stream);

/* Backward of dist_render_depth_fwd for upstream gZ[P] (on Zdepth) and gM[P] (on min_sdf; only sphere-hit pixels are
 * used): replays the saved top-B sample points.  Outputs acc0/accl as in dist_decoder_backward, d_cam_pos[3] and
 * d_ray[3][P] (gradient w.r.t. camera centre and per-pixel unit ray, for the host-side camera chain).
 * Either gZ or gM may be NULL.  scratch_* hold the compacted replay rows: rows up to P*buffer_size.
 * d_ray_coarse ([3][P1] then [3][P2], DIST_MARCH_PYRAMID with camera gradients only, else NULL): gradient w.r.t. the
 * unit rays of the 1/2- and 1/4-resolution pixel centres for samples taken on parent rays.
 * rows_evaluated (optional): int64[2] counters, [0] += rows replayed in full (forward + transposed chain, 2F flop each),
 * [1] += rows replayed from the mask cache (transposed chain only, F flop each). */
int dist_render_depth_bwd(const dist_net_t* net, int engine, const dist_camera_t* cam, const dist_march_t* mp,
                          const dist_workspace_t* ws, const float* gZ, const float* gM, float* acc0, float* accl,
                          float* d_cam_pos, float* d_ray, float* d_ray_coarse, int32_t* scratch_row_pix, float* scratch_pts,
                          float* scratch_coef, uint8_t* scratch_clamp, float* scratch_dpts, int32_t* scratch_count,
                          int64_t* rows_evaluated, void* stream);

/* ---- two-view photometric warp (renderer_warp.py:18-101, loss_utils.py:9-25) ---- */

/* For every pixel of view 1 with mask1 != 0: p = cam_pos1 + ray1 * Zdepth1 (world frame), xyz = K (R2 p + T2), (u, v) =
 * xyz.xy / xyz.z; the pixel is kept when (xyz.z - bilinear(depth2, u, v))^2 < thres_depth (depth2: view 2's z-depth map,
 * [P]); for kept pixels the colour of img1 [P][3] is compared with the bilinear sample of img2 [P][3] at (u, v)
 * (torch-1.1 grid_sample convention: align_corners=True, zero padding).  Outputs: loss_sum[1] = sum of |c1 - c2| over kept
 * pixels and channels, count[1] = kept pixels (the reference's loss is loss_sum / (3 count)), keep[P], vis1 / vis2 [P][3]
 * (the two colours at kept pixels, zero elsewhere).  cam1: view 1 (full image, one view); K_host: intrinsic, HOST [9];
 * R2, T2: device.  Replaces get_valid_points / valid_points_depth / compute_loss_color + grid_sample_on_img. */
int dist_warp_loss_fwd(const dist_camera_t* cam1, const float* K_host, const float* R2, const float* T2, const float* Zdepth1,
                       const uint8_t* mask1, const float* depth2, const float* img1, const float* img2, float thres_depth,
                       float* loss_sum, int32_t* count, uint8_t* keep, float* vis1, float* vis2, void* stream);

/* Backward of dist_warp_loss_fwd for gscale[0] = dL/d(loss_sum) (device): dZdepth1[P], d_ray1[3][P] (w.r.t. view 1's unit
 * rays), d_cam_pos1[3], dR2[9], dT2[3].  The depth-consistency test and the images carry no gradient, as in the reference. */
int dist_warp_loss_bwd(const dist_camera_t* cam1, const float* K_host, const float* R2, const float* T2, const float* Zdepth1,
                       const uint8_t* keep, const float* img1, const float* img2, const float* gscale, float* dZdepth1,
                       float* d_ray1, float* d_cam_pos1, float* dR2, float* dT2, void* stream);

/* ---- mesh extraction (SURVEY.md 8f next-2): device replacements for the host half of latent_vec_to_points -------------
 * Reference: core/evaluation/create_mesh.py:144-175 (skimage.measure.marching_cubes_lewiner on a host copy of the grid),
 * core/evaluation/transforms.py:8-32 (.ply on disk -> trimesh.sample.sample_surface), core/evaluation/eval_func.py:5-39
 * (scipy cKDTree chamfer).  All pointers are device pointers unless they say _host; nothing is allocated inside.
 *
 * Marching cubes over vol[n0][n1][n2] (fp32, axis 2 fastest), inside = value < level.  Two calls because the output size
 * is data dependent:
 *   dist_mc_count  fills scan[M] (M = n0*n1*n2; low 32 bits = index of the grid point's first vertex, high 32 bits = index
 *                  of its cube's first triangle), mask[M] (which of the point's +axis edges carry a vertex) and
 *                  totals[0] = n_vertices + (n_triangles << 32); scratch holds dist_scan_scratch_elems(M) int64.
 *   dist_mc_emit   writes verts[n_vertices][3] = origin_host + spacing_host * (grid index + t) and faces[n_triangles][3]
 *                  (vertex order: grid point, then axis; face order: cube, then the case table's order; normals point
 *                  towards larger values).  Case table and conventions: dist-renderer_b200/mc_tables.py. */
int64_t dist_scan_scratch_elems(int64_t n);
int dist_mc_count(const float* vol, int n0, int n1, int n2, float level, int64_t* scan, uint8_t* mask, int64_t* scratch,
                  int64_t* totals, void* stream);
int dist_mc_emit(const float* vol, int n0, int n1, int n2, float level, const float* origin_host, const float* spacing_host,
                 const int64_t* scan, const uint8_t* mask, float* verts, int32_t* faces, void* stream);

/* Area-weighted surface sampling (trimesh.sample.sample_surface's scheme).  dist_tri_area_scan: cum[n_faces] = exclusive
 * prefix sums (fp64) of the fp32 triangle areas, total[0] = their sum; scratch holds dist_scan_scratch_elems(n_faces)
 * doubles.  dist_surface_sample: for uniforms u[count][3] in [0,1), u[.][0] picks the face whose cumulative-area interval
 * holds u*total, (u[.][1], u[.][2]) the point (reflected when their sum exceeds 1); points[count][3], face_index[count]
 * (may be NULL). */
int dist_tri_area_scan(const float* verts, const int32_t* faces, int64_t n_faces, double* cum, double* scratch, double* total,
                       void* stream);
int dist_surface_sample(const float* verts, const int32_t* faces, int64_t n_faces, const double* cum, const double* total,
                        const float* u, int64_t count, float* points, int32_t* face_index, void* stream);

/* d2[i] = squared distance from query[i] to its nearest point of ref (fp32, brute force), index[i] = that point (may be
 * NULL); best[n_query] is uint64 scratch.  cKDTree(ref).query(query) of eval_func.py:10-11,19-20. */
int dist_nearest_sqdist(const float* ref, int64_t n_ref, const float* query, int64_t n_query, uint64_t* best, float* d2,
                        int32_t* index, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIST_B200_H_ */
