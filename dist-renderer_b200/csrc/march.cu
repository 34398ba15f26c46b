// Ray set-up, sphere tracing state machine, sample selection, normals and backward row generation.
//
// These are the per-ray (elementwise) parts of the path; every decoder evaluation goes through the engines in
// mlp_simt.cu / mlp_tc.cu.  Arithmetic mirrors the reference's op order (separately rounded mul/add where PyTorch
// issues separate elementwise ops): this file is compiled with -fmad=false and uses fmaf() only where the
// reference's op is a matmul.
//
// Reference: core/sdfrenderer/renderer.py:171-282 (rays, unit-sphere clip), :472-583 (marching), :304-420 (sample
// selection and depth estimate), :836-910 (render_depth / render_normal).
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>
#include "common.cuh"

namespace dist {
namespace {

struct Cam {
  float Kinv[9], M[9], Mn[9];
  const float* R;      // [n_views][9]
  const float* c;      // [n_views][3]
  int W, H, row0, row_step, n_rows, row_group;   // local row l is image row row0 + (l / row_group) * row_step + l % row_group
  int n_views, Pv;     // views rendered by this call, pixels per view (W * n_rows); global pixel lp = v * Pv + lpv
  float radius;
};

// per-view bookkeeping of a multi-view call (ws.view_stat, [n_views][4] int32): live rays at step 0, executed march
// steps (renderer.py:562 breaks per render, i.e. per view), float bits of the coarsest level's largest sphere entry
enum { LVL_APPROX = 0x80, LVL_REQUERIED = 0x40 };   // flag bits of ws.top_lvl (bits 0-1: pyramid level)
enum { VS_LIVE0 = 0, VS_STEPS = 1, VS_MAXENTRY = 2, VS_NONFINITE = 3, VS_STRIDE = 4 };

__device__ __forceinline__ void load_view(const Cam& cam, int v, float (&R)[9], float (&c)[3]) {
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = cam.R[9 * v + i];
#pragma unroll
  for (int i = 0; i < 3; ++i) c[i] = cam.c[3 * v + i];
}
__device__ __forceinline__ void load_view_pos(const Cam& cam, int v, float (&c)[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) c[i] = cam.c[3 * v + i];
}
// Row layout of the march's query arrays (ws.pts, ws.sdf, ws.list_a/b, ws.seg_approx): two segments of capacity
// SEG = round_up(P + 1, 128) each.  Segment 1 = rows [0, n1): rays predicted far from the surface, evaluated with one fp16
// pass first when dist_march_t.screen is on; segment 2 = rows [SEG, SEG + n2): everything else (and the origin query of step
// 0), always at full precision.  counts[2 s] / counts[2 s + 1] hold n1 / n2 of step s.
__host__ __device__ inline int seg_capacity(int P) { return (P + 1 + 127) / 128 * 128; }

// one atomic per (warp, view) instead of one per thread; every lane of the warp must call it (v < 0: nothing to add)
__device__ __forceinline__ void view_atomic_add(int32_t* view_stat, int slot, int v) {
  const unsigned peers = __match_any_sync(0xffffffffu, v);
  if (v >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(view_stat + VS_STRIDE * v + slot, __popc(peers));
}
__device__ __forceinline__ void view_atomic_max(int32_t* view_stat, int slot, int v, int value) {
  const unsigned peers = __match_any_sync(0xffffffffu, v);
  if (v >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicMax(view_stat + VS_STRIDE * v + slot, value);
}

__device__ __forceinline__ int warp_append(int32_t* counter, bool pred) {
  const unsigned m = __ballot_sync(0xffffffffu, pred);
  if (m == 0) return -1;
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(m) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(counter, __popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  return pred ? base + __popc(m & ((1u << lane) - 1)) : -1;
}

// two appends at once: counters[0] / counters[1] are adjacent (8-byte aligned) and advance with ONE 64-bit atomic per warp
__device__ __forceinline__ void warp_append2(int32_t* counters, bool p1, bool p2, int& idx1, int& idx2) {
  const unsigned m1 = __ballot_sync(0xffffffffu, p1), m2 = __ballot_sync(0xffffffffu, p2);
  idx1 = idx2 = -1;
  if ((m1 | m2) == 0) return;
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(m1 | m2) - 1;
  unsigned long long base = 0;
  if (lane == leader)
    base = atomicAdd(reinterpret_cast<unsigned long long*>(counters),
                     (unsigned long long)__popc(m1) | ((unsigned long long)__popc(m2) << 32));
  base = __shfl_sync(0xffffffffu, base, leader);
  const unsigned below = (1u << lane) - 1;
  if (p1) idx1 = (int)(uint32_t)base + __popc(m1 & below);
  if (p2) idx2 = (int)(uint32_t)(base >> 32) + __popc(m2 & below);
}

// unit ray through pixel coordinates (x, y), world frame (renderer.py:39,190-200; :631-636 for pyramid levels)
__device__ __forceinline__ void coord_ray(const Cam& cam, const float* R, float x, float y, float (&ray)[3]) {
  float hc[3], v[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) hc[i] = fmaf(cam.Kinv[i * 3 + 2], 1.f, fmaf(cam.Kinv[i * 3 + 1], y, cam.Kinv[i * 3] * x));
#pragma unroll
  for (int i = 0; i < 3; ++i) v[i] = fmaf(R[6 + i], hc[2], fmaf(R[3 + i], hc[1], R[i] * hc[0]));
  const float nrm = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]) + 1e-12f;
#pragma unroll
  for (int i = 0; i < 3; ++i) ray[i] = v[i] / nrm;
}
// image row of local row l of this call's band (interleaved groups of row_group rows, SURVEY 8e)
__device__ __forceinline__ int global_row(const Cam& cam, int l) {
  return cam.row0 + (l / cam.row_group) * cam.row_step + (l % cam.row_group);
}
// lpv: pixel index inside its view
__device__ __forceinline__ void pixel_ray(const Cam& cam, const float* R, int lpv, float (&ray)[3]) {
  coord_ray(cam, R, (float)(lpv % cam.W), (float)global_row(cam, lpv / cam.W), ray);
}

// unit-sphere geometry of one ray (renderer.py:225-282): distance to the origin, hit flag, entry and exit depth
__device__ __forceinline__ void sphere_geom(const float (&c)[3], const float (&ray)[3], float radius, float& dist, bool& hit,
                                            float& entry, float& ex) {
  const float ptq = (c[0] * ray[0] + c[1] * ray[1]) + c[2] * ray[2];
  const float d0 = c[0] - ptq * ray[0], d1 = c[1] - ptq * ray[1], d2 = c[2] - ptq * ray[2];
  dist = sqrtf(d0 * d0 + d1 * d1 + d2 * d2);
  hit = dist <= radius;
  const float value = radius * radius - dist * dist;
  const float chord = (value >= 0.f) ? 2.f * sqrtf(value) : 0.f;
  const float cd = sqrtf((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]);
  entry = (cd < radius) ? 0.f : sqrtf(cd * cd - dist * dist) - chord / 2.0f;
  ex = entry + chord;
}

// Insertion into the per-ray top-B records (the B samples with the smallest |sdf|; replaces topk over the step lists,
// renderer.py:316-319).  During the march the records are an UNORDERED set: a new sample replaces the record with the
// largest |sdf| if it beats it -- one pass over B values and one record write per sample instead of shifting a sorted list
// (the march update kernel is bound by exactly this traffic).  k_finalize sorts each ray's records once, ascending.
__device__ __forceinline__ void topk_insert(const dist_workspace_t& ws, int P, int B, int lp, float sdf, float px, float py,
                                            float pz, float zafter, float zgen, int lvl, int slot = -1) {
  const float asdf = fabsf(sdf);
  int pos = 0;
  float worst = -1.f;
  for (int b = 0; b < B; ++b) {
    const float a = fabsf(ws.top_sdf[(size_t)b * P + lp]);
    if (a >= worst) { worst = a; pos = b; }
  }
  if (!(asdf < worst)) return;
  ws.top_sdf[(size_t)pos * P + lp] = sdf;
  ws.top_zafter[(size_t)pos * P + lp] = zafter;
  ws.top_zgen[(size_t)pos * P + lp] = zgen;
  ws.top_lvl[(size_t)pos * P + lp] = (uint8_t)lvl;
  if (ws.top_slot) ws.top_slot[(size_t)pos * P + lp] = slot;      // mask-cache slot of the sample's decoder row (-1: none)
  ws.top_pt[((size_t)pos * 3 + 0) * P + lp] = px;
  ws.top_pt[((size_t)pos * 3 + 1) * P + lp] = py;
  ws.top_pt[((size_t)pos * 3 + 2) * P + lp] = pz;
}

// One coarse level of the pyramid (renderer.py:713-805): arrays carved from ws.pyr_{f,i,b}
struct Level {
  int w, h, Pv, P, scale;   // per-view w x h = Pv pixels, P = n_views * Pv; scale = 4 (1/4 resolution) or 2
  float *ray, *start, *z, *s_sdf, *s_pt, *s_zabs, *s_zgen;   // [3][P], [P], [P], [3][P], [3][3][P], [3][P], [3][P]
  uint8_t* hit;             // [P] max-pooled sphere-hit mask (renderer.py:668-680)
  int32_t* list;            // [P]
  int32_t* count;           // [1]
  int32_t* s_slot;          // [3][P] mask-cache slot of each recorded sample's decoder row (-1: none)
};

// p = M^T (c + ray * depth)   (renderer.py:202-223, :119)
__device__ __forceinline__ void point_on_ray(const Cam& cam, const float (&c)[3], const float (&ray)[3], float depth,
                                             float (&p)[3]) {
  float q[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) q[i] = ray[i] * depth + c[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) p[i] = fmaf(cam.M[6 + i], q[2], fmaf(cam.M[3 + i], q[1], cam.M[i] * q[0]));
}

__device__ __forceinline__ float clampf(float v, float c) { return fminf(fmaxf(v, -c), c); }

// ---------------------------------------------------------------------------------------------- set-up
// Thread -> pixel assignment of the set-up kernel: 16 x 8 pixel blocks, blocks row-major, view-major.  The initial active
// list (and, since compaction keeps the order, every later one) is therefore sorted by 2-D block, so a 128-row decoder
// tile holds one compact image patch: its rays are all far from the surface or all near it much more often than a
// 128-pixel strip of an image row -- which is what the two-tier precision of the decoder tiles (dist_march_t.screen) lives on.
constexpr int BLK_W = 16, BLK_H = 8;
__host__ __device__ inline int setup_threads_per_view(int W, int n_rows) {
  return ((W + BLK_W - 1) / BLK_W) * ((n_rows + BLK_H - 1) / BLK_H) * (BLK_W * BLK_H);
}

__global__ void k_setup(Cam cam, dist_march_t mp, dist_workspace_t ws, float* Zdepth, uint8_t* mask, float* min_sdf,
                        int P, Level L1, Level L2) {
  const int tpv = setup_threads_per_view(cam.W, cam.n_rows);
  const int gi = blockIdx.x * blockDim.x + threadIdx.x;
  const int vv = gi / tpv, r = gi - vv * tpv;
  const int wb = (cam.W + BLK_W - 1) / BLK_W;
  const int blk = r / (BLK_W * BLK_H), inb = r % (BLK_W * BLK_H);
  const int bx = (blk % wb) * BLK_W + inb % BLK_W, by = (blk / wb) * BLK_H + inb / BLK_W;
  const bool in = vv < cam.n_views && bx < cam.W && by < cam.n_rows;
  const int lp = in ? vv * cam.Pv + by * cam.W + bx : 0;
  const bool pyr = mp.marching_type == DIST_MARCH_PYRAMID;
  float R[9], c[3] = {0.f, 0.f, 0.f};
  const int v = in ? lp / cam.Pv : 0, lpv = lp - v * cam.Pv;
  bool live = false;
  float ray[3] = {0.f, 0.f, 1.f}, start = 0.f;
  if (in) {
    load_view(cam, v, R, c);
    pixel_ray(cam, R, lpv, ray);
    float dist, entry, ex;
    bool hit;
    sphere_geom(c, ray, cam.radius, dist, hit, entry, ex);
    start = entry;
    ws.ray[lp] = ray[0]; ws.ray[P + lp] = ray[1]; ws.ray[2 * P + lp] = ray[2];
    ws.exit_[lp] = ex; ws.dist[lp] = dist; ws.z[lp] = 0.f;
    ws.flags[lp] = hit ? 1 : 0;
    ws.nreal[lp] = 0;
    if (ws.sprev) ws.sprev[lp] = 0.f;
    for (int b = 0; b < mp.buffer_size; ++b) {
      ws.top_sdf[(size_t)b * P + lp] = 1.0f;  // filler entries: sdf 1, point 0 (renderer.py:539-540,555)
      ws.top_zafter[(size_t)b * P + lp] = 0.f;
      ws.top_zgen[(size_t)b * P + lp] = nanf("");
      ws.top_lvl[(size_t)b * P + lp] = 0;
      if (ws.top_slot) ws.top_slot[(size_t)b * P + lp] = -1;
#pragma unroll
      for (int k = 0; k < 3; ++k) ws.top_pt[((size_t)b * 3 + k) * P + lp] = 0.f;
    }
    if (pyr) {
      // the full-resolution march starts at the parent's last depth (renderer.py:769) and inherits the samples taken
      // on the grandparent and parent rays (index up-sampling, renderer.py:787-801)
      const int x = lpv % cam.W, y = lpv / cam.W;
      const int p1 = v * L1.Pv + (y >> 1) * L1.w + (x >> 1), p2 = v * L2.Pv + (y >> 2) * L2.w + (x >> 2);
      start = L1.start[p1] + (L1.hit[p1] ? L1.z[p1] : 0.f);
      if (hit) {
        for (int lv = 2; lv >= 1; --lv) {
          const Level& L = (lv == 2) ? L2 : L1;
          const int pp = (lv == 2) ? p2 : p1;
          if (!L.hit[pp]) continue;
          const int ns = mp.coarse_steps[2 - lv];
          for (int st = 0; st < ns; ++st)
            topk_insert(ws, P, mp.buffer_size, lp, L.s_sdf[(size_t)st * L.P + pp], L.s_pt[((size_t)st * 3 + 0) * L.P + pp],
                        L.s_pt[((size_t)st * 3 + 1) * L.P + pp], L.s_pt[((size_t)st * 3 + 2) * L.P + pp],
                        L.s_zabs[(size_t)st * L.P + pp] - entry, L.s_zgen[(size_t)st * L.P + pp], lv,
                        L.s_slot[(size_t)st * L.P + pp]);
        }
      }
    }
    ws.entry[lp] = start; ws.entry0[lp] = entry;
    if (!hit) {
      Zdepth[lp] = 1e11f; mask[lp] = 0;
      min_sdf[lp] = dist + mp.threshold - cam.radius;  // renderer.py:863
    }
    live = hit && (mp.marching_type == DIST_MARCH_TRIVIAL || (0.f + start < ex));  // renderer.py:526
  }
  view_atomic_add(ws.view_stat, VS_LIVE0, live ? v : -1);
  const int idx = warp_append(ws.counts + 0, live);
  if (idx >= 0) {
    float p[3];
    point_on_ray(cam, c, ray, start + 0.f, p);
    ws.list_a[idx] = lp;
    ws.pts[(size_t)idx * 3] = p[0]; ws.pts[(size_t)idx * 3 + 1] = p[1]; ws.pts[(size_t)idx * 3 + 2] = p[2];
  }
}

// sphere-hit flags of the full image only (needed before the pyramid levels can be pooled)
__global__ void k_hit_flags(Cam cam, dist_workspace_t ws, int P) {
  const int lp = blockIdx.x * blockDim.x + threadIdx.x;
  if (lp >= P) return;
  float R[9], c[3], ray[3], dist, entry, ex;
  bool hit;
  const int v = lp / cam.Pv;
  load_view(cam, v, R, c);
  pixel_ray(cam, R, lp - v * cam.Pv, ray);
  sphere_geom(c, ray, cam.radius, dist, hit, entry, ex);
  ws.flags[lp] = hit ? 1 : 0;
}

// coarse level: rays through the pooled pixel centres, own sphere entry, max-pooled hit mask (renderer.py:604-680)
__global__ void k_pyr_rays(Cam cam, Level L, const uint8_t* fine_hit, int fine_w, int fine_h, int32_t* view_stat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.P) return;
  const int v = i / L.Pv, il = i - v * L.Pv;
  const int ix = il % L.w, iy = il / L.w;
  float R[9], c[3], ray[3], dist, entry, ex;
  bool ownhit;
  load_view(cam, v, R, c);
  const float off = ((float)L.scale - 1.f) / 2.f;
  // the L.scale fine rows pooled into coarse row iy are consecutive image rows (row_group is a multiple of 4 on bands)
  coord_ray(cam, R, (float)L.scale * (float)ix + off, (float)global_row(cam, L.scale * iy) + off, ray);
  sphere_geom(c, ray, cam.radius, dist, ownhit, entry, ex);
  L.ray[i] = ray[0]; L.ray[L.P + i] = ray[1]; L.ray[2 * L.P + i] = ray[2];
  bool pooled = false;
  for (int dy = 0; dy < 2; ++dy)
    for (int dx = 0; dx < 2; ++dx) {
      const int fx = 2 * ix + dx, fy = 2 * iy + dy;
      if (fx < fine_w && fy < fine_h) pooled |= (fine_hit[(size_t)v * fine_w * fine_h + fy * fine_w + fx] & 1) != 0;
    }
  L.hit[i] = pooled ? 1 : 0;
  L.z[i] = 0.f;
  // coarsest level: own entry where the coarse ray meets the sphere, else the largest entry of those that do
  // (renderer.py:270-272); stash the own entry, resolve after the max is known
  L.start[i] = ownhit ? entry : -1.f;
  if (view_stat && ownhit) atomicMax(view_stat + VS_STRIDE * v + VS_MAXENTRY, __float_as_int(fmaxf(entry, 0.f)));
}

// Row bands: the fill value of renderer.py:270-272 is the largest sphere entry over the coarsest level of the WHOLE image,
// not of this rank's band.  Geometry only (no decoder rows): every rank evaluates the full 1/4-resolution grid.
__global__ void k_pyr_global_maxentry(Cam cam, int w2, int h2, int32_t* view_stat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = w2 * h2;
  if (i >= n * cam.n_views) return;
  const int v = i / n, il = i - v * n;
  float R[9], c[3], ray[3], dist, entry, ex;
  bool hit;
  load_view(cam, v, R, c);
  coord_ray(cam, R, 4.f * (float)(il % w2) + 1.5f, 4.f * (float)(il / w2) + 1.5f, ray);
  sphere_geom(c, ray, cam.radius, dist, hit, entry, ex);
  if (hit) atomicMax(view_stat + VS_STRIDE * v + VS_MAXENTRY, __float_as_int(fmaxf(entry, 0.f)));
}

// start depth of a coarse level + its (fixed) active list and first query points
__global__ void k_pyr_start(Cam cam, Level L, Level parent, int has_parent, const int32_t* view_stat, float* pts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool on = false;
  float start = 0.f;
  const int v = (i < L.P) ? i / L.Pv : 0;
  if (i < L.P) {
    if (has_parent) {
      const int il = i - v * L.Pv;
      const int ix = il % L.w, iy = il / L.w, pp = v * parent.Pv + (iy >> 1) * parent.w + (ix >> 1);
      start = parent.start[pp] + (parent.hit[pp] ? parent.z[pp] : 0.f);   // renderer.py:769,779
    } else {
      start = (L.start[i] >= 0.f) ? L.start[i] : __int_as_float(view_stat[VS_STRIDE * v + VS_MAXENTRY]);
    }
    L.start[i] = start;
    on = L.hit[i] != 0;
  }
  const int idx = warp_append(L.count, on);
  if (idx >= 0) {
    float c[3], ray[3] = {L.ray[i], L.ray[L.P + i], L.ray[2 * L.P + i]}, p[3];
    load_view_pos(cam, v, c);
    point_on_ray(cam, c, ray, start + 0.f, p);
    L.list[idx] = i;
    pts[(size_t)idx * 3] = p[0]; pts[(size_t)idx * 3 + 1] = p[1]; pts[(size_t)idx * 3 + 2] = p[2];
  }
}

// one trivial march step of a coarse level (renderer.py:472-510 via :773): every listed ray advances, samples are
// recorded per (step, ray); the query point of the next step overwrites this thread's own slot
__global__ void k_pyr_step(Cam cam, dist_march_t mp, Level L, int step, float* pts, const float* sdfbuf, int64_t slot_base,
                           int64_t slot_cap) {
  const int n = *L.count;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int id = L.list[i];
    // (the decoder launch of this step recorded row i at mask-cache slot slot_base + i; < 0: cache off)
    L.s_slot[(size_t)step * L.P + id] = (slot_base >= 0 && slot_base + i < slot_cap) ? (int32_t)(slot_base + i) : -1;
    float c[3];
    load_view_pos(cam, id / L.Pv, c);
    const float sdf = sdfbuf[i];
    const float zc = L.z[id], start = L.start[id];
    const float znew = zc + clampf(sdf, mp.clamp_dist) * mp.ratio;
    L.z[id] = znew;
    L.s_sdf[(size_t)step * L.P + id] = sdf;
#pragma unroll
    for (int k = 0; k < 3; ++k) L.s_pt[((size_t)step * 3 + k) * L.P + id] = pts[(size_t)i * 3 + k];
    L.s_zabs[(size_t)step * L.P + id] = znew + start;     // renderer.py:779
    L.s_zgen[(size_t)step * L.P + id] = start + zc;
    float ray[3] = {L.ray[id], L.ray[L.P + id], L.ray[2 * L.P + id]}, p[3];
    point_on_ray(cam, c, ray, start + znew, p);
    pts[(size_t)i * 3] = p[0]; pts[(size_t)i * 3 + 1] = p[1]; pts[(size_t)i * 3 + 2] = p[2];
  }
}

// the origin (filler samples, renderer.py:539-540) is the only row of segment 2 at step 0: always at full precision.
// With one latent code per view there is one origin row per view (n_origin = n_views), listed as pixel v * Pv so that the
// row's code is its view like every other row of the march.
__global__ void k_append_origin(dist_workspace_t ws, int SEG, int mask_slots_used, int n_origin, int Pv) {
  for (int o = threadIdx.x; o < n_origin; o += blockDim.x) {
    const size_t r = (size_t)SEG + o;
    ws.pts[r * 3] = 0.f; ws.pts[r * 3 + 1] = 0.f; ws.pts[r * 3 + 2] = 0.f;
    ws.list_a[r] = o * Pv;
  }
  if (threadIdx.x == 0) {
    ws.counts[1] = n_origin;
    if (ws.mask_base) ws.mask_base[0] = mask_slots_used;    // the coarse pyramid levels recorded their rows before the march
  }
}

// ---------------------------------------------------------------------------------------------- one march step
__global__ void k_march_update(Cam cam, dist_march_t mp, dist_workspace_t ws, int step, int P, int n_origin) {
  const int SEG = seg_capacity(P);
  const int n1 = ws.counts[2 * step];
  const int n2 = (step == 0) ? 0 : ws.counts[2 * step + 1];      // (step 0: segment 2 holds the origin query only)
  const int n = n1 + n2;
  const bool scr = ws.seg_approx != nullptr;
  const int32_t* cur = (step & 1) ? ws.list_b : ws.list_a;
  int32_t* nxt = (step & 1) ? ws.list_a : ws.list_b;
  const float* pts_cur = ws.pts + (size_t)(step & 1) * (size_t)(2 * SEG) * 3;       // points of this step
  float* pts_nxt = ws.pts + (size_t)((step + 1) & 1) * (size_t)(2 * SEG) * 3;       // points of the next step
  if (step == 0 && blockIdx.x == 0)
    for (int o = threadIdx.x; o < n_origin; o += blockDim.x) ws.sdf_origin[o] = ws.sdf[SEG + o];   // (one per view: per-view codes)
  // mask cache: the decoder launch of this step recorded the rows of segment 2 at slots mask_base[step] + (i - SEG)
  const bool mc = scr && ws.mask_buf != nullptr;
  const int mbase = mc ? ws.mask_base[step] : 0;
  if (mc && blockIdx.x == 0 && threadIdx.x == 0)
    ws.mask_base[step + 1] = mbase + (ws.counts[2 * step + 1] + 127) / 128 * 128;   // (slots are handed out tile by tile)
  const int B = mp.buffer_size;
  const float far_thresh = mp.clamp_dist + mp.screen_margin;
  for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const int j = base + threadIdx.x;
    bool live = false, approx = false, pred_far = false;
    int lp = 0, v = -1;
    float znew = 0.f, entry = 0.f;
    if (j < n) {
      const int i = (j < n1) ? j : SEG + (j - n1);
      lp = cur[i];
      v = lp / cam.Pv;
      const float sdf = ws.sdf[i];
      const float px = pts_cur[(size_t)i * 3], py = pts_cur[(size_t)i * 3 + 1], pz = pts_cur[(size_t)i * 3 + 2];
      const float zc = ws.z[lp];
      entry = ws.entry[lp];
      znew = zc + clampf(sdf, mp.clamp_dist) * mp.ratio;  // renderer.py:548-551
      ws.z[lp] = znew;
      ws.nreal[lp] = step + 1;
      if (step == 0 && sdf > mp.threshold) ws.flags[lp] |= 2;  // renderer.py:581
      const float asdf = fabsf(sdf);
      approx = scr && ws.seg_approx[i >> 6] != 0;   // one-pass value: |sdf| > clamp + margin is all that is known exactly
      if (scr) {
        // Will the next sample of this ray be beyond the clamp band again?  Yes if this one is far beyond it (the march
        // moves by ratio * clamp per step), or if the linear extrapolation of the last two samples stays beyond it with a
        // safety margin.  A wrong "yes" costs a re-evaluation of one tile, never a wrong value.
        const float ext = sdf + (sdf - ws.sprev[lp]);
        pred_far = asdf > mp.screen_tpred ||
                   (step >= 1 && asdf > far_thresh && fabsf(ext) > far_thresh + mp.screen_ext_margin && (ext > 0.f) == (sdf > 0.f));
        ws.sprev[lp] = sdf;
      }
      // a tanh output is in [-1, 1]: anything else is an overflow of the engine's operands (fp16 range of the tensor-core
      // engine) -- flagged per view, raised by the host when it reads view_stat back
      if (!(asdf <= 1.0f)) atomicOr(ws.view_stat + VS_STRIDE * v + VS_NONFINITE, 1);
      // marching depth relative to the true sphere entry (renderer.py:800-804 for the pyramid variant)
      const float zstore = (mp.marching_type == DIST_MARCH_PYRAMID) ? (znew + entry) - ws.entry0[lp] : znew;
      int slot = -1;
      if (mc && i >= SEG && (int64_t)mbase + (i - SEG) < ws.mask_cap) slot = mbase + (i - SEG);
      topk_insert(ws, P, B, lp, sdf, px, py, pz, zstore, entry + zc, approx ? LVL_APPROX : 0, slot);
      if (step + 1 < mp.march_step) {
        if (mp.marching_type == DIST_MARCH_TRIVIAL) live = true;
        else live = (znew + entry < ws.exit_[lp]) && (asdf >= mp.threshold);  // renderer.py:559-561
      }
    }
    view_atomic_max(ws.view_stat, VS_STEPS, v, step + 1);   // view v executed this step
    // compaction into the next step's two segments (without screening everything goes to segment 1)
    const bool to1 = live && (!scr || pred_far), to2 = live && !to1;
    // the next query point does not depend on where the row lands: it is computed before the atomic, not behind it
    float p[3] = {0.f, 0.f, 0.f};
    if (live) {
      float ray[3] = {ws.ray[lp], ws.ray[P + lp], ws.ray[2 * P + lp]}, c[3];
      load_view_pos(cam, v, c);
      point_on_ray(cam, c, ray, entry + znew, p);
    }
    int idx, idx2;
    warp_append2(ws.counts + 2 * (step + 1), to1, to2, idx, idx2);
    if (idx2 >= 0) idx = SEG + idx2;
    if (idx >= 0) {
      nxt[idx] = lp;
      pts_nxt[(size_t)idx * 3] = p[0]; pts_nxt[(size_t)idx * 3 + 1] = p[1]; pts_nxt[(size_t)idx * 3 + 2] = p[2];
    }
  }
}

// ---------------------------------------------------------------------------------------------- exact re-query
// Two-tier precision: the recorded sdf of a sample evaluated with one pass is accurate to E = screen_margin / 2 and known to
// lie beyond the clamp.  That is enough everywhere (clamped value +-clamp_dist, zero gradient coefficient) except for the
// ray's SMALLEST |sdf| -- min_sdf (renderer.py:382-390) and the depth estimate (:407-408) use its value.  Every one-pass
// record that could be the true minimum (its lower bound is below the smallest upper bound) is re-evaluated at full precision.
__global__ void k_requery_gen(dist_march_t mp, dist_workspace_t ws, int P) {
  const int lp = blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = lp < P && (ws.flags[lp] & 1);
  const int B = mp.buffer_size;
  const float E = 0.5f * mp.screen_margin;
  float U = 3.0e38f;
  if (on)
    for (int b = 0; b < B; ++b)
      U = fminf(U, fabsf(ws.top_sdf[(size_t)b * P + lp]) + ((ws.top_lvl[(size_t)b * P + lp] & LVL_APPROX) ? E : 0.f));
  for (int b = 0; b < B; ++b) {
    const bool cand = on && (ws.top_lvl[(size_t)b * P + lp] & LVL_APPROX) && (fabsf(ws.top_sdf[(size_t)b * P + lp]) - E <= U);
    const int idx = warp_append(ws.rq_cnt, cand);
    if (idx >= 0) {
      ws.rq_idx[idx] = lp * DIST_MAX_BUFFER + b;
#pragma unroll
      for (int k = 0; k < 3; ++k) ws.rq_pts[(size_t)idx * 3 + k] = ws.top_pt[((size_t)b * 3 + k) * P + lp];
    }
  }
}

__global__ void k_requery_apply(dist_workspace_t ws, int P, int base_index) {
  const int n = *ws.rq_cnt;
  const bool mc = ws.mask_buf != nullptr && ws.top_slot != nullptr;
  const int mbase = mc ? ws.mask_base[base_index] : 0;      // the re-query launch recorded its rows at mbase + i
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int lp = ws.rq_idx[i] / DIST_MAX_BUFFER, b = ws.rq_idx[i] % DIST_MAX_BUFFER;
    ws.top_sdf[(size_t)b * P + lp] = ws.rq_sdf[i];
    if (mc) ws.top_slot[(size_t)b * P + lp] = ((int64_t)mbase + i < ws.mask_cap) ? mbase + i : -1;
    ws.top_lvl[(size_t)b * P + lp] = (uint8_t)((ws.top_lvl[(size_t)b * P + lp] & ~LVL_APPROX) | LVL_REQUERIED);
  }
}

// ---------------------------------------------------------------------------------------------- finalize
__global__ void k_finalize(dist_march_t mp, dist_workspace_t ws, float* Zdepth, uint8_t* mask, float* min_sdf, int P, int Pv,
                           int origin_per_view) {
  const int lp = blockIdx.x * blockDim.x + threadIdx.x;
  if (lp >= P || !(ws.flags[lp] & 1)) return;
  const int B = mp.buffer_size;
  // steps this ray's view executed before all of its rays had finished (the early break of renderer.py:562 is per render)
  const int S = ws.view_stat[VS_STRIDE * (lp / Pv) + VS_STEPS];
  int nreal = ws.nreal[lp];
  const float so = ws.sdf_origin[origin_per_view ? lp / Pv : 0];
  const float zfin = ws.z[lp];
  // renderer.py:562-567: an early break of the (full-resolution) march before buffer_size steps pads its lists with
  // copies of the last executed step; in the pyramid variant the padded fine-level lists are then concatenated with the
  // coarse samples (renderer.py:795-801), so the copies compete with those for the top-B slots
  if (S < B && nreal == S && nreal > 0) {
    const float zkey = (mp.marching_type == DIST_MARCH_PYRAMID) ? (zfin + ws.entry[lp]) - ws.entry0[lp] : zfin;
    int j = -1;
    for (int b = 0; b < B; ++b)
      if (ws.top_zafter[(size_t)b * P + lp] == zkey && (ws.top_lvl[(size_t)b * P + lp] & 3) == 0 &&
          ws.top_sdf[(size_t)b * P + lp] != 1.0f) j = b;
    if (j >= 0) {   // (evicted already: its copies would not enter either)
      const float r_sdf = ws.top_sdf[(size_t)j * P + lp], r_za = ws.top_zafter[(size_t)j * P + lp],
                  r_zg = ws.top_zgen[(size_t)j * P + lp];
      const float r_p[3] = {ws.top_pt[((size_t)j * 3 + 0) * P + lp], ws.top_pt[((size_t)j * 3 + 1) * P + lp],
                            ws.top_pt[((size_t)j * 3 + 2) * P + lp]};
      const int r_lvl = ws.top_lvl[(size_t)j * P + lp];
      const int r_slot = ws.top_slot ? ws.top_slot[(size_t)j * P + lp] : -1;
      for (int i = 0; i < B - S; ++i) topk_insert(ws, P, B, lp, r_sdf, r_p[0], r_p[1], r_p[2], r_za, r_zg, r_lvl, r_slot);
    }
    nreal = B;
    ws.nreal[lp] = B;
  }
  {   // the records are an unordered set until here: ascending |sdf| (stable), the minimum to slot 0 (renderer.py:316-319).
      // The insertion sort runs on the keys in registers (the same comparisons in the same order as sorting the records
      // themselves); every field is then read once and written once in its sorted place.
    float key[DIST_MAX_BUFFER];
    int ord[DIST_MAX_BUFFER];
#pragma unroll
    for (int b = 0; b < DIST_MAX_BUFFER; ++b) {
      key[b] = (b < B) ? fabsf(ws.top_sdf[(size_t)b * P + lp]) : 0.f;
      ord[b] = b;
    }
    bool moved = false;
#pragma unroll
    for (int a = 1; a < DIST_MAX_BUFFER; ++a) {
      if (a < B) {
        bool go = true;
#pragma unroll
        for (int b = a; b > 0; --b) {
          go = go && (key[b] < key[b - 1]);
          if (go) {
            const float tk = key[b]; key[b] = key[b - 1]; key[b - 1] = tk;
            const int to = ord[b]; ord[b] = ord[b - 1]; ord[b - 1] = to;
            moved = true;
          }
        }
      }
    }
    if (moved) {
      // out[d] = in[ord[d]] without dynamic register indexing
      auto permute_f = [&](float* base, size_t stride) {
        float v[DIST_MAX_BUFFER];
#pragma unroll
        for (int b = 0; b < DIST_MAX_BUFFER; ++b) v[b] = (b < B) ? base[(size_t)b * stride + lp] : 0.f;
#pragma unroll
        for (int d = 0; d < DIST_MAX_BUFFER; ++d) {
          if (d < B && ord[d] != d) {
            float o = 0.f;
#pragma unroll
            for (int sidx = 0; sidx < DIST_MAX_BUFFER; ++sidx) o = (ord[d] == sidx) ? v[sidx] : o;
            base[(size_t)d * stride + lp] = o;
          }
        }
      };
      permute_f(ws.top_sdf, (size_t)P);
      permute_f(ws.top_zafter, (size_t)P);
      permute_f(ws.top_zgen, (size_t)P);
      for (int k = 0; k < 3; ++k) permute_f(ws.top_pt + (size_t)k * P, (size_t)3 * P);
      {
        int v[DIST_MAX_BUFFER];
#pragma unroll
        for (int b = 0; b < DIST_MAX_BUFFER; ++b) v[b] = (b < B) ? (int)ws.top_lvl[(size_t)b * P + lp] : 0;
#pragma unroll
        for (int d = 0; d < DIST_MAX_BUFFER; ++d) {
          if (d < B && ord[d] != d) {
            int o = 0;
#pragma unroll
            for (int sidx = 0; sidx < DIST_MAX_BUFFER; ++sidx) o = (ord[d] == sidx) ? v[sidx] : o;
            ws.top_lvl[(size_t)d * P + lp] = (uint8_t)o;
          }
        }
      }
      if (ws.top_slot) {
        int v[DIST_MAX_BUFFER];
#pragma unroll
        for (int b = 0; b < DIST_MAX_BUFFER; ++b) v[b] = (b < B) ? ws.top_slot[(size_t)b * P + lp] : -1;
#pragma unroll
        for (int d = 0; d < DIST_MAX_BUFFER; ++d) {
          if (d < B && ord[d] != d) {
            int o = -1;
#pragma unroll
            for (int sidx = 0; sidx < DIST_MAX_BUFFER; ++sidx) o = (ord[d] == sidx) ? v[sidx] : o;
            ws.top_slot[(size_t)d * P + lp] = o;
          }
        }
      }
    }
  }
  const float s0 = ws.top_sdf[lp];
  const float entry = ws.entry[lp];
  const bool real0 = (s0 != 1.0f);   // a filler record has sdf exactly 1 (tanh output is < 1)
  const bool first_ok = (nreal == 0) || (ws.flags[lp] & 2);
  const bool valid = (zfin + entry < ws.exit_[lp]) && (fabsf(s0) <= mp.threshold) &&
                     (!mp.first_query_check || first_ok);  // renderer.py:574-582
  min_sdf[lp] = real0 ? s0 : so;  // renderer.py:382-390 (value of the re-query at the min-|sdf| point)
  // renderer.py:407-408
  float zz = ws.top_zafter[lp] + (1.f - mp.ratio) * clampf(s0, mp.clamp_dist);
  // renderer.py:414-417: z - s.detach()*ratio + s*ratio, value-neutral up to rounding; per view (bit v, bit 31 = every view):
  // a view rendered with no_grad_depth skips the additions (renderer.py:413), and its last bit with them
  const int vw = lp / Pv;
  if ((mp.replay_grad_rounding >> 31) & 1 || (vw < 31 && ((mp.replay_grad_rounding >> vw) & 1))) {
    for (int b = 0; b < B; ++b) {
      const float sb = ws.top_sdf[(size_t)b * P + lp];
      const float s = clampf((sb != 1.0f) ? sb : so, mp.clamp_dist);
      const float a = s * mp.ratio;
      zz = zz - a;
      zz = zz + a;
    }
  }
  Zdepth[lp] = ws.entry0[lp] + zz;  // renderer.py:868
  mask[lp] = valid ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------- normals
__global__ void k_normal_gen(Cam cam, const float* Zdepth, const uint8_t* mask, int32_t* idx_out, float* pts,
                             int32_t* count, int P) {
  const int lp = blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = lp < P && mask[lp] != 0;
  const int idx = warp_append(count, on);
  if (idx >= 0) {
    float R[9], c[3], ray[3], p[3];
    const int v = lp / cam.Pv;
    load_view(cam, v, R, c);
    pixel_ray(cam, R, lp - v * cam.Pv, ray);
    point_on_ray(cam, c, ray, Zdepth[lp], p);
    idx_out[idx] = lp;
    pts[(size_t)idx * 3] = p[0]; pts[(size_t)idx * 3 + 1] = p[1]; pts[(size_t)idx * 3 + 2] = p[2];
  }
}

__global__ void k_normal_finish(Cam cam, const int32_t* idx_in, const float* grad, const int32_t* count, int normalize,
                                float* Znormal, int P) {
  const int n = *count;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int lp = idx_in[i];
    float g[3] = {grad[(size_t)i * 3], grad[(size_t)i * 3 + 1], grad[(size_t)i * 3 + 2]};
    if (normalize) {  // renderer.py:171-178
      const float nrm = sqrtf(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]) + 1e-12f;
      g[0] = g[0] / nrm; g[1] = g[1] / nrm; g[2] = g[2] / nrm;
    }
#pragma unroll
    for (int k = 0; k < 3; ++k)  // renderer.py:97 transform_matrix @ n
      Znormal[(size_t)k * P + lp] = fmaf(cam.Mn[k * 3 + 2], g[2], fmaf(cam.Mn[k * 3 + 1], g[1], cam.Mn[k * 3] * g[0]));
  }
}

// ---------------------------------------------------------------------------------------------- backward rows
// Replay rows of the backward: one per selected sample with a non-zero upstream coefficient.  Samples whose decoder row left
// its ReLU masks in the mask cache (ws.top_slot >= 0) go to the "masked" list (ws.bm_*: transposed chain only), the others
// (fillers, coarse pyramid samples, rows of re-evaluated tiles, everything when the cache is off) to the full replay list.
__global__ void k_bwd_gen(dist_march_t mp, dist_workspace_t ws, const float* gZ, const float* gM, int32_t* row_pix,
                          float* pts, float* coef, int32_t* count, int P, int use_masks, int Pv, int origin_per_view) {
  const int lp = blockIdx.x * blockDim.x + threadIdx.x;
  const bool hit = lp < P && (ws.flags[lp] & 1);
  const int B = mp.buffer_size;
  const float so = hit ? ws.sdf_origin[origin_per_view ? lp / Pv : 0] : 0.f;
  const float gz = (hit && gZ) ? gZ[lp] : 0.f;
  const float gm = (hit && gM) ? gM[lp] : 0.f;
  for (int b = 0; b < B; ++b) {
    float cf = 0.f, s = 0.f;
    int slot = -1;
    if (hit) {
      const float sb = ws.top_sdf[(size_t)b * P + lp];
      s = (sb != 1.0f) ? sb : so;
      const bool cm = (s >= -mp.clamp_dist) && (s <= mp.clamp_dist);
      cf = cm ? mp.ratio * gz : 0.f;  // renderer.py:414-417
      if (b == 0) cf += gm;           // renderer.py:386 (unclamped re-query at the min-|sdf| sample)
      if (use_masks && sb != 1.0f) slot = ws.top_slot[(size_t)b * P + lp];
    }
    const int idx = warp_append(count, cf != 0.f && slot < 0);
    if (idx >= 0) {
      row_pix[idx] = lp * DIST_MAX_BUFFER + b;
      coef[idx] = cf;
#pragma unroll
      for (int k = 0; k < 3; ++k) pts[(size_t)idx * 3 + k] = ws.top_pt[((size_t)b * 3 + k) * P + lp];
    }
    if (use_masks) {
      const int im = warp_append(ws.bm_cnt, cf != 0.f && slot >= 0);
      if (im >= 0) { ws.bm_row[im] = lp * DIST_MAX_BUFFER + b; ws.bm_slot[im] = slot; ws.bm_sdf[im] = s; ws.bm_coef[im] = cf; }
    }
  }
}

__global__ void k_bwd_scatter(Cam cam, dist_workspace_t ws, const int32_t* row_pix, const float* dpts,
                              const int32_t* count, float* d_cam, float* d_ray, float* d_ray_coarse, int w1, int P1v, int w2,
                              int P2v, int P, int cam_levels) {
  const int n = *count;
  const size_t P1 = (size_t)cam.n_views * P1v, P2 = (size_t)cam.n_views * P2v;
  // d_cam[v] accumulates per thread while consecutive rows stay in one view (rows are generated in pixel order)
  float acc[3] = {0.f, 0.f, 0.f};
  int acc_v = -1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int lp = row_pix[i] / DIST_MAX_BUFFER, b = row_pix[i] % DIST_MAX_BUFFER;
    const float zg = ws.top_zgen[(size_t)b * P + lp];
    if (zg != zg) continue;  // filler / off-ray sample: no camera dependence
    const int lvl = ws.top_lvl[(size_t)b * P + lp] & 3;
    // which samples keep their camera graph: bit 0 the full-resolution march (detached under no_grad_camera,
    // renderer.py:536-537,543-544), bit 1 the trivial marches of the coarse pyramid levels (never detached, :481-484)
    if (!((cam_levels >> (lvl ? 1 : 0)) & 1)) continue;
    const int v = lp / cam.Pv, lpv = lp - v * cam.Pv;
    if (v != acc_v) {
      if (acc_v >= 0)
        for (int k = 0; k < 3; ++k)
          if (acc[k] != 0.f) atomicAdd(d_cam + 3 * acc_v + k, acc[k]);
      acc[0] = acc[1] = acc[2] = 0.f;
      acc_v = v;
    }
    const float d[3] = {dpts[(size_t)i * 3], dpts[(size_t)i * 3 + 1], dpts[(size_t)i * 3 + 2]};
#pragma unroll
    for (int k = 0; k < 3; ++k) {  // p = M^T q  ->  dL/dq = M dL/dp
      const float g = fmaf(cam.M[k * 3 + 2], d[2], fmaf(cam.M[k * 3 + 1], d[1], cam.M[k * 3] * d[0]));
      acc[k] += g;
      if (lvl == 0) atomicAdd(d_ray + (size_t)k * P + lp, g * zg);
      else if (d_ray_coarse) {   // sample taken on the parent (1/2) or grandparent (1/4 resolution) ray
        const int x = lpv % cam.W, y = lpv / cam.W;
        if (lvl == 1) atomicAdd(d_ray_coarse + (size_t)k * P1 + (size_t)v * P1v + (y >> 1) * w1 + (x >> 1), g * zg);
        else atomicAdd(d_ray_coarse + 3 * P1 + (size_t)k * P2 + (size_t)v * P2v + (y >> 2) * w2 + (x >> 2), g * zg);
      }
    }
  }
  // flush: one atomic per warp when the whole warp ended in the same view, else one per thread
  const unsigned same = __match_any_sync(0xffffffffu, acc_v);
  const bool uniform = (same == 0xffffffffu);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float t = acc[k];
    if (uniform) {
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if ((threadIdx.x & 31) == 0 && acc_v >= 0 && t != 0.f) atomicAdd(d_cam + 3 * acc_v + k, t);
    } else if (acc_v >= 0 && t != 0.f) {
      atomicAdd(d_cam + 3 * acc_v + k, t);
    }
  }
}

int make_cam(const dist_camera_t* cam, Cam* out) {
  DIST_REQUIRE(cam && cam->R && cam->cam_pos, "camera: null pointer");
  DIST_REQUIRE(cam->width > 0 && cam->n_rows > 0 && cam->row_step > 0, "camera: bad image/tile description");
  const int n_views = cam->n_views > 0 ? cam->n_views : 1;
  DIST_REQUIRE((int64_t)cam->width * cam->n_rows * n_views < (int64_t)(1u << 31) / DIST_MAX_BUFFER, "camera: tile too large");
  for (int i = 0; i < 9; ++i) { out->Kinv[i] = cam->Kinv[i]; out->M[i] = cam->M[i]; out->Mn[i] = cam->Mn[i]; }
  out->R = cam->R; out->c = cam->cam_pos;
  out->W = cam->width; out->H = cam->height; out->row0 = cam->row0; out->row_step = cam->row_step;
  out->n_rows = cam->n_rows; out->radius = cam->radius;
  out->row_group = cam->row_group > 0 ? cam->row_group : 1;
  DIST_REQUIRE(cam->row0 >= 0 && cam->row0 + ((cam->n_rows - 1) / out->row_group) * cam->row_step + (cam->n_rows - 1) % out->row_group < cam->height,
               "camera: row band outside the image");
  out->n_views = n_views; out->Pv = cam->width * cam->n_rows;
  return DIST_OK;
}

// one latent code per view (dist_net_t.n_codes > 1): the code of a decoder row is the view of its pixel
int check_codes(const NetDev& nd, const Cam& cam) {
  DIST_REQUIRE(nd.n_codes <= 1 || nd.n_codes == cam.n_views, "net: n_codes = %d, but the call renders %d views", nd.n_codes,
               cam.n_views);
  return DIST_OK;
}
// rows whose array entries are pixels (active lists, normal rows) or pixel * DIST_MAX_BUFFER + record (re-query, backward rows)
void set_codes(const NetDev& nd, MlpArgs& a, const int32_t* rows, int div) {
  if (nd.n_codes > 1) { a.row_code = rows; a.code_div = div; }
}

}  // namespace

// =============================================================================================== host entry points
static void carve_levels(const Cam& cam, const dist_workspace_t* ws, Level* L1, Level* L2) {
  Level* Ls[2] = {L1, L2};
  int w = cam.W, h = cam.n_rows;
  float* f = ws->pyr_f;
  int32_t* li = ws->pyr_i;
  uint8_t* bb = ws->pyr_b;
  const int w1 = (w + 1) / 2, h1 = (h + 1) / 2, w2 = (w1 + 1) / 2, h2 = (h1 + 1) / 2;
  const int dims[2][2] = {{w1, h1}, {w2, h2}};
  // pyr_i: [lists P1 + P2][slots 3 (P1 + P2)][8 counters]
  int32_t* slots = li + ((size_t)w1 * h1 + (size_t)w2 * h2) * cam.n_views;
  int32_t* counts = li + 4 * ((size_t)w1 * h1 + (size_t)w2 * h2) * cam.n_views;
  for (int i = 0; i < 2; ++i) {
    Level& L = *Ls[i];
    L.w = dims[i][0]; L.h = dims[i][1]; L.Pv = L.w * L.h; L.P = L.Pv * cam.n_views; L.scale = (i == 0) ? 2 : 4;
    L.ray = f; f += 3 * (size_t)L.P;
    L.start = f; f += L.P;
    L.z = f; f += L.P;
    L.s_sdf = f; f += 3 * (size_t)L.P;
    L.s_pt = f; f += 9 * (size_t)L.P;
    L.s_zabs = f; f += 3 * (size_t)L.P;
    L.s_zgen = f; f += 3 * (size_t)L.P;
    L.hit = bb; bb += L.P;
    L.list = li; li += L.P;
    L.s_slot = slots; slots += 3 * (size_t)L.P;
    L.count = counts + i;
  }
}

int render_depth_fwd(const dist_net_t* net, int engine, const dist_camera_t* camh, const dist_march_t* mp_in,
                     const dist_workspace_t* ws, float* Zdepth, uint8_t* mask, float* min_sdf, int64_t* rows_eval,
                     cudaStream_t st) {
  Cam cam;
  int rc = make_cam(camh, &cam);
  if (rc) return rc;
  NetDev nd;
  rc = make_netdev(net, &nd);
  if (rc) return rc;
  rc = check_codes(nd, cam);
  if (rc) return rc;
  const bool codes = nd.n_codes > 1;
  dist_march_t mpv = *mp_in;
  dist_march_t* mp = &mpv;
  DIST_REQUIRE(mp->buffer_size >= 1 && mp->buffer_size <= DIST_MAX_BUFFER, "buffer_size must be in [1,%d]", DIST_MAX_BUFFER);
  DIST_REQUIRE(mp->march_step >= 1, "march_step must be >= 1");
  DIST_REQUIRE(mp->marching_type >= DIST_MARCH_TRIVIAL && mp->marching_type <= DIST_MARCH_PYRAMID, "bad marching_type");
  DIST_REQUIRE(ws->entry0 && ws->top_lvl && ws->view_stat, "workspace: entry0 / top_lvl / view_stat missing");
  DIST_REQUIRE(ws->ray && ws->entry && ws->exit_ && ws->dist && ws->z && ws->flags && ws->nreal && ws->top_sdf && ws->top_pt &&
                   ws->top_zafter && ws->top_zgen && ws->list_a && ws->list_b && ws->pts && ws->sdf && ws->counts && ws->sdf_origin,
               "workspace: a march buffer is missing");
  const bool pyr = mp->marching_type == DIST_MARCH_PYRAMID;
  const int P = cam.Pv * cam.n_views;
  DIST_CHECK_CUDA(cudaMemsetAsync(ws->view_stat, 0, sizeof(int32_t) * VS_STRIDE * cam.n_views, st));
  const int S_total = mp->march_step;
  const int tb = 256, gb = (P + tb - 1) / tb;
  // two-tier precision of the march rows (tensor-core engine only)
  const bool scr = mp->screen != 0 && engine == DIST_ENGINE_TC;
  const int SEG = seg_capacity(P);
  dist_workspace_t wsv = *ws;
  if (scr) {
    DIST_REQUIRE(ws->seg_approx && ws->sprev && ws->rq_idx && ws->rq_pts && ws->rq_sdf && ws->rq_cnt,
                 "workspace: two-tier precision buffers missing");
    DIST_REQUIRE(mp->screen_margin > 0.f && mp->screen_tpred >= mp->clamp_dist && mp->screen_ext_margin >= 0.f,
                 "two-tier precision: bad margin / prediction thresholds");
    DIST_CHECK_CUDA(cudaMemsetAsync(ws->rq_cnt, 0, sizeof(int32_t), st));
  } else {
    wsv.seg_approx = nullptr;     // the kernels key on seg_approx
  }
  // mask cache (tensor-core engine with two precision tiers only)
  const bool mc = scr && ws->mask_buf != nullptr;
  if (mc) {
    DIST_REQUIRE(ws->mask_base && ws->top_slot && ws->mask_cap > 0 && ws->mask_cap < (int64_t)1 << 31, "workspace: mask cache buffers missing");
    DIST_CHECK_CUDA(cudaMemsetAsync(ws->mask_base, 0, sizeof(int32_t) * (S_total + 3), st));
  } else {
    wsv.mask_buf = nullptr; wsv.top_slot = nullptr;
  }
  ws = &wsv;
  Level L1, L2;
  memset(&L1, 0, sizeof(L1)); memset(&L2, 0, sizeof(L2));
  int64_t coarse_slots = 0;      // mask-cache slots taken by the coarse pyramid levels
  if (pyr) {
    DIST_REQUIRE(ws->pyr_f && ws->pyr_i && ws->pyr_b, "workspace: pyramid buffers missing");
    const bool full_image = cam.row0 == 0 && cam.row_step == cam.row_group && cam.n_rows == cam.H;
    DIST_REQUIRE(full_image || cam.row_group % 4 == 0,
                 "pyramid marching on a row band needs bands made of 4-row groups (row_group % 4 == 0) so that the 1/2- and "
                 "1/4-resolution levels stay band-local");
    DIST_REQUIRE(mp->coarse_steps[0] >= 1 && mp->coarse_steps[0] <= 3 && mp->coarse_steps[1] >= 1 && mp->coarse_steps[1] <= 3 &&
                     mp->coarse_steps[0] + mp->coarse_steps[1] < S_total, "pyramid marching: coarse step counts must be in [1,3]");
    carve_levels(cam, ws, &L1, &L2);
    mp->march_step = S_total - mp->coarse_steps[0] - mp->coarse_steps[1];   // renderer.py:724-725
    mp->first_query_check = 0;                                               // renderer.py:795
    DIST_CHECK_CUDA(cudaMemsetAsync(L1.count, 0, sizeof(int32_t) * 8, st));
    k_hit_flags<<<gb, tb, 0, st>>>(cam, *ws, P); count_launch();
    k_pyr_rays<<<(L1.P + tb - 1) / tb, tb, 0, st>>>(cam, L1, ws->flags, cam.W, cam.n_rows, nullptr); count_launch();
    k_pyr_rays<<<(L2.P + tb - 1) / tb, tb, 0, st>>>(cam, L2, L1.hit, L1.w, L1.h, full_image ? ws->view_stat : nullptr); count_launch();
    if (!full_image) {
      const int w2g = ((cam.W + 1) / 2 + 1) / 2, h2g = ((cam.H + 1) / 2 + 1) / 2;
      k_pyr_global_maxentry<<<(w2g * h2g * cam.n_views + tb - 1) / tb, tb, 0, st>>>(cam, w2g, h2g, ws->view_stat); count_launch();
    }
    for (int lv = 2; lv >= 1; --lv) {
      Level& L = (lv == 2) ? L2 : L1;
      k_pyr_start<<<(L.P + tb - 1) / tb, tb, 0, st>>>(cam, L, L2, lv == 1 ? 1 : 0, ws->view_stat, ws->pts); count_launch();
      const int ns = mp->coarse_steps[2 - lv];
      for (int s = 0; s < ns; ++s) {
        MlpArgs a{};
        a.points = ws->pts; a.n_host = L.P; a.n_dev = L.count; a.clamp_dist = 0.f; a.sdf = ws->sdf; a.rows_evaluated = rows_eval;
        a.tile_counters = ws->tile_counters;
        // mask cache: a coarse step's rows take L.P slots (its capacity), handed out in launch order
        const int64_t slot_base = mc ? coarse_slots : -1;
        if (mc) { a.mask_buf = ws->mask_buf; a.mask_cap = ws->mask_cap; a.mask_base_host = slot_base; coarse_slots += (L.P + 127) / 128 * 128; }
        set_codes(nd, a, L.list, L.Pv);
        rc = mlp_launch(net, nd, engine, 0, a, st);
        if (rc) return rc;
        k_pyr_step<<<min((L.P + tb - 1) / tb, 4 * num_sms()), tb, 0, st>>>(cam, *mp, L, s, ws->pts, ws->sdf, slot_base,
                                                                           mc ? ws->mask_cap : 0); count_launch();
      }
    }
  }
  const int S = mp->march_step;
  DIST_CHECK_CUDA(cudaMemsetAsync(ws->counts, 0, sizeof(int32_t) * 2 * (S_total + 2), st));
  k_setup<<<(cam.n_views * setup_threads_per_view(cam.W, cam.n_rows) + tb - 1) / tb, tb, 0, st>>>(cam, *mp, *ws, Zdepth, mask, min_sdf, P,
                                                                                                L1, L2); count_launch();
  const int n_origin = codes ? cam.n_views : 1;
  k_append_origin<<<1, 256, 0, st>>>(*ws, SEG, (int)coarse_slots, n_origin, cam.Pv); count_launch();
  DIST_CHECK_CUDA(cudaGetLastError());
  const int gu = min(gb, 4 * num_sms());
  for (int s = 0; s < S; ++s) {
    MlpArgs a{};
    // segment 1 (rays predicted far from the surface; one-pass tiles when screening) + segment 2 (the rest, full precision)
    a.points = ws->pts + (size_t)(s & 1) * (size_t)(2 * SEG) * 3;
    a.n_host = P; a.n_dev = ws->counts + 2 * s;
    a.n2_host = P + 1; a.n2_dev = ws->counts + 2 * s + 1; a.seg2_offset = SEG;
    a.clamp_dist = 0.f; a.sdf = ws->sdf; a.rows_evaluated = rows_eval;
    a.tile_counters = ws->tile_counters;
    if (scr) { a.screen_seg1 = 1; a.screen_thresh = mp->clamp_dist + mp->screen_margin; a.seg_approx = ws->seg_approx; }
    if (mc) { a.mask_buf = ws->mask_buf; a.mask_cap = ws->mask_cap; a.mask_base_dev = ws->mask_base + s; }
    set_codes(nd, a, (s & 1) ? ws->list_b : ws->list_a, cam.Pv);     // both segments: the rows' entries of the active list
    rc = mlp_launch(net, nd, engine, 0, a, st);
    if (rc) return rc;
    k_march_update<<<gu, tb, 0, st>>>(cam, *mp, *ws, s, P, n_origin); count_launch();
  }
  if (scr) {
    k_requery_gen<<<gb, tb, 0, st>>>(*mp, *ws, P); count_launch();
    MlpArgs a{};
    a.points = ws->rq_pts; a.n_host = (int64_t)P * mp->buffer_size; a.n_dev = ws->rq_cnt; a.clamp_dist = 0.f; a.sdf = ws->rq_sdf;
    a.tile_counters = ws->tile_counters;
    if (mc) { a.mask_buf = ws->mask_buf; a.mask_cap = ws->mask_cap; a.mask_base_dev = ws->mask_base + S; }   // after the last step's rows
    set_codes(nd, a, ws->rq_idx, cam.Pv * DIST_MAX_BUFFER);
    rc = mlp_launch(net, nd, engine, 0, a, st);
    if (rc) return rc;
    k_requery_apply<<<gu, tb, 0, st>>>(*ws, P, S); count_launch();
  }
  k_finalize<<<gb, tb, 0, st>>>(*mp, *ws, Zdepth, mask, min_sdf, P, cam.Pv, codes ? 1 : 0); count_launch();
  DIST_CHECK_CUDA(cudaGetLastError());
  return DIST_OK;
}

int render_normal_fwd(const dist_net_t* net, int engine, const dist_camera_t* camh, const float* Zdepth,
                      const uint8_t* mask, float clamp_dist, int normalize, float* Znormal, int32_t* s_idx,
                      float* s_pts, float* s_grad, int32_t* s_count, int64_t* rows_eval, cudaStream_t st) {
  Cam cam;
  int rc = make_cam(camh, &cam);
  if (rc) return rc;
  NetDev nd;
  rc = make_netdev(net, &nd);
  if (rc) return rc;
  rc = check_codes(nd, cam);
  if (rc) return rc;
  const int P = cam.Pv * cam.n_views;
  DIST_CHECK_CUDA(cudaMemsetAsync(s_count, 0, sizeof(int32_t), st));
  DIST_CHECK_CUDA(cudaMemsetAsync(Znormal, 0, sizeof(float) * 3 * (size_t)P, st));
  const int tb = 256, gb = (P + tb - 1) / tb;
  k_normal_gen<<<gb, tb, 0, st>>>(cam, Zdepth, mask, s_idx, s_pts, s_count, P); count_launch();
  MlpArgs a{};
  a.points = s_pts; a.n_host = P; a.n_dev = s_count; a.clamp_dist = clamp_dist; a.grad = s_grad;
  a.rows_evaluated = rows_eval;
  set_codes(nd, a, s_idx, cam.Pv);
  rc = mlp_launch(net, nd, engine, 1, a, st);
  if (rc) return rc;
  k_normal_finish<<<min(gb, 4 * num_sms()), tb, 0, st>>>(cam, s_idx, s_grad, s_count, normalize, Znormal, P); count_launch();
  DIST_CHECK_CUDA(cudaGetLastError());
  return DIST_OK;
}

int render_depth_bwd(const dist_net_t* net, int engine, const dist_camera_t* camh, const dist_march_t* mp,
                     const dist_workspace_t* ws, const float* gZ, const float* gM, float* acc0, float* accl,
                     float* d_cam, float* d_ray, float* d_ray_coarse, int32_t* s_row_pix, float* s_pts, float* s_coef, uint8_t* s_clamp,
                     float* s_dpts, int32_t* s_count, int64_t* rows_eval, cudaStream_t st) {
  (void)s_clamp;
  Cam cam;
  int rc = make_cam(camh, &cam);
  if (rc) return rc;
  NetDev nd;
  rc = make_netdev(net, &nd);
  if (rc) return rc;
  rc = check_codes(nd, cam);
  if (rc) return rc;
  const bool codes = nd.n_codes > 1;
  const int P = cam.Pv * cam.n_views;
  DIST_CHECK_CUDA(cudaMemsetAsync(s_count, 0, sizeof(int32_t), st));
  const int tb = 256, gb = (P + tb - 1) / tb;
  // samples whose decoder row left its ReLU masks in the cache are replayed with the transposed chain alone
  const bool mc = engine == DIST_ENGINE_TC && ws->mask_buf && ws->top_slot && ws->bm_row && ws->bm_slot && ws->bm_sdf && ws->bm_coef &&
                  ws->bm_dpts && ws->bm_cnt;
  if (mc) DIST_CHECK_CUDA(cudaMemsetAsync(ws->bm_cnt, 0, sizeof(int32_t), st));
  k_bwd_gen<<<gb, tb, 0, st>>>(*mp, *ws, gZ, gM, s_row_pix, s_pts, s_coef, s_count, P, mc ? 1 : 0, cam.Pv,
                                codes ? 1 : 0); count_launch();
  MlpArgs a{};
  a.points = s_pts; a.n_host = (int64_t)P * mp->buffer_size; a.n_dev = s_count; a.clamp_dist = 0.f;
  a.grad = s_dpts; a.coef = s_coef; a.acc0 = acc0; a.accl = accl; a.rows_evaluated = rows_eval;
  set_codes(nd, a, s_row_pix, cam.Pv * DIST_MAX_BUFFER);
  rc = mlp_launch(net, nd, engine, 2, a, st);
  if (rc) return rc;
  if (mc) {
    MlpArgs b{};
    b.n_host = (int64_t)P * mp->buffer_size; b.n_dev = ws->bm_cnt; b.clamp_dist = 0.f;
    b.grad = ws->bm_dpts; b.coef = ws->bm_coef; b.acc0 = acc0; b.accl = accl;
    b.rows_evaluated = rows_eval ? rows_eval + 1 : nullptr;      // counted apart: these rows cost F, not 2F
    b.mask_buf = ws->mask_buf; b.mask_cap = ws->mask_cap; b.slots = ws->bm_slot; b.sdf_in = ws->bm_sdf;
    set_codes(nd, b, ws->bm_row, cam.Pv * DIST_MAX_BUFFER);
    rc = mlp_launch(net, nd, engine, 3, b, st);
    if (rc) return rc;
  }
  if (d_cam && d_ray) {
    const int w1 = (cam.W + 1) / 2, h1 = (cam.n_rows + 1) / 2, w2 = (w1 + 1) / 2, h2 = (h1 + 1) / 2;
    const int gs = min((int)(((int64_t)P * mp->buffer_size + tb - 1) / tb), 4 * num_sms());
    const int lv = mp->cam_grad_levels ? mp->cam_grad_levels : 3;
    k_bwd_scatter<<<gs, tb, 0, st>>>(cam, *ws, s_row_pix, s_dpts, s_count, d_cam, d_ray, d_ray_coarse, w1, w1 * h1, w2, w2 * h2, P, lv);
    count_launch();
    if (mc) {
      k_bwd_scatter<<<gs, tb, 0, st>>>(cam, *ws, ws->bm_row, ws->bm_dpts, ws->bm_cnt, d_cam, d_ray, d_ray_coarse, w1, w1 * h1, w2,
                                       w2 * h2, P, lv);
      count_launch();
    }
  }
  DIST_CHECK_CUDA(cudaGetLastError());
  return DIST_OK;
}

}  // namespace dist
