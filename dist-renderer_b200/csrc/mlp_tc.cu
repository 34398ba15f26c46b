// tcgen05 tensor-core engine for the folded DeepSDF decoder (DIST_ENGINE_TC), sm_100a only.
//
// A cluster of two CTAs (one SM pair) owns a tile of 128 decoder rows (64 per CTA) and carries it through the whole
// network on-chip:
//   * layer 0 (K = 3, xyz) and the last layer (N = 1, dot product + tanh) run on CUDA cores in the epilogue warps;
//   * every hidden layer is a tcgen05.mma.cta_group::2.kind::f16 GEMM (M = 128 over the pair, N = 256 per instruction,
//     K = 16) with split-fp16 operands: D += A_hi*W_hi + A_lo*W_hi + A_hi*W_lo, fp32 accumulation in TMEM
//     (see tc.py for the precision argument and the truncation pre-compensation);
//   * A (activations, 64 rows x K x {hi,lo} fp16 = 128 KB) is resident in shared memory in the UMMA no-swizzle
//     K-major "panel" layout and is rewritten in place by the epilogue of each layer (TMEM -> registers -> bias,
//     ReLU, split -> smem); it never touches HBM;
//   * W streams L2 -> smem through a 6-stage ring of 16 KB TMA box copies per CTA (each CTA holds half of the
//     256 N-rows of a stage; `.cta_group::2` copies signal the leader CTA's mbarrier), released by tcgen05.commit;
//   * the MMA order is N-half outer / K block inner: accumulator half 0 (128 TMEM columns) completes while half 1 is
//     still being computed, so its epilogue -- which produces the first eight 32-feature A blocks of the NEXT layer --
//     overlaps the second pass; an A block is overwritten in place only after the last pass has read it (A_FREE
//     barriers committed by the MMA issuer), and the next layer starts on block 0 the moment the current one ends;
//   * accumulators ping-pong between two 256-column TMEM buffers; 16 epilogue warps own 32 rows x 32 columns each;
//   * the transposed chain (input gradient / backward replay) is the same machinery on W^T tiles, with the ReLU sign
//     bits kept per thread and the latent gradient accumulated as per-lane running column sums.
//   * two precision tiers (MODE 0, round 2): rows of the first row segment -- rays the march predicts to stay beyond its
//     clamp band -- are evaluated with ONE fp16 pass (A_hi W_hi, hi halves of the weight stages only), two tiles at a time
//     ("pair mode": the second tile's activations occupy the lo region, its accumulators the second TMEM buffer, both tiles
//     consume every weight stage); a half-tile keeps its one-pass values only if all of its rows come out beyond the band,
//     otherwise the tile is recorded in a per-CTA bitmap and re-evaluated with the three passes in a second sweep over the
//     cluster's tiles after one cluster barrier (the CTAs read each other's bitmap through distributed shared memory);
// Warp roles per CTA (640 threads): warp 0 TMA producer, warp 1 MMA issuer (leader CTA), warp 2 TMEM allocator,
// warps 4-19 epilogue (TMEM lane quarter = warp % 4, 32-column quarter = (warp-4)/4).
// DIST_TC_DEBUG (env): bit 2 prints cycles/ns of CTA 0 (+ a per-layer timeline when compiled with -DDIST_TC_TIMELINE).
//
// Replaces: Decoder.inference / decode_sdf / decode_sdf_gradient and the autograd backward through them
// (core/graph/deep_sdf_decoder.py:80-111, core/utils/decoder_utils.py:53-92)
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"

namespace dist {
namespace {

// -DDIST_TC_TIMELINE: the MMA issuer of cluster 0 also accumulates, for its second tile, the cycles it spends waiting for
// activation blocks (A_FULL) and for weight stages (W_FULL) per layer: dbg_out[256 + 2 m], dbg_out[257 + 2 m]
#ifdef DIST_TC_TIMELINE
#define TL_BEGIN() const long long tl_c0 = clock64()
#define TL_TILE (c1 > 0 ? 2 : 1)     /* the traced tile: the cluster's second tile / second pair */
#define TL_END(slot_) do { if (io.dbg_out && cluster_id == 0 && i == TL_TILE && lane == 0) io.dbg_out[256 + 2 * m + (slot_)] += clock64() - tl_c0; } while (0)
#define TL_MARK(idx_) do { if (io.dbg_out && cluster_id == 0 && i == TL_TILE && lane == 0) io.dbg_out[idx_] = clock64(); } while (0)
#else
#define TL_BEGIN() do {} while (0)
#define TL_END(slot_) do {} while (0)
#define TL_MARK(idx_) do {} while (0)
#endif

constexpr int NST = 6;                 // weight ring stages
constexpr int STAGE_BYTES = 16384;     // per CTA: [hi 8 KB][lo 8 KB]
constexpr int OFF_AHI = 0, OFF_ALO = 65536, OFF_W = 131072;
constexpr int OFF_BAR = OFF_W + NST * STAGE_BYTES;   // 229376
constexpr int OFF_HDR = OFF_BAR + 448;               // three int64: row counts of the two segments, mask-cache base
constexpr int OFF_PART = OFF_BAR + 512;              // per-row partial sums [64][8] (8 threads share a row)
constexpr int OFF_ROWD = OFF_PART + 2048;            // per-row scalar [64]
constexpr int OFF_FAIL = OFF_ROWD + 256;             // two-tier precision: [near flag u32][pad][fail bitmap, FAIL_WORDS u32]
constexpr int FAIL_WORDS = 32;                       // 1024 tiles per cluster and launch (9 M rows on 74 clusters)
constexpr int SMEM_BYTES = OFF_FAIL + 16 + 4 * FAIL_WORDS;   // 232336 (limit 232448)
constexpr int NTHREADS = 640;                        // 4 service warps + 16 epilogue warps
constexpr int MAX_PROG = 2 * 10;                     // forward + transposed chain, at most 10 tensor-core layers each

struct LayerTC {
  int kc32;          // number of 32-wide K chunks (K padded to a multiple of 64)
  int nh;            // number of 256-wide N halves
  int stage_base;    // first stage of this layer in the blob
  int N;             // forward: logical outputs (hidden width); transposed chain: hidden width of the PREVIOUS net layer
  int app_xyz;       // forward: append xyz at columns N..N+2 of the produced activation (next layer is latent_in)
                     // transposed chain: columns N..N+2 of the result are d/dxyz (this net layer is latent_in)
  float inv_scale;   // 1 / (operand scale * weight scale)
  const float* bias;
};

struct TcParams {
  int n_mma;                       // tensor-core layers of the forward pass (net layers 1 .. n-2)
  int n_prog;                      // layers per tile: n_mma (forward only) or 2 n_mma (forward + transposed chain)
  int acc_l_prog;                  // program layer whose produced delta is accumulated into accl (-1: none)
  int accl_N;                      // width of the latent_in layer
  LayerTC L[MAX_PROG];
  const float* w0;                 // Wt[0]: [8][N0p4], rows 0..2 = weights of x,y,z
  const float* bias0;
  int N0, N0p4;
  const float* wlast;              // W[last] row 0, [K_last]
  const float* blast;
  int K_last;
  int use_tanh;
  float sA, sD;                    // activation / gradient operand scales
  int first_append;                // layer 0's output gets xyz appended (latent_in == 1)
  int dbg;                         // diagnostics (DIST_TC_DEBUG), see the file header
  int stage_rows;                  // tensor-map rows per 16 KB weight stage (STAGE_BYTES / bytes per box row)
  // several latent codes (MC instantiations): bias0 is [n_codes][N0p4]; the forward program layer lat_m (the latent_in
  // layer, -1: none) reads its bias from [n_codes][lat_stride]
  int lat_m, lat_stride;
};

struct TcIO {
  const float* points; int64_t n_host; const int32_t* n_dev; float clamp_dist;
  int64_t n2_host; const int32_t* n2_dev; int64_t seg2_offset;   // optional second row segment [seg2_offset, seg2_offset + n2)
  float* sdf; float* grad; const float* coef; const uint8_t* use_clamp; float* acc0; float* accl;
  int64_t* rows_evaluated;
  long long* dbg_out;   // DIST_TC_DEBUG bit2: [cycles, ns] of CTA 0
  // two-tier precision (MODE 0 only; see the kernel comment).  screen_seg1 == 0: every tile at full precision.
  int screen_seg1;              // tiles of the first row segment try ONE fp16 pass first ("screen"); the second segment
                                // always gets the three split-precision passes
  float screen_thresh;          // a screened half-tile passes when all its rows have |sdf| > screen_thresh
  uint8_t* seg_approx;          // [rows / 64] out: 1 = the sdf of this 64-row half-tile are one-pass values
  unsigned long long* tile_counters;   // optional [2]: += tiles evaluated with one pass / with three passes
  // ReLU-mask cache (see "mask cache" in the kernel comment).  MODE 0 writes, MODE 3 reads.
  uint32_t* mask_buf;           // [mask words][mask_cap] one 32-bit word per (net layer, 32-feature block) and row slot
  int64_t mask_cap;             // row slots in mask_buf
  int64_t mask_base_host;       // first slot of this launch's full-precision rows (when mask_base_dev == nullptr); < 0: off
  const int32_t* mask_base_dev;
  const int32_t* slots;         // MODE 3: [n] mask slot of each row
  const float* sdf_in;          // MODE 3: [n] the (unclamped) decoder output of each row, as recorded by the forward
  const int32_t* row_code;      // MC: code of row r = row_code[r] / code_div (MlpArgs.row_code)
  int32_t code_div;
};

// --------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(bar), "r"(parity) : "memory");
}
// wait with cluster-scope acquire: for barriers the peer CTA arrives on remotely
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(bar), "r"(parity) : "memory");
}
// arrive (count 1) on the barrier at the same smem offset in CTA `target_rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_local, uint32_t target_rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar_local), "r"(target_rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// 32-bit load from the same shared-memory offset of CTA `rank` of this cluster (distributed shared memory)
__device__ __forceinline__ uint32_t ld_dsmem_u32(uint32_t local_addr, uint32_t rank) {
  uint32_t remote, v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(rank));
  asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(remote) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
__device__ __forceinline__ void mma_f16_2cta(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void commit_mc(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
      "%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Writes 8 consecutive features (one K-group panel row) of this thread's row: x[] already multiplied by sA.
__device__ __forceinline__ void store_group(uint8_t* smem, int feat0, int row, const float* x) {
  __half2 h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    h[i] = __floats2half2_rn(x[2 * i], x[2 * i + 1]);
    const float2 hf = __half22float2(h[i]);
    l[i] = __floats2half2_rn(x[2 * i] - hf.x, x[2 * i + 1] - hf.y);
  }
  const int off = (feat0 >> 3) * 1024 + row * 16;
  *reinterpret_cast<uint4*>(smem + OFF_AHI + off) = *reinterpret_cast<uint4*>(h);
  *reinterpret_cast<uint4*>(smem + OFF_ALO + off) = *reinterpret_cast<uint4*>(l);
}

// pair mode: hi halves only, into the activation region at byte offset `region` (OFF_AHI: tile 0, OFF_ALO: tile 1)
__device__ __forceinline__ void store_group_hi(uint8_t* smem, int region, int feat0, int row, const float* x) {
  __half2 h[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(x[2 * i], x[2 * i + 1]);
  *reinterpret_cast<uint4*>(smem + region + (feat0 >> 3) * 1024 + row * 16) = *reinterpret_cast<uint4*>(h);
}

// --------------------------------------------------------------------------------------------- kernel
// MODE 0: forward (sdf).  MODE 1: forward + transposed chain -> d clamp(sdf)/d xyz.  MODE 2: backward replay with per-row
// upstream coefficients: d/dxyz per row and the row-summed pre-activation gradients of layer 0 / the latent_in layer.
// MODE 3: MODE 2 without its forward half: the ReLU sign bits come from the mask cache a MODE 0 launch wrote (io.slots), the
// decoder output from io.sdf_in; only the transposed chain runs (program layers n_mma .. 2 n_mma - 1).
// MC: several latent codes (dist_net_t.n_codes > 1).  Each thread owns one row in the epilogue, so it reads the folded
// biases (layer 0, the latent_in layer) at its row's code -- rows of a warp mostly share a code and the loads broadcast --
// and MODE 2/3 accumulate the latent gradient per code (see "per-code running sums").  MC = false is the one-code kernel
// with none of this in it.
template <int MODE, bool MC>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
mlp_tc_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_hi, const TcParams P, const TcIO io) {
  extern __shared__ __align__(1024) uint8_t smem[];
  // rows: segment 1 = [0, n1), segment 2 = [seg2_offset, seg2_offset + n2) (seg2_offset a multiple of 128).
  // Device-side counts are read by ONE thread per CTA and handed round through shared memory: 20 warps x 148 CTAs loading the
  // same word at kernel start queue up on one L2 sector.
  volatile int64_t* hdr = reinterpret_cast<volatile int64_t*>(smem + OFF_HDR);
  if (threadIdx.x == 0) {
    const int64_t v0 = io.n_dev ? (int64_t)*io.n_dev : io.n_host;          // three independent loads in flight
    const int64_t v1 = io.n2_dev ? (int64_t)*io.n2_dev : io.n2_host;
    const int64_t v2 = (MODE == 0 && io.mask_buf) ? (io.mask_base_dev ? (int64_t)*io.mask_base_dev : io.mask_base_host) : -1;
    hdr[0] = v0; hdr[1] = v1; hdr[2] = v2;
  }
  __syncthreads();
  const int64_t n1 = hdr[0], n2 = hdr[1];
  const int64_t n = n1 + n2;
  if (n <= 0) return;
  const uint32_t rank = cluster_ctarank();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  const int64_t tiles1 = (n1 + 127) / 128, n_tiles = tiles1 + (n2 + 127) / 128;
  if ((blockIdx.x >> 1) >= n_tiles) return;     // a cluster without a tile (grid sized for a device-side row count): both CTAs leave
  auto row0_of = [&](int64_t t) -> int64_t { return (t < tiles1) ? t * 128 : io.seg2_offset + (t - tiles1) * 128; };
  auto lim_of = [&](int64_t t) -> int64_t { return (t < tiles1) ? n1 : io.seg2_offset + n2; };
  if (blockIdx.x == 0 && tid == 0 && io.rows_evaluated)
    atomicAdd(reinterpret_cast<unsigned long long*>(io.rows_evaluated), (unsigned long long)n);
  // ---- mask cache: a MODE 0 launch records, for every row it evaluates at full precision in its first sweep, the ReLU sign
  // bits of all hidden layers (one word per layer and 32-feature block, 512 B per row for the 8x512 network) at slot
  // mask_base + (index of the row among those rows).  The backward replay (MODE 3) then runs the transposed chain alone:
  // the forward half of MODE 2 only existed to recompute these bits.
  const int64_t mask_base = hdr[2];

  long long dbg_c0 = 0, dbg_t0 = 0;
  if (io.dbg_out && blockIdx.x == 0 && tid == 0) { dbg_c0 = clock64(); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t0)); }
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + OFF_BAR;
  auto W_FULL = [&](int s) { return bar0 + 8 * s; };
  auto W_EMPTY = [&](int s) { return bar0 + 8 * (NST + s); };
  auto A_FULL = [&](int c) { return bar0 + 8 * (2 * NST + c); };
  auto A_FREE = [&](int c) { return bar0 + 8 * (2 * NST + 16 + c); };          // last read of A block c is complete
  auto D_FULL = [&](int b, int h) { return bar0 + 8 * (2 * NST + 32 + 2 * b + h); };  // N-half h of buffer b complete
  const uint32_t FIN = bar0 + 8 * (2 * NST + 36);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 8 * (2 * NST + 37));
  const int n_prog = P.n_prog;
  const int m0 = (MODE == 3) ? P.n_mma : 0;      // first program layer of a tile

  // ---- two-tier precision (MODE 0 with io.screen_seg1): a tile of the first row segment is first evaluated with ONE fp16 pass
  // (A_hi W_hi; only the hi halves of the weight stages are fetched).  If all 64 rows of a CTA come out with
  // |sdf| > screen_thresh (safely beyond the march's clamp, so the step they cause does not depend on their last bits)
  // the half-tile is done and flagged in io.seg_approx; if either CTA of the pair sees a nearer row the tile is recorded
  // in that CTA's fail bitmap and re-evaluated at full precision in a second pass over this cluster's tiles ("phase 1")
  // after a cluster barrier -- no other communication between roles or CTAs is needed, every role walks the same lists.
  const int cnt = (cluster_id < n_tiles) ? (int)((n_tiles - cluster_id + n_clusters - 1) / n_clusters) : 0;  // tiles of this cluster
  const bool screening = (MODE == 0) && io.screen_seg1 != 0 && cnt <= 32 * FAIL_WORDS;
  volatile uint32_t* near_flag = reinterpret_cast<volatile uint32_t*>(smem + OFF_FAIL);
  volatile uint32_t* fail_words = reinterpret_cast<volatile uint32_t*>(smem + OFF_FAIL + 16);
  const uint32_t fail_addr = sbase + OFF_FAIL + 16;
  auto tile_of = [&](int i) -> int64_t { return cluster_id + (int64_t)i * n_clusters; };
  // One-pass tiles are processed TWO AT A TIME ("pair mode"): the second tile's activations live where a full-precision tile
  // keeps its lo halves (OFF_ALO), its accumulators in the second TMEM buffer, and both tiles consume every weight stage --
  // the weight stream and the barrier traffic are paid once per 256 rows, and the tensor pipe has the other tile's MMAs to
  // run while one tile's epilogue is on the critical path.  c1 = this cluster's one-pass tiles (the first c1 of its list).
  const int c1 = (screening && cluster_id < tiles1) ? (int)((tiles1 - cluster_id + n_clusters - 1) / n_clusters) : 0;
  // next tile index of this cluster after i (i = -1: the first), -1 when exhausted.  phase 0: all tiles; phase 1: tiles
  // whose fail bit is set in this CTA's or the peer's bitmap (read through distributed shared memory)
  auto next_tile = [&](int phase, int i) -> int {
    if (phase == 0) {     // pairs (i, i + 1) inside [0, c1), single tiles after that
      const int j = (i < 0) ? 0 : ((i < c1) ? min(i + 2, c1) : i + 1);
      return (j < cnt) ? j : -1;
    }
    int j = i + 1;
    while (j < cnt) {
      const uint32_t w = (fail_words[j >> 5] | ld_dsmem_u32(fail_addr + 4 * (j >> 5), rank ^ 1u)) >> (j & 31);
      if (w) { j += __ffs(w) - 1; return (j < cnt) ? j : -1; }
      j = (j | 31) + 1;
    }
    return -1;
  };

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) { mbar_init(W_FULL(s), 1); mbar_init(W_EMPTY(s), 1); }
    for (int c = 0; c < 16; ++c) mbar_init(A_FULL(c), 4);  // 2 warps x 2 CTAs produce each 32-feature block
    for (int c = 0; c < 16; ++c) mbar_init(A_FREE(c), 1);
    for (int b = 0; b < 2; ++b) { mbar_init(D_FULL(b, 0), 1); mbar_init(D_FULL(b, 1), 1); }
    mbar_init(FIN, 32);                                     // 16 epilogue warps x 2 CTAs
    near_flag[0] = 0u; near_flag[1] = 0u;
    for (int w = 0; w < FAIL_WORDS; ++w) fail_words[w] = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // =============================================================== TMA producer (both CTAs)
    // the whole warp runs the loop (warp-uniform control flow keeps addresses in uniform registers); one elected
    // lane issues the copies
    {
      uint32_t p_slot = 0, p_phase = 0;
      const uint32_t bar_leader_mask = 0xFEFFFFFFu;
      for (int phase = 0; phase < 2; ++phase) {
        for (int i = next_tile(phase, -1); i >= 0; i = next_tile(phase, i)) {
          const bool exact = !(phase == 0 && i < c1);      // one-pass tiles come in pairs that share one weight stream
          for (int m = m0; m < n_prog; ++m) {
            const int kc32 = P.L[m].kc32, sb = P.L[m].stage_base;
            // full precision: one ring slot = one 32-wide K chunk, [hi 8 KB][lo 8 KB] per CTA.
            // one pass: one ring slot = the hi halves of TWO consecutive K chunks (the same bytes in flight per slot: the ring
            // of NST slots covers the L2 -> smem round trip only with 16 KB per slot; 8 KB slots ran at a third of the MMA rate)
            const int nslot = exact ? kc32 * P.L[m].nh : (kc32 / 2) * P.L[m].nh;
            for (int s = 0; s < nslot; ++s) {
              const uint32_t slot = p_slot, ph = p_phase;
              if (++p_slot == NST) { p_slot = 0; p_phase ^= 1; }
              mbar_wait(W_EMPTY(slot), ph ^ 1);
              if (elect_one()) {
                if (rank == 0) mbar_expect_tx(W_FULL(slot), 2 * STAGE_BYTES);
                const uint32_t dst = sbase + OFF_W + slot * STAGE_BYTES;
                const uint32_t bar = W_FULL(slot) & bar_leader_mask;
                if (exact) {
                  const int row = ((sb + s) * 2 + (int)rank) * P.stage_rows;
                  asm volatile(
                      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
                          "r"(dst), "l"(&tmap), "r"(bar), "r"(0), "r"(row)
                      : "memory");
                } else {
#pragma unroll
                  for (int c = 0; c < 2; ++c) {
                    const int row = ((sb + 2 * s + c) * 2 + (int)rank) * P.stage_rows;
                    asm volatile(
                        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
                            "r"(dst + c * (STAGE_BYTES / 2)), "l"(&tmap_hi), "r"(bar), "r"(0), "r"(row)
                        : "memory");
                  }
                }
              }
              __syncwarp();
            }
          }
        }
        if (phase == 0) {
          if (!screening) break;
          cluster_sync_all();     // every thread of both CTAs: the fail bitmaps are complete
        }
      }
    }
  } else if (warp == 1) {
    // =============================================================== MMA issuer (leader CTA)
    // warp-uniform loop; descriptors are advanced by adding 16-byte units to the low word; one elected lane issues
    if (rank == 0) {
      const uint32_t idesc = (1u << 4) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
      const uint64_t a_hi0 = make_desc(sbase + OFF_AHI, 1024, 128);
      const uint64_t a_lo0 = make_desc(sbase + OFF_ALO, 1024, 128);
      const uint64_t b_0 = make_desc(sbase + OFF_W, 2048, 128);
      uint32_t G = 0, a_phase = 0, fin_phase = 0, w_slot = 0, w_phase = 0;
      uint32_t d_first = 1;
      bool prev_pair = false;
      for (int phase = 0; phase < 2; ++phase) {
      for (int i = next_tile(phase, -1); i >= 0; i = next_tile(phase, i)) {
        const int64_t t = tile_of(i);
        const bool exact = !(phase == 0 && i < c1);   // pair mode: two one-pass tiles, A_hi W_hi only
        const bool has_b = !exact && (i + 1 < c1);    // (an odd count leaves the last pair with one tile)
        (void)t;
        for (int m = m0; m < n_prog; ++m, ++G) {
          const int kc32 = P.L[m].kc32, nh = P.L[m].nh;
          const uint32_t buf = exact ? (G & 1) : 0u;
          // The last accumulator of the previous tile lives in a TMEM buffer until its epilogue drained it (FIN).  Single tiles
          // ping-pong between the two buffers layer by layer, so layer 0 may start early and only layer 1 waits; a pair uses
          // both buffers in every layer, so a pair -- and the tile after a pair -- waits before its layer 0.
          if (!d_first && m == m0 + ((!exact || prev_pair) ? 0 : 1)) { mbar_wait_cluster(FIN, fin_phase); fin_phase ^= 1; }
          // N-half outer, K block inner: half 0 of the accumulator completes while half 1 is still being computed, so
          // its epilogue (the first A blocks of the next layer) overlaps the second pass.  A_FREE(kc) tells the epilogue
          // when the last pass has consumed A block kc and its slot may be overwritten in place.
          // The issuing thread is the bottleneck of this kernel (6 MMAs = 384 tensor cycles per stage): two stages are
          // issued per barrier round trip, ring slot / phase are tracked incrementally, nothing else is in the loop.
          for (int h = 0; h < nh; ++h) {
            const uint32_t d_addr = tmem + buf * 256 + h * 128;
            const bool last_pass = (h == nh - 1);
            if (!exact) {
              // one pass: a ring slot holds the hi halves of two K chunks -> 4 MMAs per slot, two slots per round trip
              for (int kc = 0; kc < kc32; kc += 4) {
                const int nsl = (kc + 2 < kc32) ? 2 : 1;
                if (h == 0) {
                  TL_BEGIN();
                  for (int c = 0; c < 2 * nsl; ++c) mbar_wait_cluster(A_FULL(kc + c), (a_phase >> (kc + c)) & 1);
                  if (kc == 0) TL_MARK(8 + m * 4 + 0);
                  // A pair keeps its accumulators in fixed TMEM buffers (no ping-pong between layers): the first MMA of this
                  // pass overwrites N-half 0 of the previous layer, which the epilogue has read completely only once ALL the
                  // blocks made from it (0..7) are written -- wait for those too (they are waited on again, and consumed, below)
                  if (kc == 0)
                    for (int c = 2 * nsl; c < min(8, kc32); ++c) mbar_wait_cluster(A_FULL(c), (a_phase >> c) & 1);
                  a_phase ^= (nsl == 2 ? 15u : 3u) << kc;
                  TL_END(0);
                }
                const uint32_t slot0 = w_slot, ph0 = w_phase;
                uint32_t slot1 = slot0, ph1 = ph0;
                if (++w_slot == NST) { w_slot = 0; w_phase ^= 1; }
                if (nsl == 2) {
                  slot1 = w_slot; ph1 = w_phase;
                  if (++w_slot == NST) { w_slot = 0; w_phase ^= 1; }
                }
                {
                  TL_BEGIN();
                  mbar_wait(W_FULL(slot0), ph0);
                  if (nsl == 2) mbar_wait(W_FULL(slot1), ph1);
                  TL_END(1);
                }
                tc_fence_after();
                if (elect_one()) {
                  for (int u = 0; u < nsl; ++u) {
                    const uint32_t slot = u ? slot1 : slot0;
                    for (int ts = 0; ts < (has_b ? 2 : 1); ++ts) {     // both tiles of the pair read this weight slot
                      const uint64_t a_base = ts ? a_lo0 : a_hi0;      // tile 1's activations live in the lo region
                      const uint32_t d_ts = d_addr + ts * 256;
#pragma unroll
                      for (int c = 0; c < 2; ++c) {
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                          const int kk = kc + 2 * u + c;
                          const uint64_t a_off = (uint64_t)((kk * 4 + ks * 2) * 64);
                          const uint64_t b_off = (uint64_t)(slot * (STAGE_BYTES / 16) + c * 512 + ks * 256);
                          mma_f16_2cta(d_ts, a_base + a_off, b_0 + b_off, idesc, (kk | ks) ? 1u : 0u);
                        }
                      }
                    }
                    commit_mc(W_EMPTY(slot));
                    if (last_pass) { commit_mc(A_FREE(kc + 2 * u)); commit_mc(A_FREE(kc + 2 * u + 1)); }
                  }
                  if (kc + 4 >= kc32) commit_mc(D_FULL(buf, h));
                }
                __syncwarp();
                if (kc + 4 >= kc32 && last_pass) TL_MARK(8 + m * 4 + 1);
              }
            } else
            for (int kc = 0; kc < kc32; kc += 2) {
              if (h == 0) {
                TL_BEGIN();
                mbar_wait_cluster(A_FULL(kc), (a_phase >> kc) & 1);
                mbar_wait_cluster(A_FULL(kc + 1), (a_phase >> (kc + 1)) & 1);
                a_phase ^= (3u << kc);
                TL_END(0);
#ifdef DIST_TC_TIMELINE
                if (io.dbg_out && cluster_id == 0 && t == cluster_id + n_clusters && lane == 0 && kc == 0) io.dbg_out[8 + m * 4 + 0] = clock64();
#endif
              }
              const uint32_t slot0 = w_slot, ph0 = w_phase;
              uint32_t slot1 = slot0 + 1, ph1 = ph0;
              if (slot1 == NST) { slot1 = 0; ph1 ^= 1; }
              w_slot = slot1 + 1; w_phase = ph1;
              if (w_slot == NST) { w_slot = 0; w_phase ^= 1; }
              {
                TL_BEGIN();
                mbar_wait(W_FULL(slot0), ph0);
                mbar_wait(W_FULL(slot1), ph1);
                TL_END(1);
              }
              tc_fence_after();
              if (elect_one()) {
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                  const uint32_t slot = u ? slot1 : slot0;
#pragma unroll
                  for (int ks = 0; ks < 2; ++ks) {
                    const uint64_t a_off = (uint64_t)(((kc + u) * 4 + ks * 2) * 64);
                    const uint64_t b_off = (uint64_t)(slot * (STAGE_BYTES / 16) + ks * 256);
                    mma_f16_2cta(d_addr, a_hi0 + a_off, b_0 + b_off, idesc, ((kc + u) | ks) ? 1u : 0u);
                    mma_f16_2cta(d_addr, a_lo0 + a_off, b_0 + b_off, idesc, 1u);
                    mma_f16_2cta(d_addr, a_hi0 + a_off, b_0 + b_off + 512, idesc, 1u);
                  }
                  commit_mc(W_EMPTY(slot));
                  if (last_pass) commit_mc(A_FREE(kc + u));
                }
                if (kc + 2 >= kc32) commit_mc(D_FULL(buf, h));
              }
              __syncwarp();
#ifdef DIST_TC_TIMELINE
              if (io.dbg_out && cluster_id == 0 && t == cluster_id + n_clusters && lane == 0 && kc + 2 >= kc32 && last_pass) io.dbg_out[8 + m * 4 + 1] = clock64();
              if (io.dbg_out && cluster_id == 0 && t == cluster_id && lane == 0 && kc + 2 >= kc32 && last_pass && m == n_prog - 1) io.dbg_out[200] = clock64();
#endif
            }
          }
        }
        d_first = 0;
        prev_pair = !exact;
      }
        if (phase == 0) {
          if (!screening) break;
          cluster_sync_all();
        }
      }
    } else if (screening) {
      cluster_sync_all();     // the non-leader CTA's MMA warp only takes part in the phase barrier
    }
  } else if (warp < 4) {
    if (screening) cluster_sync_all();   // TMEM-allocator warp and the spare warp: phase barrier only
  } else {
    // =============================================================== epilogue warps (16 warps, 32 rows x 32 columns each)
    const int ew = warp - 4;
    const int qq = warp & 3;             // TMEM lane quarter accessible to this warp
    const int q = qq >> 1;               // which 128-feature half of an N-half this lane quarter holds
    const int ch = ew >> 2;              // which 32-column quarter of those 128 this warp handles (0..3)
    const int row = 32 * (qq & 1) + lane;
    const uint32_t lane_base = (uint32_t)(32 * qq) << 16;
    const float sA = P.sA, sD = P.sD;
    const int n_mma = P.n_mma;
    float* part = reinterpret_cast<float*>(smem + OFF_PART);
    float* rowd = reinterpret_cast<float*>(smem + OFF_ROWD);
    const int pslot = 4 * q + ch;        // this thread's slot among the 8 threads that share a row
    uint32_t G = 0, d_phase = 0, free_phase = 0;
    float px = 0.f, py = 0.f, pz = 0.f;
    uint32_t mk[DIST_MAX_LAYERS][2];     // ReLU sign bits of this thread's (row, 32 features x 2 halves) per net layer
    float acc0r[2] = {0.f, 0.f}, acclr[2] = {0.f, 0.f};  // MODE 2: per-lane running column sums
    // per-code running sums (MC): the sums above belong to code acc_code (warp-uniform) and are flushed into acc[acc_code]
    // when a tile whose 32 rows of this warp share another code comes along; tiles with mixed rows bypass them
    int acc_code = 0;
    auto flush_sums = [&]() {
      // lane j of this warp holds column 32*kb + j of its blocks
      const size_t o0 = MC ? (size_t)acc_code * P.N0 : 0, ol = MC ? (size_t)acc_code * P.accl_N : 0;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int f = 32 * (8 * h + 4 * q + ch) + lane;
        if (io.acc0 && f < P.N0 && acc0r[h] != 0.f) atomicAdd(io.acc0 + o0 + f, acc0r[h] * (1.f / sD));
        if (io.accl && P.acc_l_prog >= 0 && f < P.accl_N && acclr[h] != 0.f) atomicAdd(io.accl + ol + f, acclr[h] * (1.f / sD));
        acc0r[h] = 0.f; acclr[h] = 0.f;
      }
    };

    // mask-cache slot of this thread's row in tile t (-1: not recorded): only rows evaluated at full precision in the first
    // sweep -- the second row segment when the first is screened, every row of a plain single-segment launch
    auto rec_slot = [&](int64_t t) -> int64_t {
      if (MODE != 0 || mask_base < 0) return -1;
      const int64_t r = row0_of(t) + rank * 64 + row;
      if (r >= lim_of(t)) return -1;
      int64_t idx;
      if (io.screen_seg1) { if (t < tiles1) return -1; idx = r - io.seg2_offset; }
      else { if (n2 > 0) return -1; idx = r; }
      const int64_t sl = mask_base + idx;
      return (sl < io.mask_cap) ? sl : -1;
    };
    const bool rec_on = (MODE == 0) && mask_base >= 0;
    // MC: code of this thread's row in tile t; a row past the end takes the last row's code (its contributions are zero,
    // and it does not split the warp's code group)
    auto code_of = [&](int64_t t) -> int {
      if constexpr (!MC) { return 0; }
      else {
        const int64_t lim = lim_of(t);
        const int64_t r = min(row0_of(t) + rank * 64 + row, lim - 1);
        return io.row_code[r] / io.code_div;
      }
    };
    int pc = 0, qc = 0;                  // MC: codes of the rows whose points are in (px, py, pz) / (qx, qy, qz)
    auto load_point = [&](int64_t t) {
      const int64_t gr = row0_of(t) + rank * 64 + row;
      if (gr < lim_of(t)) { px = io.points[gr * 3]; py = io.points[gr * 3 + 1]; pz = io.points[gr * 3 + 2]; }
      else { px = py = pz = 0.f; }
      if (MC) pc = code_of(t);
    };
    auto signal_block = [&](int kc) {   // this warp's 32 rows x 32 features of A block kc are written
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(A_FULL(kc), 0);
    };
    // layer 0 on CUDA cores: A <- split(sA * relu(b0' + W0 xyz)) for this thread's 32-feature blocks
    // guard_kc32 > 0: the previous tile's LAST layer is still being read by its final MMA pass -- block kb is overwritten
    // only once A_FREE(kb) of that layer has fired (blocks >= guard_kc32 are not read by it), so this tile's layer 0 runs
    // underneath the previous tile's last pass instead of after it
    auto layer0 = [&](int64_t slot, int guard_kc32) {
      const int kblocks = P.L[0].kc32;                          // 32-feature blocks the first MMA layer consumes
      const int nh0 = (P.N0 + 255) >> 8;
      for (int h = 0; h < nh0; ++h) {
        const int kb = 8 * h + 4 * q + ch;
        if (kb >= kblocks) continue;
        const int f0 = 32 * kb;
        uint32_t m0 = 0;
        if (kb < guard_kc32) mbar_wait(A_FREE(kb), (free_phase >> kb) & 1);
        const float* bias0 = MC ? P.bias0 + (size_t)pc * P.N0p4 : P.bias0;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float x[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int f = f0 + 8 * g + e;
            float v = 0.f;
            if (f < P.N0) {
              v = fmaf(__ldg(P.w0 + 2 * P.N0p4 + f), pz, fmaf(__ldg(P.w0 + P.N0p4 + f), py, __ldg(P.w0 + f) * px)) + __ldg(bias0 + f);
              if (v > 0.f) m0 |= 1u << (8 * g + e); else v = 0.f;
            } else if (P.first_append && f < P.N0 + 3) {
              v = (f == P.N0) ? px : ((f == P.N0 + 1) ? py : pz);
            }
            x[e] = v * sA;
          }
          store_group(smem, f0 + 8 * g, row, x);
        }
        if (MODE != 0) mk[0][h] = m0;
        if (MODE == 0 && slot >= 0) io.mask_buf[(size_t)kb * io.mask_cap + slot] = m0;      // mask cache: net layer 0
        signal_block(kb);
      }
    };
    // sum over the 32 lanes (rows) of this warp of v[j], result for column j lands in lane j  (reduce-scatter)
    auto colsum32 = [&](float (&v)[32]) -> float {
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int j = 0; j < o; ++j) {
          const float mine = up ? v[j + o] : v[j];
          const float send = up ? v[j] : v[j + o];
          v[j] = mine + __shfl_xor_sync(0xffffffffu, send, o);
        }
      }
      return v[0];
    };
    auto row_sum8 = [&]() -> float {     // fixed-order sum of the 8 partials of this row
      const float* pr = part + row * 8;
      return ((pr[0] + pr[1]) + (pr[2] + pr[3])) + ((pr[4] + pr[5]) + (pr[6] + pr[7]));
    };

    unsigned int n_tiles_1pass = 0, n_tiles_3pass = 0;   // tile programs this cluster evaluated (rank 0, warp 4, lane 0)

    // ---------------------------------------------------------------- pair mode (two one-pass tiles in lockstep, MODE 0)
    float qx = 0.f, qy = 0.f, qz = 0.f;      // this thread's point of the pair's second tile
    auto load_points_pair = [&](int i) {
      load_point(tile_of(i));
      const int64_t tb = tile_of(i + 1);
      const int64_t grb = row0_of(tb) + rank * 64 + row;
      if (i + 1 < c1 && grb < n1) { qx = io.points[grb * 3]; qy = io.points[grb * 3 + 1]; qz = io.points[grb * 3 + 2]; }
      else { qx = qy = qz = 0.f; }
      if (MC) qc = (i + 1 < c1) ? code_of(tb) : pc;
    };
    auto layer0_pair = [&](int guard_kc32) {     // layer 0 of both tiles on CUDA cores: hi halves into the two activation regions
      const int kblocks = P.L[0].kc32;
      const int nh0 = (P.N0 + 255) >> 8;
      for (int h = 0; h < nh0; ++h) {
        const int kb = 8 * h + 4 * q + ch;
        if (kb >= kblocks) continue;
        const int f0 = 32 * kb;
        if (kb < guard_kc32) mbar_wait(A_FREE(kb), (free_phase >> kb) & 1);      // (see layer0)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float xa[8], xb[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int f = f0 + 8 * g + e;
            float va = 0.f, vb = 0.f;
            if (f < P.N0) {
              const float wx = __ldg(P.w0 + f), wy = __ldg(P.w0 + P.N0p4 + f), wz = __ldg(P.w0 + 2 * P.N0p4 + f);
              float b = 0.f, bq = 0.f;
              if (MC) { b = __ldg(P.bias0 + (size_t)pc * P.N0p4 + f); bq = __ldg(P.bias0 + (size_t)qc * P.N0p4 + f); }
              else { b = __ldg(P.bias0 + f); bq = b; }
              va = fmaxf(fmaf(wz, pz, fmaf(wy, py, wx * px)) + b, 0.f);
              vb = fmaxf(fmaf(wz, qz, fmaf(wy, qy, wx * qx)) + bq, 0.f);
            } else if (P.first_append && f < P.N0 + 3) {
              va = (f == P.N0) ? px : ((f == P.N0 + 1) ? py : pz);
              vb = (f == P.N0) ? qx : ((f == P.N0 + 1) ? qy : qz);
            }
            xa[e] = va * sA; xb[e] = vb * sA;
          }
          store_group_hi(smem, OFF_AHI, f0 + 8 * g, row, xa);
          store_group_hi(smem, OFF_ALO, f0 + 8 * g, row, xb);
        }
        signal_block(kb);
      }
    };
    // MODE 3: start of a tile = its row scalars, its ReLU masks from the cache, and the seed of the transposed chain
    // (delta of the last hidden layer: w_last[f] * relu'(f), unit upstream) as the A operand of the first program layer
    float seed_scale = 0.f;
    auto seed = [&](int64_t t) {
      const int64_t r = row0_of(t) + rank * 64 + row;
      const bool ok = r < lim_of(t);
      int64_t sl = -1;
      float o = 0.f, cf = 0.f;
      if (ok) { sl = io.slots[r]; o = io.sdf_in[r]; cf = io.coef ? io.coef[r] : 1.f; }
      float d = 1.f - o * o;                                  // tanh' at the recorded output (deep_sdf_decoder.py:109-110)
      if (P.use_tanh) { const float t1 = atanhf(o); d *= (1.f - t1 * t1); }
      bool uc = io.clamp_dist > 0.f;
      if (io.use_clamp) uc = ok ? (io.use_clamp[r] != 0) : false;
      if (uc && !(o >= -io.clamp_dist && o <= io.clamp_dist)) d = 0.f;
      seed_scale = (ok && sl >= 0) ? d * cf : 0.f;
      for (int l = 0; l <= n_mma; ++l)
#pragma unroll
        for (int h = 0; h < 2; ++h)
          mk[l][h] = (ok && sl >= 0) ? io.mask_buf[((size_t)l * 16 + (8 * h + 4 * q + ch)) * io.mask_cap + sl] : 0u;
      const int LNl = P.L[n_mma - 1].N, kblocks = P.L[n_mma].kc32;
      for (int h = 0; h < 2; ++h) {
        const int kb = 8 * h + 4 * q + ch;
        if (kb >= kblocks) continue;
        const int f0 = 32 * kb;
        const uint32_t mb = mk[n_mma][h];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float x[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int f = f0 + 8 * g + e;
            x[e] = (f < LNl && ((mb >> (8 * g + e)) & 1u)) ? __ldg(P.wlast + f) * sD : 0.f;
          }
          store_group(smem, f0 + 8 * g, row, x);
        }
        signal_block(kb);
      }
    };
    // what the next tile needs before the current one is drained: its points, then (A being free) its layer 0
    auto prefetch_points = [&](int phase, int inext) {
      if (inext < 0 || MODE == 3) return;
      if (phase == 0 && inext < c1) load_points_pair(inext); else load_point(tile_of(inext));
    };
    auto start_layer0 = [&](int phase, int inext, int guard_kc32) {
      if (inext < 0) return;
      if (MODE == 3) { seed(tile_of(inext)); return; }
      if (phase == 0 && inext < c1) layer0_pair(guard_kc32); else layer0(rec_slot(tile_of(inext)), guard_kc32);
    };
    // the whole forward program of one pair (tiles i and, if has_b, i + 1 of this cluster's list)
    auto run_pair = [&](int i, int inext, bool has_b) {
      const int64_t ta = tile_of(i), tb = tile_of(i + 1);
      const int64_t gra = row0_of(ta) + rank * 64 + row, grb = row0_of(tb) + rank * 64 + row;
      const bool oka = gra < n1, okb = has_b && grb < n1;
      const int ca = MC ? code_of(ta) : 0, cb = (MC && has_b) ? code_of(tb) : ca;   // for the latent_in layer's bias
      float dota = 0.f, dotb = 0.f;
      for (int m = 0; m < n_mma; ++m, ++G) {
        const bool last = (m == n_mma - 1);
        const int LN = P.L[m].N, Lnh = P.L[m].nh, Lapp = P.L[m].app_xyz;
        const float cscale = P.L[m].inv_scale;
        const float* Lbias = P.L[m].bias;
        const int kc32_cur = P.L[m].kc32;
        const int kblocks_next = last ? 0 : P.L[m + 1].kc32;
        auto wait_h = [&](int h) {      // a pair always accumulates in TMEM buffer 0 (tile 0) and 1 (tile 1); barrier set 0
          mbar_wait(D_FULL(0, h), (d_phase >> h) & 1);
          d_phase ^= (1u << h);
          tc_fence_after();
        };
        if (last) prefetch_points(0, inext);
        for (int h = 0; h < Lnh; ++h) {
          const int kb = 8 * h + 4 * q + ch;
          const int fb = 32 * kb;
          const bool need_store = !last && kb < kblocks_next;
          const bool process = last ? (fb < LN) : need_store;
          // last layer: the next tile's layer 0 is written block by block while the final pass still runs (A_FREE guards)
          if (last && h == Lnh - 1) start_layer0(0, inext, kc32_cur);
          wait_h(h);
          if (!process) continue;
          const bool interior = (fb + 32 <= LN);
          if (h == 0 && rank == 0 && warp == 4) TL_MARK(8 + m * 4 + 2);
          if (need_store && kb < kc32_cur) mbar_wait(A_FREE(kb), (free_phase >> kb) & 1);   // the last pass has read block kb
          for (int ts = 0; ts < (has_b ? 2 : 1); ++ts) {
            float v[32];
            tmem_ld32(tmem + lane_base + ts * 256 + h * 128 + 32 * ch, v);
            const float* Lb = Lbias;
            if (MC && m == P.lat_m) Lb += (size_t)(ts ? cb : ca) * P.lat_stride;
            if (interior) {
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(Lb + fb) + j4);
                v[4 * j4] = fmaxf(fmaf(v[4 * j4], cscale, b4.x), 0.f);
                v[4 * j4 + 1] = fmaxf(fmaf(v[4 * j4 + 1], cscale, b4.y), 0.f);
                v[4 * j4 + 2] = fmaxf(fmaf(v[4 * j4 + 2], cscale, b4.z), 0.f);
                v[4 * j4 + 3] = fmaxf(fmaf(v[4 * j4 + 3], cscale, b4.w), 0.f);
              }
            } else {
              const float ax = ts ? qx : px, ay = ts ? qy : py, az = ts ? qz : pz;
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int f = fb + j;
                float a = 0.f;
                if (f < LN) a = fmaxf(fmaf(v[j], cscale, __ldg(Lb + f)), 0.f);
                else if (Lapp && f < LN + 3) a = ((f == LN) ? ax : ((f == LN + 1) ? ay : az)) * sA;
                v[j] = a;
              }
            }
            if (last) {
              float d = 0.f;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (interior || fb + j < LN) d = fmaf(v[j], __ldg(P.wlast + fb + j), d);
              if (ts) dotb += d; else dota += d;
            } else {
#pragma unroll
              for (int g = 0; g < 4; ++g) store_group_hi(smem, ts ? OFF_ALO : OFF_AHI, fb + 8 * g, row, &v[8 * g]);
            }
          }
          if (need_store) signal_block(kb);
        }
        if (rank == 0 && warp == 4) TL_MARK(8 + m * 4 + 3);
        free_phase ^= (kc32_cur >= 16) ? 0xFFFFu : ((1u << kc32_cur) - 1u);
        if (last) {
          // both accumulators are in registers: release TMEM for the next tile, then finish the two dot products
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(FIN, 0);
          for (int ts = 0; ts < (has_b ? 2 : 1); ++ts) {
            part[row * 8 + pslot] = ts ? dotb : dota;
            epi_bar_sync();
            if (pslot == 0) {
              const float sv = row_sum8() * (1.f / sA) + __ldg(P.blast);
              float o = tanhf(sv);
              if (P.use_tanh) o = tanhf(o);
              float oc = o;
              if (io.clamp_dist > 0.f) oc = fminf(fmaxf(o, -io.clamp_dist), io.clamp_dist);
              const bool ok = ts ? okb : oka;
              if (ok && io.sdf) io.sdf[ts ? grb : gra] = oc;
              if (ok && !(fabsf(o) > io.screen_thresh)) near_flag[ts] = 1u;   // may be inside the clamp band (or NaN)
            }
            epi_bar_sync();
          }
          if (ew == 0 && lane == 0) {
            for (int ts = 0; ts < (has_b ? 2 : 1); ++ts) {
              const bool fail = near_flag[ts] != 0u;
              if (fail) { fail_words[(i + ts) >> 5] |= 1u << ((i + ts) & 31); near_flag[ts] = 0u; }   // redo in phase 1
              const int64_t r0 = row0_of(ts ? tb : ta) + rank * 64;
              if (io.seg_approx && r0 < n1) io.seg_approx[r0 >> 6] = fail ? 0 : 1;
              ++n_tiles_1pass;
            }
          }
        }
      }
    };

    for (int phase = 0; phase < 2; ++phase) {
    int i = next_tile(phase, -1);
    prefetch_points(phase, i);
    start_layer0(phase, i, 0);
    while (i >= 0) {
      const int64_t t = tile_of(i);
      const int inext = next_tile(phase, i);
      if (MODE == 0 && phase == 0 && i < c1) {     // a pair of one-pass tiles
        run_pair(i, inext, i + 1 < c1);
        i = inext;
        continue;
      }
      const int64_t gr = row0_of(t) + rank * 64 + row;
      const bool row_ok = gr < lim_of(t);
      const int64_t slot = rec_slot(t);
      float dot = 0.f, rowscale = (MODE == 3) ? seed_scale : 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
      uint32_t mk0s[2] = {0u, 0u};
      // MC: this row's code, and whether the warp's 32 rows share it (then the latent gradient goes to the running sums)
      const int code_t = MC ? code_of(t) : 0;
      bool code_uni = true;
      if constexpr (MC && (MODE == 2 || MODE == 3)) {
        code_uni = __match_any_sync(0xffffffffu, code_t) == 0xffffffffu;
        if (code_uni && code_t != acc_code) { flush_sums(); acc_code = code_t; }
      }
      for (int m = m0; m < n_prog; ++m, ++G) {
        const uint32_t buf = G & 1;
        const bool fwd = m < n_mma;
        const bool fwd_last = (m == n_mma - 1);
        const bool prog_last = (m == n_prog - 1);
        const int LN = P.L[m].N, Lnh = P.L[m].nh, Lapp = P.L[m].app_xyz;
        const float cscale = P.L[m].inv_scale;
        const float* Lbias = P.L[m].bias;
        if (MC && m == P.lat_m) Lbias += (size_t)code_t * P.lat_stride;     // this row's folded bias of the latent_in layer
        const int kc32_cur = P.L[m].kc32;
        auto wait_half = [&](int h) {
          const int bi = 2 * buf + h;
          mbar_wait(D_FULL(buf, h), (d_phase >> bi) & 1);
          d_phase ^= (1u << bi);
          tc_fence_after();
        };
        // block kb of A may be overwritten once the last MMA pass of THIS layer has read it
        auto wait_free = [&](int kb) {
          if (kb < kc32_cur) mbar_wait(A_FREE(kb), (free_phase >> kb) & 1);
        };
        // the next tile's points are fetched before the wait so that their latency hides behind the last MMAs
        // (px/py/pz of this tile are no longer needed: xyz is only appended in earlier forward layers)
        // MODE 0 (forward only): the last layer's epilogue does not write A, so the next tile's layer 0 can be written block
        // by block under the final MMA pass (A_FREE guards, see layer0).  The other modes recycle A after all MMAs are done.
        constexpr bool EARLY0 = (MODE == 0);
        if (prog_last) prefetch_points(phase, inext);
        if (prog_last && !EARLY0) for (int h = 0; h < Lnh; ++h) wait_half(h);   // all MMAs of the tile done before A is recycled
#ifdef DIST_TC_TIMELINE
        const bool dbg_rec = io.dbg_out && cluster_id == 0 && rank == 0 && warp == 4 && lane == 0 && t == cluster_id + n_clusters;
#else
        const bool dbg_rec = false;
#endif
        if (prog_last && !EARLY0) {
          // all MMAs of this tile are complete: A is free -> start the next tile's layer 0 before draining D
          mk0s[0] = mk[0][0]; mk0s[1] = mk[0][1];
          start_layer0(phase, inext, 0);
        }
        const int kblocks_next = prog_last ? 0 : P.L[m + 1].kc32;
        // net layer whose ReLU mask gates the values produced here (transposed chain): l-1 with l = 2 n_mma - m
        const int mask_layer = fwd ? (m + 1) : (2 * n_mma - m - 1);
        for (int h = 0; h < Lnh; ++h) {
          const int kb = 8 * h + 4 * q + ch;             // 32-feature block index == K block of the next layer
          const int fb = 32 * kb;
          bool need_store = false, process = false;
          if (fwd && !fwd_last) { need_store = kb < kblocks_next; process = need_store; }
          else if (fwd_last) { process = fb < LN; }
          else if (!prog_last) { need_store = kb < kblocks_next; process = need_store || (Lapp && fb < LN + 3 && fb + 32 > LN); }
          else { process = fb < LN + 3 * Lapp; }
          if (EARLY0 && prog_last && h == Lnh - 1) start_layer0(phase, inext, kc32_cur);
          if (!prog_last || EARLY0) wait_half(h);       // every epilogue warp waits for each half exactly once per layer
          if (!process) continue;
          if (dbg_rec && h == 0) io.dbg_out[8 + m * 4 + 2] = clock64();
          float v[32];
          tmem_ld32(tmem + lane_base + buf * 256 + h * 128 + 32 * ch, v);
          const bool interior = (fb + 32 <= LN);            // warp-uniform: no per-element bounds checks
          if (fwd) {
            // ---- forward: bias + ReLU (deep_sdf_decoder.py:96,105); values are carried in units of sA
            uint32_t mb = 0;
            if (interior) {
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(Lbias + fb) + j4);
                const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int j = 4 * j4 + e;
                  const float a = fmaf(v[j], cscale, bb[e]);
                  if (MODE != 0 || rec_on) mb |= (a > 0.f) ? (1u << j) : 0u;
                  v[j] = fmaxf(a, 0.f);
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int f = fb + j;
                float a = 0.f;
                if (f < LN) {
                  a = fmaf(v[j], cscale, __ldg(Lbias + f));
                  if (a > 0.f) mb |= 1u << j; else a = 0.f;
                } else if (Lapp && f < LN + 3) {
                  a = ((f == LN) ? px : ((f == LN + 1) ? py : pz)) * sA;
                }
                v[j] = a;
              }
            }
            if (MODE != 0) mk[m + 1][h] = mb;
            if (MODE == 0 && slot >= 0) io.mask_buf[((size_t)(m + 1) * 16 + kb) * io.mask_cap + slot] = mb;   // mask cache
            if (fwd_last) {
              if (interior) {
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                  const float4 w4 = __ldg(reinterpret_cast<const float4*>(P.wlast + fb) + j4);
                  dot = fmaf(v[4 * j4], w4.x, dot); dot = fmaf(v[4 * j4 + 1], w4.y, dot);
                  dot = fmaf(v[4 * j4 + 2], w4.z, dot); dot = fmaf(v[4 * j4 + 3], w4.w, dot);
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (fb + j < LN) dot = fmaf(v[j], __ldg(P.wlast + fb + j), dot);
              }
            } else if (need_store) {
              wait_free(kb);
#pragma unroll
              for (int g = 0; g < 4; ++g) store_group(smem, fb + 8 * g, row, &v[8 * g]);
              signal_block(kb);
            }
          } else {
            // ---- transposed chain: gradient w.r.t. the input of net layer l = 2 n_mma - m (units of sD)
            const uint32_t mb = (mask_layer == 0 && prog_last) ? mk0s[h] : mk[mask_layer][h];
            if (interior) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = ((mb >> j) & 1u) ? v[j] * cscale : 0.f;
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int f = fb + j;
                const float g = v[j] * cscale;
                float d = 0.f;
                if (f < LN) d = ((mb >> j) & 1u) ? g : 0.f;
                else if (Lapp && f < LN + 3) { if (f == LN) dx += g; else if (f == LN + 1) dy += g; else dz += g; }
                v[j] = d;
              }
            }
            if (prog_last) {
              // delta of layer 0's pre-activation: chain to xyz through W0 (K = 3, CUDA cores)
              if (interior) {
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                  const float4 wx = __ldg(reinterpret_cast<const float4*>(P.w0 + fb) + j4);
                  const float4 wy = __ldg(reinterpret_cast<const float4*>(P.w0 + P.N0p4 + fb) + j4);
                  const float4 wz = __ldg(reinterpret_cast<const float4*>(P.w0 + 2 * P.N0p4 + fb) + j4);
                  const int j = 4 * j4;
                  dx = fmaf(v[j], wx.x, dx); dx = fmaf(v[j + 1], wx.y, dx); dx = fmaf(v[j + 2], wx.z, dx); dx = fmaf(v[j + 3], wx.w, dx);
                  dy = fmaf(v[j], wy.x, dy); dy = fmaf(v[j + 1], wy.y, dy); dy = fmaf(v[j + 2], wy.z, dy); dy = fmaf(v[j + 3], wy.w, dy);
                  dz = fmaf(v[j], wz.x, dz); dz = fmaf(v[j + 1], wz.y, dz); dz = fmaf(v[j + 2], wz.z, dz); dz = fmaf(v[j + 3], wz.w, dz);
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const int f = fb + j;
                  if (f < LN) {
                    dx = fmaf(v[j], __ldg(P.w0 + f), dx);
                    dy = fmaf(v[j], __ldg(P.w0 + P.N0p4 + f), dy);
                    dz = fmaf(v[j], __ldg(P.w0 + 2 * P.N0p4 + f), dz);
                  }
                }
              }
            } else if (need_store) {
              wait_free(kb);
#pragma unroll
              for (int g = 0; g < 4; ++g) store_group(smem, fb + 8 * g, row, &v[8 * g]);
              signal_block(kb);
            }
            if ((MODE == 2 || MODE == 3) && (prog_last || m == P.acc_l_prog)) {
              // row-sum of rowscale * delta for the latent gradient; column j of this 32-block ends in lane j
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] *= rowscale;
              if (MC && !code_uni) {
                // the warp's rows hold several codes: one reduction per code group, straight into acc[code]
                float* accp = prog_last ? io.acc0 : io.accl;
                const int Nacc = prog_last ? P.N0 : P.accl_N;
                const int f = fb + lane;
                unsigned rem = 0xffffffffu;
                while (rem) {
                  const int c = __shfl_sync(0xffffffffu, code_t, __ffs(rem) - 1);
                  const bool mine = code_t == c;
                  float w[32];
#pragma unroll
                  for (int j = 0; j < 32; ++j) w[j] = mine ? v[j] : 0.f;
                  const float sres = colsum32(w);
                  if (accp && f < Nacc && sres != 0.f) atomicAdd(accp + (size_t)c * Nacc + f, sres * (1.f / sD));
                  rem &= ~__ballot_sync(0xffffffffu, mine);
                }
              } else {
                const float sres = colsum32(v);
                if (prog_last) acc0r[h] += sres; else acclr[h] += sres;
              }
            }
          }
        }
        if (dbg_rec) io.dbg_out[8 + m * 4 + 3] = clock64();
        free_phase ^= (kc32_cur >= 16) ? 0xFFFFu : ((1u << kc32_cur) - 1u);   // A_FREE(kb), kb < kc32, completed once this layer
        if (fwd_last) {
          // combine the 8 partial dot products of each row: bias, tanh (deep_sdf_decoder.py:109-110)
          part[row * 8 + pslot] = dot;
          epi_bar_sync();
          if (pslot == 0) {
            const float s = row_sum8() * (1.f / sA) + __ldg(P.blast);
            float t1 = s, o = tanhf(s);
            if (P.use_tanh) { t1 = o; o = tanhf(o); }
            float oc = o;
            if (io.clamp_dist > 0.f) oc = fminf(fmaxf(o, -io.clamp_dist), io.clamp_dist);
            if (row_ok && io.sdf) io.sdf[gr] = oc;
            if (MODE != 0) {
              float d = 1.f - o * o;
              if (P.use_tanh) d *= (1.f - t1 * t1);
              bool uc = io.clamp_dist > 0.f;
              if (MODE == 2 && io.use_clamp) uc = row_ok ? (io.use_clamp[gr] != 0) : false;
              if (uc && !(o >= -io.clamp_dist && o <= io.clamp_dist)) d = 0.f;
              float cf = 1.f;
              if (MODE == 2 && io.coef) cf = row_ok ? io.coef[gr] : 0.f;
              if (!row_ok) cf = 0.f;
              rowd[row] = d * cf;
            }
          }
          epi_bar_sync();
          if (MODE == 0 && ew == 0 && lane == 0) {     // a single tile is always a full-precision tile (one-pass tiles: run_pair)
            if (io.seg_approx && row0_of(t) + rank * 64 < lim_of(t)) io.seg_approx[(row0_of(t) >> 6) + rank] = 0;
            ++n_tiles_3pass;
          }
          if (MODE != 0) {
            rowscale = rowd[row];
            // seed of the transposed chain (unit): delta[f] = w_last[f] * relu'(f), as A of the first transposed layer
            const int kblocks = P.L[n_mma].kc32;
            for (int h = 0; h < Lnh; ++h) {
              const int kb = 8 * h + 4 * q + ch;
              if (kb >= kblocks) continue;
              const int f0 = 32 * kb;
              const uint32_t mb = mk[n_mma][h];
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                float x[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const int f = f0 + 8 * g + e;
                  x[e] = (f < LN && ((mb >> (8 * g + e)) & 1u)) ? __ldg(P.wlast + f) * sD : 0.f;
                }
                store_group(smem, f0 + 8 * g, row, x);
              }
              signal_block(kb);
            }
          }
        }
        if (prog_last) {
          // the last accumulator is drained: release it for the second layer of the next tile
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(FIN, 0);
          if (MODE != 0) {
            // combine the 8 partial d/dxyz of each row, scale by the row's upstream factor, write out
            float res[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
              part[row * 8 + pslot] = (k == 0) ? dx : ((k == 1) ? dy : dz);
              epi_bar_sync();
              res[k] = row_sum8();
              epi_bar_sync();
            }
            if (pslot == 0 && row_ok && io.grad) {
              const float rs = rowscale * (1.f / sD);
              io.grad[gr * 3] = res[0] * rs; io.grad[gr * 3 + 1] = res[1] * rs; io.grad[gr * 3 + 2] = res[2] * rs;
            }
          }
        }
      }
      i = inext;
    }
      if (phase == 0) {
        if (!screening) break;
        cluster_sync_all();       // both CTAs' fail bitmaps are final; phase 1 re-evaluates those tiles at full precision
      }
    }
    if (io.tile_counters && rank == 0 && ew == 0 && lane == 0) {
      if (MODE != 0) n_tiles_3pass = (MODE == 3 ? 1u : 2u) * (unsigned)cnt;      // forward + transposed chain
      if (n_tiles_1pass) atomicAdd(io.tile_counters, (unsigned long long)n_tiles_1pass);
      if (n_tiles_3pass) atomicAdd(io.tile_counters + 1, (unsigned long long)n_tiles_3pass);
    }
    if (MODE == 2 || MODE == 3) flush_sums();
  }
  if (io.dbg_out && blockIdx.x == 0 && tid == 0) {
    long long t1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    io.dbg_out[0] = clock64() - dbg_c0; io.dbg_out[1] = t1 - dbg_t0;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    cudaDriverEntryPointQueryResult q;
    void* p = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess) fn = (EncodeFn)p;
  }
  return fn;
}

}  // namespace

int mlp_tc_launch(const dist_net_t* net, const NetDev& nd, int mode, const MlpArgs& a, cudaStream_t stream) {
  DIST_REQUIRE(mode >= 0 && mode <= 3, "tensor-core engine: bad mode %d", mode);
  DIST_REQUIRE(mode != 3 || (a.slots && a.sdf_in && a.mask_buf && a.mask_cap > 0), "tensor-core engine: mode 3 needs the mask cache");
  DIST_REQUIRE(net->tc_blob && net->tc_scale, "tensor-core engine: operands not prepared (tc.prepare)");
  const int nl = nd.n_layers;
  DIST_REQUIRE(nl >= 4 && nl <= 10, "tensor-core engine: %d layers unsupported", nl);
  if (a.n_host <= 0 && !a.n_dev && a.n2_host <= 0 && !a.n2_dev) return DIST_OK;
  EncodeFn encode = get_encode();
  if (!encode) { set_error("cuTensorMapEncodeTiled not available"); return DIST_E_UNSUPPORTED; }

  TcParams P;
  memset(&P, 0, sizeof(P));
  P.n_mma = nl - 2;
  P.n_prog = (mode == 0) ? P.n_mma : 2 * P.n_mma;
  P.acc_l_prog = -1;
  int stage = 0;
  for (int m = 0; m < P.n_mma; ++m) {   // forward layers: net layer l = m + 1
    const int l = m + 1;
    LayerTC& L = P.L[m];
    L.kc32 = round_up(nd.K[l], 64) / 32;
    L.nh = (nd.N[l] + 255) / 256;
    L.stage_base = stage;
    stage += L.kc32 * L.nh;
    L.N = nd.N[l];
    L.app_xyz = (l + 1 == nd.latent_in) ? 1 : 0;
    L.inv_scale = net->tc_scale[m];
    L.bias = net->tc_bias[l];
    DIST_REQUIRE(L.bias != nullptr, "tensor-core engine: scaled bias missing for layer %d", l);
    DIST_REQUIRE(nd.N[l] + 3 * L.app_xyz <= 256 * L.nh && nd.N[l] <= 512, "tensor-core engine: layer %d width unsupported", l);
  }
  for (int j = 0; j < P.n_mma; ++j) {   // transposed chain: net layer l = n_mma - j, B operand = W_l^T
    const int l = P.n_mma - j;
    LayerTC& L = P.L[P.n_mma + j];
    L.kc32 = round_up(nd.N[l], 64) / 32;
    L.nh = (nd.K[l] + 255) / 256;
    L.stage_base = stage;
    stage += L.kc32 * L.nh;
    L.N = nd.N[l - 1];
    L.app_xyz = (l == nd.latent_in) ? 1 : 0;
    L.inv_scale = net->tc_scale[P.n_mma + j];
    L.bias = nullptr;
    if (l - 1 == nd.latent_in) P.acc_l_prog = P.n_mma + j;   // this layer produces delta of the latent_in layer
  }
  DIST_REQUIRE((int64_t)stage * 2 * STAGE_BYTES == net->tc_blob_bytes, "tensor-core engine: operand blob size mismatch");
  P.accl_N = (nd.latent_in >= 0) ? nd.N[nd.latent_in] : 0;
  P.w0 = nd.Wt[0]; P.bias0 = nd.bias[0]; P.N0 = nd.N[0]; P.N0p4 = round_up(nd.N[0], 4);
  P.wlast = nd.W[nl - 1]; P.blast = nd.bias[nl - 1]; P.K_last = nd.K[nl - 1];
  P.use_tanh = nd.use_tanh; P.sA = 32.0f; P.sD = 256.0f;
  P.first_append = (nd.latent_in == 1) ? 1 : 0;
  P.lat_m = (nd.latent_in >= 1) ? nd.latent_in - 1 : -1;
  P.lat_stride = (nd.latent_in >= 1) ? round_up(nd.N[nd.latent_in], 4) : 0;
  const bool mc = nd.n_codes > 1;
  DIST_REQUIRE(!mc || (a.row_code && a.code_div > 0), "tensor-core engine: %d latent codes need per-row codes", nd.n_codes);
  { const char* e = getenv("DIST_TC_DEBUG"); P.dbg = e ? atoi(e) : 0; }

  TcIO io;
  io.points = a.points; io.n_host = a.n_host; io.n_dev = a.n_dev; io.clamp_dist = a.clamp_dist;
  io.sdf = a.sdf; io.grad = a.grad; io.coef = a.coef; io.use_clamp = a.use_clamp; io.acc0 = a.acc0; io.accl = a.accl;
  io.rows_evaluated = a.rows_evaluated;
  io.n2_host = a.n2_host; io.n2_dev = a.n2_dev; io.seg2_offset = a.seg2_offset;
  io.screen_seg1 = (mode == 0) ? a.screen_seg1 : 0;
  io.screen_thresh = a.screen_thresh; io.seg_approx = a.seg_approx;
  io.tile_counters = a.tile_counters;
  io.mask_buf = a.mask_buf; io.mask_cap = a.mask_cap; io.mask_base_host = a.mask_buf ? a.mask_base_host : -1;
  io.mask_base_dev = a.mask_base_dev; io.slots = a.slots; io.sdf_in = a.sdf_in;
  io.row_code = mc ? a.row_code : nullptr; io.code_div = mc ? a.code_div : 1;
  DIST_REQUIRE(!io.screen_seg1 || io.seg_approx != nullptr, "tensor-core engine: two-tier precision needs seg_approx");
  DIST_REQUIRE((a.n2_host == 0 && !a.n2_dev) || (a.seg2_offset % 128 == 0 && a.seg2_offset >= a.n_host),
               "tensor-core engine: the second row segment must start at a multiple of 128 behind the first");
  io.dbg_out = nullptr;
  static long long* dbg_buf = nullptr;
  if (P.dbg & 4) { if (!dbg_buf) { cudaMalloc(&dbg_buf, 4096); cudaMemset(dbg_buf, 0, 4096); } io.dbg_out = dbg_buf; }

  // tensor map over the blob, which is laid out stage by stage: one box = one contiguous 16 KB stage of one CTA.  The box row
  // length only decides how many row requests the TMA unit issues per stage (DIST_TC_BOXROW = 128/256/512 bytes: measured
  // identical, profiles/r2_tc_summary.md -- the weight stream is not limited by TMA request issue)
  static const int boxrow = [] { const char* e = getenv("DIST_TC_BOXROW"); int v = e ? atoi(e) : 128;
                                 return (v == 128 || v == 256 || v == 512) ? v : 128; }();
  P.stage_rows = STAGE_BYTES / boxrow;
  CUtensorMap tmap;
  const cuuint64_t rows = (cuuint64_t)(net->tc_blob_bytes / boxrow);
  const cuuint64_t gdim[2] = {(cuuint64_t)(boxrow / 2), rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)boxrow};
  const cuuint32_t box[2] = {(cuuint32_t)(boxrow / 2), (cuuint32_t)(STAGE_BYTES / boxrow)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(net->tc_blob), gdim, gstr, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)cr); return DIST_E_CUDA; }
  // same blob, boxes of the first 8 KB ([hi]) of a stage only: what a one-pass tile fetches
  CUtensorMap tmap_hi;
  const cuuint32_t box_hi[2] = {(cuuint32_t)(boxrow / 2), (cuuint32_t)(STAGE_BYTES / 2 / boxrow)};
  cr = encode(&tmap_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(net->tc_blob), gdim, gstr, box_hi, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (hi box) failed (%d)", (int)cr); return DIST_E_CUDA; }

  static bool attr_done_dev[64] = {false};
  int cur_dev = 0;
  cudaGetDevice(&cur_dev);
  bool& attr_done = attr_done_dev[cur_dev & 63];
  if (!attr_done) {
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    DIST_CHECK_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_done = true;
  }
  const int64_t tiles = (a.n_host + 127) / 128 + (a.n2_host + 127) / 128;   // capacities when the counts live on the device
  int clusters = num_sms() / 2;
  if (tiles < clusters) clusters = (int)tiles;
  if (clusters < 1) clusters = 1;
  const int g = clusters * 2;
  if (!mc) {
    if (mode == 0) { mlp_tc_kernel<0, false><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
    else if (mode == 1) { mlp_tc_kernel<1, false><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
    else if (mode == 2) { mlp_tc_kernel<2, false><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
    else { mlp_tc_kernel<3, false><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
  } else {
    if (mode == 0) { mlp_tc_kernel<0, true><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
    else if (mode == 1) { mlp_tc_kernel<1, true><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
    else if (mode == 2) { mlp_tc_kernel<2, true><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
    else { mlp_tc_kernel<3, true><<<g, NTHREADS, SMEM_BYTES, stream>>>(tmap, tmap_hi, P, io); }
  }
  count_launch();
  DIST_CHECK_CUDA(cudaGetLastError());
  if (P.dbg & 4) {
    long long h[2] = {0, 0};
    cudaStreamSynchronize(stream);
    cudaMemcpy(h, dbg_buf, 16, cudaMemcpyDeviceToHost);
    fprintf(stderr, "[tc dbg] mode %d: %lld cycles, %lld ns -> %.3f GHz\n", mode, h[0], h[1], h[1] ? (double)h[0] / h[1] : 0.0);
#ifdef DIST_TC_TIMELINE
    {
      long long ev[256];
      cudaMemcpy(ev, dbg_buf, 2048, cudaMemcpyDeviceToHost);
      const long long t0 = ev[8];
      fprintf(stderr, "[tc dbg] previous tile: last MMA issue at %lld (relative to this tile's first MMA)\n", ev[200] - t0);
      long long wt[64];
      cudaMemcpy(wt, dbg_buf + 256, sizeof(wt), cudaMemcpyDeviceToHost);
      for (int m = 0; m < P.n_prog; ++m)
        fprintf(stderr, "[tc dbg] layer %2d: mma start %7lld  issue end %7lld | epi start %7lld  epi end %7lld | issuer waited for A %6lld, for W %6lld\n",
                m, ev[8 + m * 4] - t0, ev[8 + m * 4 + 1] - t0, ev[8 + m * 4 + 2] - t0, ev[8 + m * 4 + 3] - t0, wt[2 * m], wt[2 * m + 1]);
      cudaMemset(dbg_buf + 256, 0, sizeof(wt));
    }
#endif
  }
  return DIST_OK;
}

}  // namespace dist
