/*
 * sdfrender.cu -- sm_100a kernels and C ABI of libsdfrender.so (see include/sdfrender.h).
 *
 * Replaces the reference's sdf_renderer_cpp extension (sdf_renderer.cpp:42-91,
 * sdf_renderer_cuda.cu:241-556).  Design (DESIGN.md has the long version):
 *
 *  - one launch renders a whole BATCH of hypotheses (blockIdx.z), the reference renders one
 *    object per launch plus 1 (fwd) / 4 (bwd) memset launches;
 *  - a CTA owns a 32x8 pixel tile; warp w owns the 8x4 sub-tile so that the 32 rays of a warp
 *    stay spatially coherent (their 8-corner gathers fall into 1-4 L1 lines) and the depth
 *    stores fill whole 32-byte sectors;
 *  - warp 0 builds the per-hypothesis Frame (rotation, object-frame origin, slab constants and
 *    the screen rectangle of the projected box) once per CTA; CTAs / warps outside the
 *    rectangle only zero-fill -- 64-99 % of the pixels of the reference workloads;
 *  - un-normalised ray components come from two per-CTA tables evaluated in double exactly as
 *    the reference does per thread (cu:146-147): 40 double divisions per CTA instead of 512;
 *  - the grid is read through the read-only path (LDG.E.CONSTANT) and stays L1/L2 resident
 *    (1 MiB at 64^3; 126 MB of L2 hold 64 distinct hypothesis grids);
 *  - backward: pose/scale gradients reduce warp-shuffle -> shared memory -> 8 atomics per CTA
 *    (the reference issues 8 same-address atomics per hit pixel, cu:459-466); SDF gradients
 *    scatter with fire-and-forget RED.ADD.F32; `flags` prunes what is not needed;
 *  - the fused render-and-compare pair evaluates the masked-L1 depth loss inside the render
 *    kernel and rebuilds the loss gradient inside the backward kernel, so no grad_depth image
 *    is ever materialised.
 *
 * No tensor cores: the path is a dependent gather chain, not a contraction.
 */
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/sdfrender.h"
#include "sdfr_core.cuh"

/* The library is one source file compiled either whole (SDFR_PART undefined / 0) or as four
 * translation units in parallel (sdfest_b200/build.py: -DSDFR_PART=1..4; 1 = forward, 2 = fused
 * forward, 3 = backward / composite / grid passes, 4 = point loss, decoder, optimiser step). */
#ifndef SDFR_PART
#define SDFR_PART 0
#endif
#define SDFR_IN_PART(k) (SDFR_PART == 0 || SDFR_PART == (k))

namespace sdfr_detail {
#if SDFR_PART <= 1
thread_local char g_err[256] = "";
#else
extern thread_local char g_err[256];
#endif
}  // namespace sdfr_detail

namespace {

using namespace sdfr;
using sdfr_detail::g_err;

constexpr int kTileW = 32;
constexpr int kTileH = 8;
constexpr int kThreads = kTileW * kTileH;  // 256 = 8 warps of 8x4 pixels
constexpr int kWarps = kThreads / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kListCap = 1024; /* warp tiles per work-list chunk of the forward kernels */

int fail(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

struct Pose {
  const float* __restrict__ position;     // [B,3]
  const float* __restrict__ orientation;  // [B,4]
  const float* __restrict__ inv_scale;    // [B]
  const CellBounds* __restrict__ bounds;  // optional cell bounds of the grids (sdfr_grid_bounds)
  int bounds_stride;                      // 0: one entry shared by all hypotheses, 1: one per hypothesis
  int R;
  float threshold;
};

struct FwdParams {
  const float* __restrict__ sdf;
  long long sdf_stride;
  Pose pose;
  Grid grid;
  Camera cam;
  float threshold;
  float* __restrict__ depth;  // [B,H,W]
  int z_offset;               // first hypothesis of this launch (gridDim.y chunking)
  int use_tables;             // ray tables fit in shared memory
  int steal;                  // more CTAs than fit at once: CTAs render unlaunched CTAs' items (WorkSteal)
  int image_tables;           // use_tables, steal and several tiles per CTA: ray tables of the whole image, once
  // compare
  const float* __restrict__ depth_obs;
  long long obs_stride;
  float* __restrict__ loss_sum;
  float* __restrict__ n_overlap;
  float* __restrict__ n_inlier;  // optional: overlap pixels with |obs - est| / obs < inlier_threshold
  float inlier_threshold;
  // stats
  unsigned long long* __restrict__ stats;
  // fused compare + backward (unnormalised gradients)
  float* __restrict__ grad_sdf;
  long long grad_sdf_stride;
  float* __restrict__ grad_position;
  float* __restrict__ grad_orientation;
  float* __restrict__ grad_inv_scale;
  unsigned flags;
};

struct BwdParams {
  const float* __restrict__ grad_depth;  // PLAIN / COMPOSITE
  const float* __restrict__ depth;
  const float* __restrict__ sdf;
  long long sdf_stride;
  Pose pose;
  Grid grid;
  Camera cam;
  float* __restrict__ grad_sdf;
  long long grad_sdf_stride;
  float* __restrict__ grad_position;
  float* __restrict__ grad_orientation;
  float* __restrict__ grad_inv_scale;
  unsigned flags;
  int z_offset;
  int use_tables;
  // compare
  const float* __restrict__ depth_obs;
  long long obs_stride;
  const float* __restrict__ n_overlap;
  const float* __restrict__ upstream;
  // composite
  const int* __restrict__ winner;
  int n_objects;
};

/* Built by warp 0: pose part by every lane (registers), the 8 box corners by lanes 0-7, the 28
 * corner pairs that may carry a silhouette edge by lanes 0-27 (edges == nullptr: no hull). */
__device__ __forceinline__ void build_frame(Frame& smemF, HullEdge* edges, const Pose& pose, int b,
                                            const Camera& cam, int lane) {
  Frame F;
  frame_pose(F, pose.position + 3 * b, pose.orientation + 4 * b, pose.inv_scale + b,
             pose.bounds ? pose.bounds + (size_t)b * pose.bounds_stride : nullptr, pose.R, pose.threshold);
  float col = 0.f, row = 0.f;
  const bool ok = project_corner(F, cam, lane & 7, col, row);
  const bool all_ok = __all_sync(kFull, ok);
  float cmin = col, cmax = col, rmin = row, rmax = row;
#pragma unroll
  for (int o = 4; o >= 1; o >>= 1) {
    cmin = fminf(cmin, __shfl_xor_sync(kFull, cmin, o));
    cmax = fmaxf(cmax, __shfl_xor_sync(kFull, cmax, o));
    rmin = fminf(rmin, __shfl_xor_sync(kFull, rmin, o));
    rmax = fmaxf(rmax, __shfl_xor_sync(kFull, rmax, o));
  }
  if (lane == 0) {
    frame_rect(F, cam, all_ok, cmin, cmax, rmin, rmax);
    smemF = F;
  }
  if (edges != nullptr) { /* same selection as build_hull_serial: first 8 accepted pairs */
    const bool sane =
        all_ok && __all_sync(kFull, fabsf(col) <= kHullCoordMax && fabsf(row) <= kHullCoordMax);
    int i = 0, j = 1;
    if (lane < 28) hull_pair(lane, i, j);
    const float xi = __shfl_sync(kFull, col, i), yi = __shfl_sync(kFull, row, i);
    const float xj = __shfl_sync(kFull, col, j), yj = __shfl_sync(kFull, row, j);
    float a = 0.f, bb = 0.f, c = 0.f;
    const bool line = sane && lane < 28 && hull_line(xi, yi, xj, yj, a, bb, c);
    float smin = 1e30f, smax = -1e30f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float sd = a * __shfl_sync(kFull, col, k) + bb * __shfl_sync(kFull, row, k) + c;
      smin = fminf(smin, sd);
      smax = fmaxf(smax, sd);
    }
    HullEdge e;
    e.a = 0.f; e.b = 0.f; e.c = 1.f; e.pad = 0.f;
    const bool valid = line && hull_accept(a, bb, c, smin, smax, e);
    const unsigned m = __ballot_sync(kFull, valid);
    const int slot = __popc(m & ((1u << lane) - 1u));
    if (valid && slot < kMaxHullEdges) edges[slot] = e;
    const int n = min(__popc(m), kMaxHullEdges);
    if (lane < kMaxHullEdges && lane >= n) { /* always-true padding */
      HullEdge t;
      t.a = 0.f; t.b = 0.f; t.c = 1.f; t.pad = 0.f;
      edges[lane] = t;
    }
  }
}

/* n / d for 0 <= n < 2^24, d > 0 with a reciprocal computed once (rd = 1.0f / d): the tile loops divide by the
 * same run-time width for every candidate, and an integer division is ~25 instructions */
__device__ __forceinline__ int div_by(int n, int d, float rd) {
  int q = __float2int_rz(__int2float_rn(n) * rd);
  const int rem = n - q * d;
  q += rem >= d ? 1 : 0;
  q -= rem < 0 ? 1 : 0;
  return q;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

/*
 * Work decomposition of the batched kernels.
 *
 * grid = (G, hypotheses): G persistent CTAs per hypothesis.  A CTA builds the hypothesis' Frame
 * and the ray tables ONCE (the forward kernels: once per logical CTA, and a resident CTA renders
 * several logical CTAs when it can steal them, see WorkSteal), then walks the 32x8-pixel tiles
 * g, g+G, g+2G, ... of that hypothesis without any further barrier: tiles outside the projected box are only zero-filled, tiles
 * inside are traced.  Per-pixel results that need a reduction (loss sums, pose gradients,
 * counters) accumulate in registers across the CTA's tiles and are reduced once at the end.
 * (Round 1 first shipped one CTA per tile: 76 800 CTAs with a prologue + barrier each -- ncu
 * showed 37 % of the stall samples on those barriers and 60 % of the executed instructions
 * outside the march loop; profiles/r01_notes.md.)
 */
struct Tiling {
  int tiles_x, tiles_y;      /* tile grid of the whole image */
  int rtx0, rty0, rtw, rth;  /* tile range covering the projected box */
  int tab_x0, tab_y0;        /* first tile column / row held by the ray tables */
};

/* (row, col) walk over a w-wide tile range in steps of G tiles without integer division in
 * the loop: one division at start, then add-and-carry. */
struct TileWalk {
  int ty, tx, dy, dx, w;
  __device__ __forceinline__ TileWalk(int first, int G, int w_) : w(w_) {
    const int ww = w_ > 0 ? w_ : 1;
    ty = first / ww;
    tx = first - ty * ww;
    dy = G / ww;
    dx = G - dy * ww;
  }
  __device__ __forceinline__ void next() {
    tx += dx;
    ty += dy;
    if (tx >= w) {
      tx -= w;
      ty += 1;
    }
  }
};

__device__ __forceinline__ Tiling make_tiling(const Frame& F, const Camera& cam) {
  Tiling T;
  T.tiles_x = (cam.W + kTileW - 1) / kTileW;
  T.tiles_y = (cam.H + kTileH - 1) / kTileH;
  if (F.x1 <= F.x0 || F.y1 <= F.y0) {
    T.rtx0 = T.rty0 = T.rtw = T.rth = 0;
  } else {
    T.rtx0 = F.x0 / kTileW;
    T.rty0 = F.y0 / kTileH;
    T.rtw = (F.x1 + kTileW - 1) / kTileW - T.rtx0;
    T.rth = (F.y1 + kTileH - 1) / kTileH - T.rty0;
  }
  T.tab_x0 = T.rtx0;
  T.tab_y0 = T.rty0;
  return T;
}

/* CTA prologue of logical CTA (g, b): Frame by warp 0, then -- with fill_tables -- the ray tables
 * (double-precision divisions as in cu:146-147, amortised over all tiles of the CTA).  When the CTA
 * owns at most one tile of the box (small batches: G >= number of box tiles) only that tile's
 * 32 + 8 entries are built.  Without fill_tables the tables are either unused or already hold the
 * whole image (fill_image_tables). */
__device__ __forceinline__ Tiling cta_prologue(Frame& Fs, HullEdge* edges, float* tables,
                                               bool fill_tables, const Pose& pose, int g, int b,
                                               const Camera& cam, float*& colx, float*& rowy) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) build_frame(Fs, edges, pose, b, cam, lane);
  __syncthreads();
  Tiling T = make_tiling(Fs, cam);
  colx = tables;
  rowy = tables + T.tiles_x * kTileW;
  if (fill_tables) {
    const int n_rect = T.rtw * T.rth;
    int ncol = T.rtw * kTileW, nrow = T.rth * kTileH;
    if (n_rect <= (int)gridDim.x) { /* this CTA traces tile g of the box, or nothing */
      if (g < n_rect) {
        const int ty = g / T.rtw;
        T.tab_x0 = T.rtx0 + (g - ty * T.rtw);
        T.tab_y0 = T.rty0 + ty;
        ncol = kTileW;
        nrow = kTileH;
      } else {
        ncol = nrow = 0;
      }
    }
    /* the tables span the whole image (table_bytes) and are indexed by the ABSOLUTE column / row; only the
     * entries of the CTA's tiles are filled.  (Indexing relative to tab_x0 / tab_y0 kept those two integers
     * live across the march: ptxas spilled them, and the reload in front of every warp tile's table look-up
     * was 3 % of the fused kernel's stall samples.) */
    for (int i = threadIdx.x; i < ncol; i += kThreads)
      colx[T.tab_x0 * kTileW + i] = pixel_dx(T.tab_x0 * kTileW + i, cam.cx, cam.fx);
    for (int i = threadIdx.x; i < nrow; i += kThreads)
      rowy[T.tab_y0 * kTileH + i] = pixel_dy(T.tab_y0 * kTileH + i, cam.cy, cam.fy);
    __syncthreads();
  }
  return T;
}

/* Ray tables of the whole image: they depend on the camera only, so a CTA that renders several
 * logical CTAs (WorkSteal) builds them once.  The caller synchronises before the first read. */
__device__ __forceinline__ void fill_image_tables(float* tables, const Camera& cam) {
  const int ncol = (cam.W + kTileW - 1) / kTileW * kTileW, nrow = (cam.H + kTileH - 1) / kTileH * kTileH;
  for (int i = threadIdx.x; i < ncol; i += kThreads) tables[i] = pixel_dx(i, cam.cx, cam.fx);
  for (int i = threadIdx.x; i < nrow; i += kThreads) tables[ncol + i] = pixel_dy(i, cam.cy, cam.fy);
}

/*
 * Work stealing by cluster launch control (sm_100, PTX clusterlaunchcontrol.*): a CTA that has
 * finished its logical CTA cancels one that the hardware has not launched yet and renders that one
 * itself, so the per-CTA fixed costs are paid about once per resident CTA.  Nothing lives in global
 * memory: no counter to reset between graph replays, nothing shared between two launches in flight.
 * The first warp that finds the work list of the current item empty issues the request for the next
 * one (the answer arrives while the other warps finish; issued at the start of the item instead, a
 * busy CTA reserved work that a CTA finishing sooner could have started: fused launch +2 us instead
 * of -10 us, DESIGN.md section 5).  Thread 0 waits on the mbarrier at the end of the item and
 * publishes the next item in `next_g`, `next_b` (next_g < 0: no CTA left to take, the CTA exits).
 * A failed request is never followed by another one (undefined in the PTX ISA): the loop ends on
 * it.  The current item is
 * copied to `g`, `b` at the start of each item and read back from there where it is needed (item_g,
 * item_b): blockIdx was a special register that ptxas re-read at will, a loop variable would be two
 * more registers live across the march.
 */
struct WorkSteal {
  alignas(16) unsigned long long response[2]; /* try_cancel response, written by the async proxy */
  unsigned long long bar;                      /* mbarrier: one arrival + 16 transaction bytes per request */
  unsigned phase;                              /* parity of the request in flight (thread 0 only) */
  int g, b;                                    /* current logical CTA: tile group, hypothesis (+ z_offset) */
  int next_g, next_b;                          /* the one after it: blockIdx.x, blockIdx.y */
  int requested;                               /* the request for next_g / next_b has been issued */
};

__device__ __forceinline__ int item_g(const WorkSteal& ws) { return *reinterpret_cast<const volatile int*>(&ws.g); }
__device__ __forceinline__ int item_b(const WorkSteal& ws) { return *reinterpret_cast<const volatile int*>(&ws.b); }

__device__ __forceinline__ void steal_init(WorkSteal& ws) {
  if (threadIdx.x == 0) {
    ws.next_g = blockIdx.x;
    ws.next_b = blockIdx.y;
    ws.phase = 0;
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(&ws.bar))
                 : "memory");
  }
}

/* one thread: ask for the next logical CTA (thread 0 read the response buffer before the last barrier) */
__device__ __forceinline__ void steal_request(WorkSteal& ws) {
  const unsigned resp = (unsigned)__cvta_generic_to_shared(ws.response);
  const unsigned bar = (unsigned)__cvta_generic_to_shared(&ws.bar);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("clusterlaunchcontrol.try_cancel.async.shared::cta.mbarrier::complete_tx::bytes.b128 [%0], [%1];"
               ::"r"(resp), "r"(bar) : "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 16;" ::"r"(bar) : "memory");
}

/* thread 0: wait for the answer and publish the next item (next_g = -1: none, or nothing was asked) */
__device__ __forceinline__ void steal_next(WorkSteal& ws) {
  if (!ws.requested) {
    ws.next_g = -1;
    return;
  }
  const unsigned bar = (unsigned)__cvta_generic_to_shared(&ws.bar);
  unsigned done = 0;
  do {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(ws.phase) : "memory");
  } while (!done);
  ws.phase ^= 1u;
  unsigned long long lo, hi;
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];"
               : "=l"(lo), "=l"(hi) : "r"((unsigned)__cvta_generic_to_shared(ws.response)) : "memory");
  unsigned ok = 0;
  asm volatile("{\n\t.reg .b128 q;\n\t.reg .pred p;\n\t"
               "mov.b128 q, {%1, %2};\n\t"
               "clusterlaunchcontrol.query_cancel.is_canceled.pred.b128 p, q;\n\t"
               "selp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok)
               : "l"(lo), "l"(hi));
  if (!ok) {
    ws.next_g = -1;
    return;
  }
  unsigned x, y;
  asm volatile("{\n\t.reg .b128 q;\n\t"
               "mov.b128 q, {%2, %3};\n\t"
               "clusterlaunchcontrol.query_cancel.get_first_ctaid.v4.b32.b128 {%0, %1, _, _}, q;\n\t}"
               : "=r"(x), "=r"(y)
               : "l"(lo), "l"(hi));
  ws.next_g = (int)x;
  ws.next_b = (int)y;
}

template <int RT>
__device__ __forceinline__ void scatter_sdf(float* __restrict__ gs, const Grid& G, int base,
                                            const float (&w)[8]) {
  const int R = RT > 0 ? RT : G.R, R2 = R * R;
  gs += base;
  atomicAdd(gs, w[0]);
  atomicAdd(gs + 1, w[1]);
  atomicAdd(gs + R, w[2]);
  atomicAdd(gs + R + 1, w[3]);
  atomicAdd(gs + R2, w[4]);
  atomicAdd(gs + R2 + 1, w[5]);
  atomicAdd(gs + R2 + R, w[6]);
  atomicAdd(gs + R2 + R + 1, w[7]);
}

/*
 * Warp-aggregated scatter: neighbouring rays of an 8x4 warp tile mostly end in the same grid cell
 * (a 64^3 grid seen at 640x480 spans ~4 pixels per cell), so their 8 corner contributions are first
 * merged inside the warp -- a 5-level butterfly in which two lanes merge when both still carry a
 * contribution for the SAME cell -- and only the surviving lanes issue RED.ADD.F32.  Must be called
 * by all 32 lanes; `has` marks lanes that carry a contribution.
 */
template <int RT>
__device__ __forceinline__ void scatter_sdf_warp(float* __restrict__ gs, const Grid& G, int base,
                                                 float (&w)[8], bool has, int lane) {
  const int key = has ? base : -1;
  bool alive = has;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const int pkey = __shfl_xor_sync(kFull, key, 1 << k);
    const bool palive = __shfl_xor_sync(kFull, (int)alive, 1 << k) != 0;
    const bool merge = alive && palive && pkey == key;
    const bool lower = (lane & (1 << k)) == 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float o = __shfl_xor_sync(kFull, w[i], 1 << k);
      if (merge && lower) w[i] += o;
    }
    if (merge && !lower) alive = false;
  }
  if (alive) scatter_sdf<RT>(gs, G, base, w);
}

/* Pose gradients of a CTA.  Every thread keeps its 13 moment sums (sdfr_core.cuh:
 * pixel_backward_moments) in SHARED memory, acc_s[i][thread] -- 13 registers that would otherwise be
 * live across the whole march loop (they were the fused kernel's spill).  A hit pixel costs 13
 * conflict-free read-modify-writes.  At the end: warp shuffle -> warp 0 applies the 13 -> 8 map of the
 * hypothesis once -> 8 atomics per CTA (the reference issues 8 same-address atomics per hit pixel,
 * cu:459-466).  Measured and dropped: double-precision per-thread sums (+30 us on the 240 us fused
 * launch: the B200's DADD / F2F.F64 rate) and a double-precision reduction + map in one thread (+15 us:
 * a serial chain of ~200 DP operations per CTA); neither moved the error, which is the fp32 rounding of
 * the per-pixel products.  Contains two barriers: call from uniform control flow. */
typedef float MomentAcc[kMoments][kThreads];

__device__ __forceinline__ void moments_clear(MomentAcc& acc_s) {
#pragma unroll
  for (int i = 0; i < kMoments; ++i) acc_s[i][threadIdx.x] = 0.0f;
}

__device__ __forceinline__ void moments_add(MomentAcc& acc_s, const float (&m)[kMoments]) {
#pragma unroll
  for (int i = 0; i < kMoments; ++i) acc_s[i][threadIdx.x] += m[i];
}

__device__ __forceinline__ void reduce_pose(MomentAcc& acc_s, const Frame& F, const Grid& G, int b,
                                            float* gp, float* gq, float* gi, unsigned flags) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __shared__ float totals[kMoments];
  __syncthreads();
  /* warp w sums moments w, w + 8 over the 256 threads */
  for (int i = warp; i < kMoments; i += kWarps) {
    float v = 0.0f;
#pragma unroll
    for (int j = 0; j < kThreads / 32; ++j) v += acc_s[i][lane + 32 * j];
    v = warp_sum(v);
    if (lane == 0) totals[i] = v;
  }
  __syncthreads();
  if (warp == 0) {
    float m[kMoments];
#pragma unroll
    for (int i = 0; i < kMoments; ++i) m[i] = totals[i];
    float out[8];
    moments_to_pose(F, G, m, out);
    float v = out[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) v = lane == i ? out[i] : v;
    if (lane < 8 && v != 0.0f) {
      if (lane < 3) {
        if (flags & SDFR_GRAD_POSITION) atomicAdd(gp + 3 * b + lane, v);
      } else if (lane < 7) {
        if (flags & SDFR_GRAD_ORIENTATION) atomicAdd(gq + 4 * b + (lane - 3), v);
      } else {
        if (flags & SDFR_GRAD_INV_SCALE) atomicAdd(gi + b, v);
      }
    }
  }
}

/* grad_sdf *= coef over the voxels of one hypothesis that can hold a gradient: the cells inside the empty-space
 * bounds the render used (every other voxel is still the zero it was cleared to), or the whole grid without
 * bounds.  `warp` of `n_warps` warps share the rows; loads bypass L1 (the values were written by RED.ADDs of
 * other SMs).  Four rows per step: the loads of all four are in flight before the first store (one dependent
 * round trip per row otherwise: 22.8 us for the stand-alone pass at C2). */
__device__ __forceinline__ void scale_sdf_grads(float* __restrict__ gs, const CellBounds* __restrict__ cbp, int R,
                                                long long grid_elems, float coef, int warp, int n_warps, int lane) {
  if (cbp) {
    const CellBounds cb = *cbp;
    if (cb.lo[0] > cb.hi[0]) return; /* no cell can be hit: the grid is all zeros */
    /* voxels of cells lo..hi are lo..hi+1; rows (x, y) of the box, a warp per row, lanes along z */
    const int x0 = cb.lo[0], nx = cb.hi[0] - cb.lo[0] + 2, y0 = cb.lo[1], ny = cb.hi[1] - cb.lo[1] + 2;
    const int z0 = cb.lo[2], z1 = cb.hi[2] + 1;
    if ((R & 3) == 0 && (reinterpret_cast<uintptr_t>(gs) & 15) == 0) {
      /* aligned 16-byte accesses over the z-range rounded out to multiples of four (the extra voxels are the
       * zeros the grid was cleared to), eight independent loads per thread in flight before the first store:
       * the single CTA that normalises a hypothesis inside the render launch moves its ~200 KB in a handful of
       * round trips instead of one per row */
      const int zv0 = z0 >> 2, nv = (z1 >> 2) - zv0 + 1, total = nx * ny * nv;
      const int tid = warp * 32 + lane, nthr = n_warps * 32;
      for (int i0 = tid; i0 < total; i0 += 8 * nthr) {
        float4 v[8];
        float4* p[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int i = i0 + j * nthr;
          const bool ok = i < total;
          const int ii = ok ? i : i0;
          const int r = ii / nv, k = ii - r * nv;
          const int rx = r / ny, ry = r - rx * ny;
          p[j] = reinterpret_cast<float4*>(gs + ((size_t)(x0 + rx) * R + (y0 + ry)) * R) + zv0 + k;
          v[j] = ok ? __ldcg(p[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (i0 + j * nthr < total) *p[j] = make_float4(v[j].x * coef, v[j].y * coef, v[j].z * coef, v[j].w * coef);
      }
      return;
    }
    for (int r0 = warp; r0 < nx * ny; r0 += 4 * n_warps) {
      for (int z = z0 + lane; z <= z1; z += 32) {
        float v[4];
        float* p[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = r0 + j * n_warps;
          const bool ok = r < nx * ny;
          const int rr = ok ? r : r0;
          p[j] = gs + ((size_t)(x0 + rr / ny) * R + (y0 + rr % ny)) * R + z;
          v[j] = ok ? __ldcg(p[j]) : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (r0 + j * n_warps < nx * ny) *p[j] = v[j] * coef;
      }
    }
    return;
  }
  const long long n4 = ((reinterpret_cast<uintptr_t>(gs) & 15) == 0) ? grid_elems / 4 : 0;
  float4* __restrict__ gs4 = reinterpret_cast<float4*>(gs);
  for (long long i = (long long)warp * 32 + lane; i < n4; i += (long long)n_warps * 32) {
    float4 v = __ldcg(gs4 + i);
    v.x *= coef; v.y *= coef; v.z *= coef; v.w *= coef;
    gs4[i] = v;
  }
  for (long long i = n4 * 4 + (long long)warp * 32 + lane; i < grid_elems; i += (long long)n_warps * 32)
    gs[i] = __ldcg(gs + i) * coef;
}

/* ------------------------------------------------------------------------------------------
 * Forward (replaces sdf_renderer_cuda_forward_kernel, cu:241-298).
 * MODE 0: depth only.  MODE 1: + masked-L1 compare sums.  MODE 2: + the backward of that loss
 * fused into the same traversal (unnormalised: d/d theta of sum |est - obs|; the per-hypothesis
 * factor upstream/n_overlap is only known once all pixels are done and is applied afterwards by
 * sdfr_scale_grads -- every gradient is linear in it).
 * ---------------------------------------------------------------------------------------- */
constexpr int kFwdBlocks = 5; /* resident CTAs per SM the forward kernels are register-budgeted for */
template <int RT, int LT, int MODE, bool STATS, bool WANT_SDF, bool WANT_POSE>
__global__ void __launch_bounds__(kThreads, kFwdBlocks)
sdfr_forward_kernel(const __grid_constant__ FwdParams P) {
  extern __shared__ float tables[];
  __shared__ Frame Fs;
  __shared__ HullEdge edges[kMaxHullEdges];
  __shared__ float acc_mem[(MODE == 2 && WANT_POSE) ? kMoments * kThreads : 1];
  MomentAcc& acc_s = *reinterpret_cast<MomentAcc*>(acc_mem);
  __shared__ int next_q, n_live;
  __shared__ unsigned worklist[kListCap];
  __shared__ WorkSteal ws;

  steal_init(ws);
  if (P.image_tables) fill_image_tables(tables, P.cam);
  __syncthreads();
  /* one logical CTA (g, b) per iteration: blockIdx first, then the CTAs this one cancels */
  for (;;) {
    const int b = ws.next_b + P.z_offset;
    const int g = ws.next_g, G = gridDim.x;
    if (threadIdx.x == 0) { /* read again from ws after cta_prologue's barrier */
      ws.g = g;
      ws.b = b;
      ws.requested = 0;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lane_x = lane & 7, lane_y = lane >> 3;
    const int W = P.cam.W, H = P.cam.H;
    float *colx, *rowy;
    const Tiling T =
        cta_prologue(Fs, edges, tables, P.use_tables && !P.image_tables, P.pose, g, b, P.cam, colx, rowy);
    const Frame& F = Fs; /* read-only from here on; the march hoists what it needs */
    float* __restrict__ out = P.depth + (size_t)b * H * W;
    const float* __restrict__ grid = P.sdf + (size_t)b * P.sdf_stride;
    const float* __restrict__ obs_img = MODE >= 1 ? P.depth_obs + (size_t)b * P.obs_stride : nullptr;
    /* keep the per-hypothesis bases in registers: ptxas otherwise re-derives b*stride inside the
     * march loop to save two registers (profiles/r01a: 8 of 68 loop instructions) */
    asm volatile("" : "+l"(out));
    asm volatile("" : "+l"(grid));

    /* pass 1: tiles that cannot see the box are zero (cu:294-296 writes 0 for these rays); one
     * whole 32x8 tile per warp, two 16-byte stores per lane */
    {
      const int n_tiles = T.tiles_x * T.tiles_y;
      const bool vec = ((W & 3) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
      for (int t = g + warp * G; t < n_tiles; t += kWarps * G) {
        const int ty = t / T.tiles_x, tx = t - ty * T.tiles_x;
        if (tx >= T.rtx0 && tx < T.rtx0 + T.rtw && ty >= T.rty0 && ty < T.rty0 + T.rth) continue;
        const int x0 = tx * kTileW, y0 = ty * kTileH;
        if (vec && x0 + kTileW <= W && y0 + kTileH <= H) {
          float4* p = reinterpret_cast<float4*>(out + (size_t)(y0 + lane_y) * W + x0) + lane_x;
          const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
          p[0] = z4;
          p[W] = z4; /* 4 rows further down: 4*W floats = W float4 */
        } else {
          for (int i = lane; i < kThreads; i += 32) {
            const int px = x0 + (i & (kTileW - 1)), py = y0 + (i / kTileW);
            if (px < W && py < H) out[(size_t)py * W + px] = 0.0f;
          }
        }
      }
    }

    /* pass 2: tiles inside the box's rectangle.  The CTA owns rectangle tiles g, g+G, ...  Their
     * 8x4-pixel warp tiles are first tested against the box silhouette by single threads (8 half-plane
     * tests each): the ones that cannot see the box are zero-filled on the spot, the others are
     * compacted into a shared-memory work list which the warps then drain dynamically (a warp whose
     * rays finish early takes the next entry).  Testing inside the drain loop instead cost ~90 warp
     * instructions per culled warp tile and ~50 per live one -- 21 % of all executed instructions at
     * BASELINE config 2 (profiles/r01g_ncu_fused_segments.txt). */
    if (MODE == 2 && WANT_POSE) moments_clear(acc_s); /* own column only: no barrier needed */
    float err_acc = 0.0f, cnt_acc = 0.0f, inl_acc = 0.0f;
    unsigned st_steps = 0, st_entered = 0, st_hit = 0, st_capped = 0;
    const int n_rect = T.rtw * T.rth;
    const int n_cand = n_rect > item_g(ws) ? ((n_rect - item_g(ws) + G - 1) / G) * kWarps : 0;
    /* compile-time grid constants (immediates) for the common resolutions */
    const Grid Gc = RT > 0 ? make_grid(RT, LT) : P.grid;
    const bool vec_ok = ((W & 3) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    for (int c0 = 0; c0 < n_cand; c0 += kListCap) {
      const int n_here = n_cand - c0 < kListCap ? n_cand - c0 : kListCap;
      __syncthreads(); /* previous chunk drained; list / counters reusable */
      if (threadIdx.x == 0) {
        n_live = 0;
        next_q = kWarps;
      }
      __syncthreads();
      /* 8 lanes per candidate: lane e tests hull edge e, then stores one float4 of the zero fill */
      const unsigned grp_mask = 0xffu << (lane & 24);
      const HullEdge my_edge = edges[lane & 7];
      const float inv_rtw = 1.0f / (float)(T.rtw > 0 ? T.rtw : 1);
      for (int i0 = 0; i0 < n_here; i0 += kThreads / 8) {
        const int i = i0 + (threadIdx.x >> 3);
        const bool have = i < n_here;
        const int cand = c0 + (have ? i : 0);
        const int r = item_g(ws) + (cand >> 3) * G, sub = cand & 7;
        const int wty = div_by(r, T.rtw, inv_rtw);
        const int tx = T.rtx0 + (r - wty * T.rtw), ty = T.rty0 + wty;
        const int wx0 = tx * kTileW + ((sub & 3) << 3), wy0 = ty * kTileH + ((sub >> 2) << 2);
        const bool out_rect = wx0 >= F.x1 || wx0 + 8 <= F.x0 || wy0 >= F.y1 || wy0 + 4 <= F.y0;
        const bool edge_out = hull_block_outside(my_edge, (float)wx0, (float)wy0, 8.0f, 4.0f);
        const bool culled = (__ballot_sync(kFull, edge_out || out_rect) & grp_mask) != 0;
        if (!have) continue;
        if (!culled) {
          if ((lane & 7) == 0)
            worklist[atomicAdd(&n_live, 1)] = (unsigned)(wx0 >> 3) | ((unsigned)(wy0 >> 2) << 16);
        } else if (wx0 < W && wy0 < H) { /* cu:294-296 writes 0 for these rays */
          const int yy = (lane & 7) >> 1, xh = (lane & 1) << 2;
          if (vec_ok && wx0 + 8 <= W && wy0 + 4 <= H) {
            *reinterpret_cast<float4*>(out + (size_t)(wy0 + yy) * W + wx0 + xh) =
                make_float4(0.f, 0.f, 0.f, 0.f);
          } else if (wy0 + yy < H) {
            for (int xx = xh; xx < xh + 4 && wx0 + xx < W; ++xx) out[(size_t)(wy0 + yy) * W + wx0 + xx] = 0.0f;
          }
        }
      }
      __syncthreads();
      const int n_q = n_live;
      for (int q = warp; q < n_q;) {
        const unsigned packed = worklist[q];
        const int px = (int)((packed & 0xffffu) << 3) + lane_x, py = (int)((packed >> 16) << 2) + lane_y;
        const bool inimg = px < W && py < H;
        float z = 0.0f;
        Ray ray;
        if (inimg && px >= F.x0 && px < F.x1 && py >= F.y0 && py < F.y1) {
          const float ux = P.use_tables ? colx[px] : pixel_dx(px, P.cam.cx, P.cam.fx);
          const float uy = P.use_tables ? rowy[py] : pixel_dy(py, P.cam.cy, P.cam.fy);
          ray = make_ray(F, ux, uy);
          float t_min, t_max;
          if (ray_cull_and_box(F, ray, t_min, t_max)) {
            int steps;
            bool capped;
            z = march<RT, LT>(grid, Gc, F, ray, t_min, t_max, P.threshold, steps, capped);
            if (STATS) {
              st_steps += steps;
              st_entered += 1;
              st_hit += z != 0.0f;
              st_capped += capped;
            }
          }
        }
        float sgn = 0.0f; /* MODE 2: sign(est - obs) on overlap pixels, 0 = nothing to back-propagate */
        if (inimg) {
          const unsigned pix = (unsigned)py * (unsigned)W + (unsigned)px;
          out[pix] = z;
          if (MODE >= 1 && z > 0.0f) {
            /* masked L1 against the observation (estimation/simple_setup.py:125-131) */
            const float obs = __ldg(obs_img + pix);
            if (obs > 0.0f) {
              err_acc += fabsf(z - obs);
              cnt_acc += 1.0f;
              /* result selection (estimation/simple_setup.py:183-185): relative error below the
               * threshold; IEEE division, the same expression the reference evaluates in torch */
              if (P.n_inlier) inl_acc += __fdiv_rn(fabsf(obs - z), obs) < P.inlier_threshold ? 1.0f : 0.0f;
              if (MODE == 2 && z != obs) sgn = z > obs ? 1.0f : -1.0f;
            }
          }
        }
        if (MODE == 2 && __any_sync(kFull, sgn != 0.0f)) {
          int base = 0;
          float w8[8];
          if (sgn != 0.0f) {
            float m[kMoments];
  #pragma unroll
            for (int i = 0; i < kMoments; ++i) m[i] = 0.0f;
            pixel_backward_moments<RT, WANT_SDF, WANT_POSE, LT>(grid, Gc, F, ray, z, sgn,
                                                                (P.flags & SDFR_SDF_GRAD_EXACT) != 0, base, w8, m);
            if (WANT_POSE) moments_add(acc_s, m);
          }
          if (WANT_SDF)
            scatter_sdf_warp<RT>(P.grad_sdf + (size_t)item_b(ws) * P.grad_sdf_stride, Gc, base, w8, sgn != 0.0f, lane);
        }
        if (lane == 0) q = atomicAdd(&next_q, 1);
        q = __shfl_sync(kFull, q, 0);
      }
    }
    /* the first warp out of the work list asks for the next logical CTA: late enough that a CTA still
     * busy with its item does not reserve one that another CTA could start sooner, early enough that
     * the answer arrives while the other warps finish */
    if (P.steal && lane == 0 && atomicExch(&ws.requested, 1) == 0) steal_request(ws);

    if (STATS) {
      const unsigned s = __reduce_add_sync(kFull, st_steps), e = __reduce_add_sync(kFull, st_entered);
      const unsigned h = __reduce_add_sync(kFull, st_hit), c = __reduce_add_sync(kFull, st_capped);
      if (lane == 0) {
        if (s) atomicAdd(P.stats + 0, (unsigned long long)s);
        if (e) atomicAdd(P.stats + 1, (unsigned long long)e);
        if (h) atomicAdd(P.stats + 2, (unsigned long long)h);
        if (c) atomicAdd(P.stats + 3, (unsigned long long)c);
      }
    }
    if (MODE >= 1) {
      err_acc = warp_sum(err_acc);
      cnt_acc = warp_sum(cnt_acc);
      if (lane == 0) {
        if (err_acc != 0.0f) atomicAdd(P.loss_sum + item_b(ws), err_acc);
        if (cnt_acc != 0.0f) atomicAdd(P.n_overlap + item_b(ws), cnt_acc);
      }
      if (P.n_inlier) {
        inl_acc = warp_sum(inl_acc);
        if (lane == 0 && inl_acc != 0.0f) atomicAdd(P.n_inlier + item_b(ws), inl_acc);
      }
    }
    if (MODE == 2 && WANT_POSE)
      reduce_pose(acc_s, F, Gc, item_b(ws), P.grad_position, P.grad_orientation, P.grad_inv_scale, P.flags);
    if (threadIdx.x == 0) steal_next(ws);
    __syncthreads(); /* next item published; Fs, acc_s, ws.g / ws.b and the work list are free again */
    if (ws.next_g < 0) break;
  }
}

/* ------------------------------------------------------------------------------------------
 * Backward (replaces sdf_renderer_cuda_backward_kernel, cu:300-468).
 * MODE 0: explicit grad_depth.  MODE 1: compare (gradient of the masked L1 rebuilt here).
 * Only tiles inside the projected box are visited: `depth` must be the image the forward
 * produced for the same pose (it is zero everywhere else).
 * ---------------------------------------------------------------------------------------- */
/* Register budget of the backward kernels: the SDF+pose variant needs ~80 registers; squeezed
 * into 64 (4 CTAs/SM) it spills, and the spill traffic (7 M write sectors per launch at C2,
 * profiles/r01d_bwd_ncu.txt) made it 4x slower than either single-purpose variant. */
constexpr int kBwdBlocks = 4;
template <int RT, int LT, int MODE, bool WANT_SDF, bool WANT_POSE>
__global__ void __launch_bounds__(kThreads, kBwdBlocks)
sdfr_backward_kernel(const __grid_constant__ BwdParams P) {
  extern __shared__ float tables[];
  __shared__ Frame Fs;
  __shared__ float acc_mem[WANT_POSE ? kMoments * kThreads : 1];
  MomentAcc& acc_s = *reinterpret_cast<MomentAcc*>(acc_mem);

  const int b = blockIdx.y + P.z_offset;
  const int g = blockIdx.x, G = gridDim.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lx = ((warp & 3) << 3) + (lane & 7);
  const int ly = ((warp >> 2) << 2) + (lane >> 3);
  const int W = P.cam.W, H = P.cam.H;

  float coef = 1.0f;
  if (MODE == 1) { /* d loss_b / d pixel = upstream_b * sign / n_overlap_b */
    const float n = __ldg(P.n_overlap + b);
    const float u = P.upstream ? __ldg(P.upstream + b) : 1.0f;
    coef = n > 0.0f ? u / n : 0.0f;
    if (coef == 0.0f) return; /* uniform over the CTA */
  }

  float *colx, *rowy;
  const Tiling T = cta_prologue(Fs, nullptr, tables, P.use_tables, P.pose, g, b, P.cam, colx, rowy);
  const Frame& F = Fs;
  const float* __restrict__ depth = P.depth + (size_t)b * H * W;
  const float* __restrict__ upimg =
      MODE == 0 ? P.grad_depth + (size_t)b * H * W : P.depth_obs + (size_t)b * P.obs_stride;
  const float* __restrict__ grid = P.sdf + (size_t)b * P.sdf_stride;
  float* __restrict__ gsdf = WANT_SDF ? P.grad_sdf + (size_t)b * P.grad_sdf_stride : nullptr;
  const bool exact = (P.flags & SDFR_SDF_GRAD_EXACT) != 0;
  const Grid Gc = RT > 0 ? make_grid(RT, LT) : P.grid;

  if (WANT_POSE) moments_clear(acc_s);

  /* the scan is latency bound (two dependent-free loads per pixel, ~7 % of the warp tiles hold
   * work): the loads of the NEXT tile are issued before the current one is processed */
  const int n_rect = T.rtw * T.rth;
  TileWalk w(g, G, T.rtw);
  int px = 0, py = 0;
  float z = 0.0f, u = 0.0f;
  bool valid = false;
  auto fetch = [&](int r) {
    valid = false;
    z = 0.0f;
    if (r < n_rect) {
      px = (T.rtx0 + w.tx) * kTileW + lx;
      py = (T.rty0 + w.ty) * kTileH + ly;
      if (px < W && py < H) {
        valid = true;
        z = __ldg(depth + (size_t)py * W + px);
        u = __ldg(upimg + (size_t)py * W + px);
      }
    }
  };
  fetch(g);
  for (int r = g; r < n_rect; r += G) {
    const float zc = z, uc = u;
    const int cpx = px, cpy = py;
    const bool cvalid = valid;
    w.next();
    fetch(r + G);
    float gup = 0.0f;
    if (cvalid && zc != 0.0f) {
      if (MODE == 0) {
        gup = uc;
      } else {
        gup = (zc > 0.0f && uc > 0.0f) ? ((zc > uc) ? coef : ((zc < uc) ? -coef : 0.0f)) : 0.0f;
      }
    }
    const bool has = gup != 0.0f;
    if (!__any_sync(kFull, has)) continue; /* the loop is uniform over the CTA: all 32 lanes are here */
    int base = 0;
    float w8[8];
    if (has) {
      const float ux = P.use_tables ? colx[cpx] : pixel_dx(cpx, P.cam.cx, P.cam.fx);
      const float uy = P.use_tables ? rowy[cpy] : pixel_dy(cpy, P.cam.cy, P.cam.fy);
      const Ray ray = make_ray(F, ux, uy);
      float m[kMoments];
#pragma unroll
      for (int i = 0; i < kMoments; ++i) m[i] = 0.0f;
      pixel_backward_moments<RT, WANT_SDF, WANT_POSE, LT>(grid, Gc, F, ray, zc, gup, exact, base, w8, m);
      if (WANT_POSE) moments_add(acc_s, m);
    }
    /* neighbouring rays of the warp's 8x4 pixels mostly end in the same cell: merge, then RED */
    if (WANT_SDF) scatter_sdf_warp<RT>(gsdf, Gc, base, w8, has, lane);
  }

  if (WANT_POSE)
    reduce_pose(acc_s, F, Gc, b, P.grad_position, P.grad_orientation, P.grad_inv_scale, P.flags);
}

/* grad *= upstream[b] / n_overlap[b]: the normalisation the fused compare kernel defers.  With `bounds`
 * (the empty-space bounds the render used) only the voxels of the cells inside them are visited: a ray can
 * only end -- and so only scatter a gradient -- in a cell whose smallest corner is below the hit-threshold
 * bound, every other voxel of the gradient grid is still the zero it was cleared to (C2: the box holds ~21 %
 * of the grid, 29 -> 7 us for 64 x 64^3). */
__global__ void __launch_bounds__(256)
sdfr_scale_grads_kernel(const float* __restrict__ n_overlap, const float* __restrict__ upstream,
                        long long grid_elems, float* __restrict__ grad_sdf, long long gs_stride,
                        float* __restrict__ gp, float* __restrict__ gq, float* __restrict__ gi,
                        unsigned flags, const CellBounds* __restrict__ bounds, int bounds_stride, int R) {
  const int b = blockIdx.y;
  const float n = __ldg(n_overlap + b);
  const float u = upstream ? __ldg(upstream + b) : 1.0f;
  const float coef = n > 0.0f ? u / n : 0.0f;
  if (blockIdx.x == 0 && threadIdx.x < 8) {
    const int i = threadIdx.x;
    if (i < 3) {
      if (flags & SDFR_GRAD_POSITION) gp[3 * b + i] *= coef;
    } else if (i < 7) {
      if (flags & SDFR_GRAD_ORIENTATION) gq[4 * b + (i - 3)] *= coef;
    } else {
      if (flags & SDFR_GRAD_INV_SCALE) gi[b] *= coef;
    }
  }
  if (flags & SDFR_GRAD_SDF)
    scale_sdf_grads(grad_sdf + (size_t)b * gs_stride, bounds ? bounds + (size_t)b * bounds_stride : nullptr, R,
                    grid_elems, coef, (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5),
                    (int)((gridDim.x * blockDim.x) >> 5), threadIdx.x & 31);
}

/* zero up to three small buffers in one launch (pose-gradient outputs) */
__global__ void sdfr_zero_small_kernel(float* a, int na, float* b, int nb, float* c, int nc) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < na + nb + nc; i += gridDim.x * blockDim.x) {
    if (i < na) a[i] = 0.0f;
    else if (i < na + nb) b[i - na] = 0.0f;
    else c[i - na - nb] = 0.0f;
  }
}

/* the per-hypothesis sums of the compare kernels (loss_sum, n_overlap, optional n_inlier: n each) and the three
 * pose-gradient outputs in ONE launch instead of three memset nodes plus a launch */
__global__ void sdfr_zero_sums_and_small_kernel(float* s0, float* s1, float* s2, int n, float* a, int na, float* b,
                                                int nb, float* c, int nc) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * n + na + nb + nc; i += gridDim.x * blockDim.x) {
    if (i < n) s0[i] = 0.0f;
    else if (i < 2 * n) s1[i - n] = 0.0f;
    else if (i < 3 * n) { if (s2) s2[i - 2 * n] = 0.0f; }
    else if (i < 3 * n + na) a[i - 3 * n] = 0.0f;
    else if (i < 3 * n + na + nb) b[i - 3 * n - na] = 0.0f;
    else c[i - 3 * n - na - nb] = 0.0f;
  }
}

/* ------------------------------------------------------------------------------------------
 * Multi-object composite: one depth map, per-pixel minimum positive depth over K objects.
 * Frames of up to kMaxObjPerPass objects live in shared memory; a pixel only traces the
 * objects whose projected rectangle contains it.
 * ---------------------------------------------------------------------------------------- */
constexpr int kMaxObjPerPass = 32;

template <int RT, int LT>
__global__ void __launch_bounds__(kThreads)
sdfr_forward_composite_kernel(const __grid_constant__ FwdParams P, int n_objects,
                              int* __restrict__ winner_out) {
  __shared__ Frame Fs[kMaxObjPerPass];
  __shared__ float colx[kTileW];
  __shared__ float rowy[kTileH];

  const int bx0 = blockIdx.x * kTileW, by0 = blockIdx.y * kTileH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lx = ((warp & 3) << 3) + (lane & 7);
  const int ly = ((warp >> 2) << 2) + (lane >> 3);
  const int px = bx0 + lx, py = by0 + ly;
  const bool inside = px < P.cam.W && py < P.cam.H;
  const Grid Gc = RT > 0 ? make_grid(RT, LT) : P.grid;

  if (warp == 1) colx[lane] = pixel_dx(bx0 + lane, P.cam.cx, P.cam.fx);
  if (warp == 2 && lane < kTileH) rowy[lane] = pixel_dy(by0 + lane, P.cam.cy, P.cam.fy);

  float best = 0.0f;
  int win = -1;
  for (int k0 = 0; k0 < n_objects; k0 += kMaxObjPerPass) {
    const int nk = min(kMaxObjPerPass, n_objects - k0);
    __syncthreads(); /* previous pass done with Fs; also publishes the tables */
    for (int k = warp; k < nk; k += kWarps) build_frame(Fs[k], nullptr, P.pose, k0 + k, P.cam, lane);
    __syncthreads();
    if (!inside) continue;
    for (int k = 0; k < nk; ++k) {
      const Frame& F = Fs[k];
      if (px < F.x0 || px >= F.x1 || py < F.y0 || py >= F.y1) continue;
      const Ray r = make_ray(F, colx[lx], rowy[ly]);
      float t_min, t_max;
      if (!ray_cull_and_box(F, r, t_min, t_max)) continue;
      int steps;
      bool capped;
      const float z = march<RT, LT>(P.sdf + (size_t)(k0 + k) * P.sdf_stride, Gc, F, r, t_min,
                                    t_max, P.threshold, steps, capped);
      if (z > 0.0f && (win < 0 || z < best)) {
        best = z;
        win = k0 + k;
      }
    }
  }
  if (inside) {
    const size_t pix = (size_t)py * P.cam.W + px;
    P.depth[pix] = best;
    winner_out[pix] = win;
  }
}

template <int RT, int LT, bool WANT_SDF, bool WANT_POSE>
__global__ void __launch_bounds__(kThreads)
sdfr_backward_composite_kernel(const __grid_constant__ BwdParams P) {
  __shared__ float colx[kTileW];
  __shared__ float rowy[kTileH];

  const int bx0 = blockIdx.x * kTileW, by0 = blockIdx.y * kTileH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lx = ((warp & 3) << 3) + (lane & 7);
  const int ly = ((warp >> 2) << 2) + (lane >> 3);
  const int px = bx0 + lx, py = by0 + ly;
  const bool inside = px < P.cam.W && py < P.cam.H;
  const size_t pix = (size_t)py * P.cam.W + px;
  const Grid Gc = RT > 0 ? make_grid(RT, LT) : P.grid;

  float z = 0.0f, gup = 0.0f;
  int win = -1;
  if (inside) {
    z = __ldg(P.depth + pix);
    if (z != 0.0f) {
      win = __ldg(P.winner + pix);
      gup = __ldg(P.grad_depth + pix);
    }
  }
  const bool active = z != 0.0f && gup != 0.0f && win >= 0 && win < P.n_objects;
  if (!__syncthreads_or(active)) return;
  if (warp == 1) colx[lane] = pixel_dx(bx0 + lane, P.cam.cx, P.cam.fx);
  if (warp == 2 && lane < kTileH) rowy[lane] = pixel_dy(by0 + lane, P.cam.cy, P.cam.fy);
  __syncthreads();

  /* a warp's 8x4 pixels almost always belong to one object: loop over the distinct winners */
  unsigned todo = __ballot_sync(kFull, active);
  while (todo) {
    const int leader = __ffs(todo) - 1;
    const int k = __shfl_sync(kFull, win, leader);
    const bool mine = active && win == k;
    todo &= ~__ballot_sync(kFull, mine);

    Frame F; /* every lane builds the pose part in registers; no rectangle needed */
    frame_pose(F, P.pose.position + 3 * k, P.pose.orientation + 4 * k, P.pose.inv_scale + k);
    float acc[kMoments];
#pragma unroll
    for (int i = 0; i < kMoments; ++i) acc[i] = 0.0f;
    int base = 0;
    float w8[8];
    if (mine) {
      const Ray r = make_ray(F, colx[lx], rowy[ly]);
      pixel_backward_moments<RT, WANT_SDF, WANT_POSE, LT>(P.sdf + (size_t)k * P.sdf_stride, Gc, F, r, z, gup,
                                                          (P.flags & SDFR_SDF_GRAD_EXACT) != 0, base, w8, acc);
    }
    if (WANT_SDF) scatter_sdf_warp<RT>(P.grad_sdf + (size_t)k * P.grad_sdf_stride, Gc, base, w8, mine, lane);
    if (WANT_POSE) {
#pragma unroll
      for (int i = 0; i < kMoments; ++i) acc[i] = warp_sum(acc[i]);
      float out[8];
      moments_to_pose(F, Gc, acc, out);
      float v = out[0];
#pragma unroll
      for (int i = 1; i < 8; ++i) v = (lane == i) ? out[i] : v;
      if (lane < 8 && v != 0.0f) {
        if (lane < 3) {
          if (P.flags & SDFR_GRAD_POSITION) atomicAdd(P.grad_position + 3 * k + lane, v);
        } else if (lane < 7) {
          if (P.flags & SDFR_GRAD_ORIENTATION) atomicAdd(P.grad_orientation + 4 * k + (lane - 3), v);
        } else {
          if (P.flags & SDFR_GRAD_INV_SCALE) atomicAdd(P.grad_inv_scale + k, v);
        }
      }
    }
  }
}

/*
 * Cell bounds of the grids (CellBounds, sdfr_core.cuh): per grid, the first / last cell index per axis
 * whose smallest corner value lies below the hit-threshold bound tau of the hypotheses that render it.
 * Rays that miss that box (plus a one-cell margin) cannot terminate anywhere, so the render kernels
 * zero them without marching; rays that enter it are marched exactly as the reference marches them.
 * For the reference workloads the object fills about a third of the [-1,1]^3 box's silhouette: two
 * thirds of the rays the reference marches are proven empty by 6 integers per grid.
 *   init kernel: tau per grid (max over the hypotheses sharing it), bounds := empty
 *   scan kernel: CTA per (x cell layer, grid); a warp owns a (x, y) row of cells, lane = z (coalesced
 *   reads of the 4 rows the cells touch), the cell minimum via one shuffle, ballots give the z range.
 */
__global__ void sdfr_bounds_init_kernel(const float* __restrict__ pos, const float* __restrict__ inv_scale,
                                        int batch, int n_grids, float threshold, CellBounds* __restrict__ out) {
  const int n = blockIdx.x;
  float tau = 0.0f;
  if (n_grids == 1) { /* one grid shared by the whole batch */
    for (int b = threadIdx.x; b < batch; b += blockDim.x) tau = fmaxf(tau, hit_tau(pos + 3 * b, inv_scale[b], threshold));
  } else if (threadIdx.x == 0) {
    tau = hit_tau(pos + 3 * n, inv_scale[n], threshold);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) tau = fmaxf(tau, __shfl_xor_sync(kFull, tau, o));
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = tau;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) tau = fmaxf(tau, red[w]);
    CellBounds cb;
    cb.lo[0] = cb.lo[1] = cb.lo[2] = 0x7fffffff;
    cb.hi[0] = cb.hi[1] = cb.hi[2] = -1;
    cb.tau = tau;
    cb.pad = 0;
    out[n] = cb;
  }
}

/* The scan.  A cell's smallest corner is below tau exactly when one of its 8 corner VOXELS is, and a
 * voxel x belongs to the cells x-1 and x of its axis (clamped to [0, R-2]), independently per axis; so
 * the box of the cells below tau is the bounding box of the voxels below tau with its low side moved
 * down by one:   lo = max(min_voxel - 1, 0),   hi = min(max_voxel, R - 2).
 * That makes the pass a streaming read -- every voxel loaded once, coalesced, one compare -- instead of
 * a stencil over cell corners (history: a shared-memory plane with 4 neighbour reads per cell was
 * issue-bound at 43 us for 64 x 64^3; a register walk over row strips with shuffles for the z pairs,
 * 34 M warp instructions, 42 us at 67 % ALU-pipe utilisation, ncu r02e).
 * CTA = (voxel layer ix, grid n): warp w walks rows y = w, w + 8, ..., lane = z.
 * WRITE_SKEW: the source is the DENSE grid and the kernel also writes the skewed copy, so that the
 * layout pass and the bounds pass are one read of the grids. */
__device__ __forceinline__ void bounds_commit(CellBounds* __restrict__ o, int axis, int vlo, int vhi, int R) {
  atomicMin(&o->lo[axis], vlo > 0 ? vlo - 1 : 0);
  atomicMax(&o->hi[axis], vhi < R - 2 ? vhi : R - 2);
}

constexpr int kScanUnroll = 4;

template <bool WRITE_SKEW>
__global__ void __launch_bounds__(256)
sdfr_bounds_scan_kernel(const float* __restrict__ sdf, long long sdf_stride, int R, int py, int px,
                        CellBounds* __restrict__ out, float* __restrict__ skew, long long skew_stride,
                        int spy, int spx) {
  __shared__ int s_lo[2], s_hi[2];
  const int n = blockIdx.y, ix = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* __restrict__ g0 = sdf + (size_t)n * sdf_stride + (size_t)ix * px;
  float* __restrict__ d0 = WRITE_SKEW ? skew + (size_t)n * skew_stride + (size_t)ix * spx : nullptr;
  const float tau = out[n].tau;
  if (threadIdx.x < 2) {
    s_lo[threadIdx.x] = 0x7fffffff;
    s_hi[threadIdx.x] = -1;
  }
  __syncthreads();
  int ylo = 0x7fffffff, yhi = -1, zlo = 0x7fffffff, zhi = -1;
  /* dense rows of a multiple of 4 voxels: 16-byte loads, lane = 4 consecutive z */
  const bool vec = (R & 3) == 0 && py == R && (px & 3) == 0 && (sdf_stride & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(sdf) & 15) == 0;
  if (vec) {
    const int q4 = R >> 2; /* float4 per row */
    const int rows_per_pass = 256 / q4; /* R <= 1024: q4 <= 256 */
    const int sub = threadIdx.x / q4, zq = threadIdx.x - sub * q4;
    if (sub < rows_per_pass) {
      /* kScanUnroll independent 16-byte loads in flight per thread (the pass is latency-bound otherwise:
       * one dependent round trip per row) */
      for (int y0 = sub; y0 < R; y0 += rows_per_pass * kScanUnroll) {
        float4 v[kScanUnroll];
#pragma unroll
        for (int j = 0; j < kScanUnroll; ++j) {
          const int y = y0 + j * rows_per_pass;
          v[j] = y < R ? __ldg(reinterpret_cast<const float4*>(g0 + (size_t)y * py) + zq)
                       : make_float4(3.0e38f, 3.0e38f, 3.0e38f, 3.0e38f);
        }
#pragma unroll
        for (int j = 0; j < kScanUnroll; ++j) {
          const int y = y0 + j * rows_per_pass;
          if (y >= R) break;
          if (WRITE_SKEW) {
            float* __restrict__ w0 = d0 + (size_t)y * spy + 4 * zq;
            w0[0] = v[j].x; w0[1] = v[j].y; w0[2] = v[j].z; w0[3] = v[j].w;
          }
          const unsigned m = (v[j].x < tau ? 1u : 0u) | (v[j].y < tau ? 2u : 0u) | (v[j].z < tau ? 4u : 0u) |
                             (v[j].w < tau ? 8u : 0u);
          if (m) {
            ylo = min(ylo, y); yhi = max(yhi, y);
            zlo = min(zlo, 4 * zq + __ffs(m) - 1);
            zhi = max(zhi, 4 * zq + 31 - __clz(m));
          }
        }
      }
    }
  } else {
    for (int y0 = warp; y0 < R; y0 += kWarps * kScanUnroll) {
      for (int z = lane; z < R; z += 32) {
        float v[kScanUnroll];
#pragma unroll
        for (int j = 0; j < kScanUnroll; ++j) {
          const int y = y0 + j * kWarps;
          v[j] = y < R ? __ldg(g0 + (size_t)y * py + z) : 3.0e38f;
        }
#pragma unroll
        for (int j = 0; j < kScanUnroll; ++j) {
          const int y = y0 + j * kWarps;
          if (y >= R) break;
          if (WRITE_SKEW) d0[(size_t)y * spy + z] = v[j];
          if (v[j] < tau) {
            ylo = min(ylo, y); yhi = max(yhi, y);
            zlo = min(zlo, z); zhi = max(zhi, z);
          }
        }
      }
    }
  }
  ylo = __reduce_min_sync(kFull, ylo); yhi = __reduce_max_sync(kFull, yhi);
  zlo = __reduce_min_sync(kFull, zlo); zhi = __reduce_max_sync(kFull, zhi);
  if (lane == 0 && yhi >= 0) {
    atomicMin(&s_lo[0], ylo); atomicMax(&s_hi[0], yhi);
    atomicMin(&s_lo[1], zlo); atomicMax(&s_hi[1], zhi);
  }
  __syncthreads();
  if (threadIdx.x == 0 && s_hi[0] >= 0) {
    bounds_commit(out + n, 0, ix, ix, R);
    bounds_commit(out + n, 1, s_lo[0], s_hi[0], R);
    bounds_commit(out + n, 2, s_lo[1], s_hi[1], R);
  }
}

/* Slab minima of a grid: minima[n][a][i] = the smallest voxel value with coordinate i on axis a (x, y,
 * z).  They do not depend on the pose: for FIXED grids they are computed once, and the cell bounds of any
 * hit-threshold bound tau follow from 3 R comparisons per grid (sdfr_bounds_from_minima_kernel) -- the
 * bounding box of the voxels below tau is, per axis, the first / last slab whose minimum is below tau.
 * Same walk as the scan; minima must be pre-filled with +large (sdfr_fill_kernel). */
__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
  /* order-preserving for IEEE floats: non-negative values compare as ints, negative ones reversed as
   * unsigned; mixed sequences stay correct because a negative float is a negative int / a huge unsigned */
  if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}

__global__ void sdfr_fill_kernel(float* __restrict__ p, long long n, float v) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    p[i] = v;
}

constexpr int kSlabMaxR = 1024;

__global__ void __launch_bounds__(256)
sdfr_slab_minima_kernel(const float* __restrict__ sdf, long long sdf_stride, int R, int py, int px,
                        float* __restrict__ minima) {
  __shared__ float s_z[kSlabMaxR];
  __shared__ float s_x[kWarps];
  const int n = blockIdx.y, ix = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* __restrict__ g0 = sdf + (size_t)n * sdf_stride + (size_t)ix * px;
  float* __restrict__ mx = minima + (size_t)n * 3 * R;
  float* __restrict__ my = mx + R;
  float* __restrict__ mz = my + R;
  for (int z = threadIdx.x; z < R; z += 256) s_z[z] = 3.0e38f;
  __syncthreads();
  float xmin = 3.0e38f;
  for (int z0 = 0; z0 < R; z0 += 32) {
    const int z = z0 + lane;
    float zmin = 3.0e38f;
    for (int y = warp; y < R; y += kWarps) {
      const float v = z < R ? __ldg(g0 + (size_t)y * py + z) : 3.0e38f;
      zmin = fminf(zmin, v);
      float r = v;
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) r = fminf(r, __shfl_xor_sync(kFull, r, o));
      if (lane == 0) atomic_min_float(my + y, r); /* R / 32 partial minima per row and layer */
    }
    if (z < R) atomic_min_float(&s_z[z], zmin);
    xmin = fminf(xmin, zmin);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) xmin = fminf(xmin, __shfl_xor_sync(kFull, xmin, o));
  if (lane == 0) s_x[warp] = xmin;
  __syncthreads();
  for (int z = threadIdx.x; z < R; z += 256) atomic_min_float(mz + z, s_z[z]);
  if (threadIdx.x == 0) {
    float m = s_x[0];
    for (int w = 1; w < kWarps; ++w) m = fminf(m, s_x[w]);
    mx[ix] = m; /* this CTA owns the layer */
  }
}

/* Cell bounds from slab minima: one CTA per grid; tau as in sdfr_bounds_init_kernel. */
__global__ void __launch_bounds__(256)
sdfr_bounds_from_minima_kernel(const float* __restrict__ minima, int R, const float* __restrict__ pos,
                               const float* __restrict__ inv_scale, int batch, int n_grids, float threshold,
                               CellBounds* __restrict__ out) {
  const int n = blockIdx.x;
  __shared__ float red[8];
  __shared__ int s_lo[3], s_hi[3];
  float tau = 0.0f;
  if (n_grids == 1) {
    for (int b = threadIdx.x; b < batch; b += blockDim.x) tau = fmaxf(tau, hit_tau(pos + 3 * b, inv_scale[b], threshold));
  } else if (threadIdx.x == 0) {
    tau = hit_tau(pos + 3 * n, inv_scale[n], threshold);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) tau = fmaxf(tau, __shfl_xor_sync(kFull, tau, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = tau;
  if (threadIdx.x < 3) {
    s_lo[threadIdx.x] = 0x7fffffff;
    s_hi[threadIdx.x] = -1;
  }
  __syncthreads();
  tau = red[0];
  for (int w = 1; w < 8; ++w) tau = fmaxf(tau, red[w]);
  const float* __restrict__ m = minima + (size_t)n * 3 * R;
  for (int i = threadIdx.x; i < 3 * R; i += blockDim.x) {
    if (m[i] < tau) {
      const int a = i / R, v = i - a * R;
      atomicMin(&s_lo[a], v > 0 ? v - 1 : 0);
      atomicMax(&s_hi[a], v < R - 2 ? v : R - 2);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    CellBounds cb;
    for (int a = 0; a < 3; ++a) {
      cb.lo[a] = s_lo[a];
      cb.hi[a] = s_hi[a];
    }
    cb.tau = tau;
    cb.pad = 0;
    out[n] = cb;
  }
}

/* Dense [R][R][R] -> skewed pitched copy (sdfr_core.cuh: kLayoutSkewed).  One warp per (x,y)
 * row: coalesced reads, coalesced (unaligned) writes; the padding is never read. */
__global__ void __launch_bounds__(256)
sdfr_skew_kernel(const float* __restrict__ src, long long src_stride, float* __restrict__ dst,
                 long long dst_stride, int R, int py, int px) {
  const int b = blockIdx.y;
  const float* __restrict__ s = src + (size_t)b * src_stride;
  float* __restrict__ d = dst + (size_t)b * dst_stride;
  if ((R & 3) == 0 && (reinterpret_cast<uintptr_t>(s) & 15) == 0) {
    /* one thread per 4 consecutive z: a 16-byte read, four 4-byte writes (rows of the skewed
     * array start at odd element offsets) */
    const int q4 = R >> 2, n4 = R * R * q4;
    const float4* __restrict__ s4 = reinterpret_cast<const float4*>(s);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
      const int row = i / q4, z = (i - row * q4) << 2;
      const int ix = row / R, iy = row - ix * R;
      const float4 v = __ldg(s4 + i);
      float* __restrict__ o = d + (size_t)ix * px + iy * py + z;
      o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
    }
    return;
  }
  const int n = R * R * R;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int row = i / R, z = i - row * R;
    const int ix = row / R, iy = row - ix * R;
    d[(size_t)ix * px + iy * py + z] = __ldg(s + i);
  }
}

/* ------------------------------------------------------------------------------------------
 * Host side
 * ---------------------------------------------------------------------------------------- */
int check_common(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                 const float* quat, const float* inv_scale, int batch, int W, int H) {
  if (layout != SDFR_LAYOUT_DENSE && layout != SDFR_LAYOUT_SKEWED) return fail(SDFR_E_FLAGS, "unknown sdf_layout");
  if (batch < 0 || W < 0 || H < 0) return fail(SDFR_E_SHAPE, "negative batch/width/height");
  if (R < 2 || R > 1024) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (sdf_stride < 0) return fail(SDFR_E_SHAPE, "negative sdf_stride");
  if (W > (1 << 19) || H > (1 << 18) || (long long)W * H >= (1ll << 30))
    return fail(SDFR_E_SHAPE, "image too large (width <= 2^19, height <= 2^18, width*height < 2^30)");
  if (batch == 0 || W == 0 || H == 0) return 0;
  if (!sdf || !pos || !quat || !inv_scale) return fail(SDFR_E_NULL, "NULL input pointer");
  return 0;
}

dim3 tile_grid(int W, int H, int z) {
  return dim3((W + kTileW - 1) / kTileW, (H + kTileH - 1) / kTileH, z);
}

int zero_async(void* p, size_t bytes, cudaStream_t s) {
  if (!p || bytes == 0) return 0;
  const cudaError_t e = cudaMemsetAsync(p, 0, bytes, s);
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "cudaMemsetAsync: %s", cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

/* CTAs per hypothesis: enough CTAs to fill the device several times over (tail effect), never
 * more than there are tiles.  148 SMs x 32 on a B200. */
int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

int ctas_per_hypothesis(int batch, int W, int H) {
  const long long n_tiles = (long long)((W + kTileW - 1) / kTileW) * ((H + kTileH - 1) / kTileH);
  /* 16 CTAs per SM in total for larger batches (measured at 64 hypotheses, profiles/r01zp_micro.json
   * c2_cta_sweep: 2368 CTAs beat 4736 by 2 % forward / fused and 6 % backward); small batches keep 32
   * so that a single large frame still gets one CTA per tile */
  const long long target = (long long)sm_count() * (batch >= 16 ? 16 : 32);
  long long g = (target + batch - 1) / batch;
  if (g > n_tiles) g = n_tiles;
  if (g > 65535) g = 65535;
  return g < 1 ? 1 : (int)g;
}

/* dynamic shared memory for the ray tables; 0 = image too wide, compute per thread instead */
size_t table_bytes(int W, int H) {
  const size_t n = (size_t)((W + kTileW - 1) / kTileW) * kTileW +
                   (size_t)((H + kTileH - 1) / kTileH) * kTileH;
  return n * sizeof(float) <= 40 * 1024 ? n * sizeof(float) : 0;
}

template <int RT, int LT, int MODE, bool STATS>
void launch_forward_rt(FwdParams& P, dim3 grid, size_t smem, cudaStream_t s) {
  /* constexpr: MODE 0 and 1 instantiate their own kernel only -- no launch of theirs can reach the
   * gradient variants below, and every instantiation is machine code the library ships */
  if constexpr (MODE != 2) {
    sdfr_forward_kernel<RT, LT, MODE, STATS, false, false><<<grid, kThreads, smem, s>>>(P);
  } else {
    const bool want_sdf = (P.flags & SDFR_GRAD_SDF) != 0;
    const bool want_pose =
        (P.flags & (SDFR_GRAD_POSITION | SDFR_GRAD_ORIENTATION | SDFR_GRAD_INV_SCALE)) != 0;
    if (want_sdf && want_pose)
      sdfr_forward_kernel<RT, LT, MODE, STATS, true, true><<<grid, kThreads, smem, s>>>(P);
    else if (want_sdf)
      sdfr_forward_kernel<RT, LT, MODE, STATS, true, false><<<grid, kThreads, smem, s>>>(P);
    else if (want_pose)
      sdfr_forward_kernel<RT, LT, MODE, STATS, false, true><<<grid, kThreads, smem, s>>>(P);
    else
      sdfr_forward_kernel<RT, LT, 1, STATS, false, false><<<grid, kThreads, smem, s>>>(P);
  }
}

/* common resolutions get compile-time pitches (immediate-offset gathers) in both layouts; every
 * other resolution runs the generic kernel with the run-time pitches of P.grid */
#define SDFR_DISPATCH_RT_LT(R, skewed, CALL)                                       \
  do {                                                                             \
    if ((R) == 64 && !(skewed)) { CALL(64, kLayoutDense); }                        \
    else if ((R) == 64) { CALL(64, kLayoutSkewed); }                               \
    else if ((R) == 128 && !(skewed)) { CALL(128, kLayoutDense); }                 \
    else if ((R) == 128) { CALL(128, kLayoutSkewed); }                             \
    else if ((R) == 32 && !(skewed)) { CALL(32, kLayoutDense); }                   \
    else if ((R) == 32) { CALL(32, kLayoutSkewed); }                               \
    else { CALL(0, kLayoutDense); }                                                \
  } while (0)

template <int MODE, bool STATS>
int launch_forward(FwdParams P, int batch, cudaStream_t s) {
  const size_t smem = table_bytes(P.cam.W, P.cam.H);
  P.use_tables = smem != 0;
  const int G = ctas_per_hypothesis(batch, P.cam.W, P.cam.H);
  const int n_tiles = ((P.cam.W + kTileW - 1) / kTileW) * ((P.cam.H + kTileH - 1) / kTileH);
  const bool skewed = P.grid.layout == kLayoutSkewed;
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid(G, batch - z0 < 65535 ? batch - z0 : 65535);
    /* a launch that fits in one wave has nothing to steal: its CTAs do not wait for a try_cancel
     * answer.  With one CTA per tile (a single frame) each item fills the 32 + 8 table entries of its
     * own tile, as without stealing: the whole image's table (1120 double divisions at 640x480)
     * would lengthen every first-wave CTA of a latency-bound launch. */
    P.steal = (long long)G * grid.y > (long long)sm_count() * kFwdBlocks;
    P.image_tables = P.use_tables && P.steal && G < n_tiles;
#define SDFR_CALL(RT, LT) launch_forward_rt<RT, LT, MODE, STATS>(P, grid, smem, s)
    SDFR_DISPATCH_RT_LT(P.grid.R, skewed, SDFR_CALL);
#undef SDFR_CALL
  }
  return check_launch("sdfr_forward_kernel");
}

template <int RT, int LT, int MODE>
void launch_backward_rt(BwdParams& P, dim3 grid, size_t smem, bool want_sdf, bool want_pose,
                        cudaStream_t s) {
  if (want_sdf && want_pose)
    sdfr_backward_kernel<RT, LT, MODE, true, true><<<grid, kThreads, smem, s>>>(P);
  else if (want_sdf)
    sdfr_backward_kernel<RT, LT, MODE, true, false><<<grid, kThreads, smem, s>>>(P);
  else
    sdfr_backward_kernel<RT, LT, MODE, false, true><<<grid, kThreads, smem, s>>>(P);
}

/*
 * The backward is launched once per slice of at most 65535 hypotheses (the gridDim.y limit).  With
 * ZERO_GRADS, the per-hypothesis gradient grids of a slice are cleared right before its launch, so
 * that the scattered RED.ADDs hit zeroed lines that are still L2-resident; a shared gradient grid
 * is cleared once before the first slice.  The clear stays next to the launch: when the zeroed
 * lines are evicted before the kernel runs, every RED becomes a 32-byte read-modify-write against
 * HBM (measured at B = 64, 64^3, 640x480: 457 us against 105 us for the pose gradients alone).
 */
template <int MODE>
int launch_backward(BwdParams P, int batch, bool zero_sdf, cudaStream_t s) {
  const bool want_sdf = (P.flags & SDFR_GRAD_SDF) != 0;
  const bool want_pose =
      (P.flags & (SDFR_GRAD_POSITION | SDFR_GRAD_ORIENTATION | SDFR_GRAD_INV_SCALE)) != 0;
  if (!want_sdf && !want_pose) return 0;
  const size_t smem = table_bytes(P.cam.W, P.cam.H);
  P.use_tables = smem != 0;
  const bool skewed = P.grid.layout == kLayoutSkewed;
  const size_t grid_bytes = sizeof(float) * (size_t)P.grid.R * P.grid.R * P.grid.R;
  if (zero_sdf && want_sdf && P.grad_sdf_stride == 0) { /* one shared gradient grid */
    if (int rc = zero_async(P.grad_sdf, grid_bytes, s)) return rc;
  }
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    const int nz = batch - z0 < 65535 ? batch - z0 : 65535;
    if (zero_sdf && want_sdf && P.grad_sdf_stride != 0) {
      if ((size_t)P.grad_sdf_stride * sizeof(float) == grid_bytes) {
        if (int rc = zero_async(P.grad_sdf + (size_t)z0 * P.grad_sdf_stride, grid_bytes * nz, s))
          return rc;
      } else {
        for (int b = z0; b < z0 + nz; ++b)
          if (int rc = zero_async(P.grad_sdf + (size_t)b * P.grad_sdf_stride, grid_bytes, s))
            return rc;
      }
    }
    P.z_offset = z0;
    const dim3 grid(ctas_per_hypothesis(nz, P.cam.W, P.cam.H), nz);
#define SDFR_CALL(RT, LT) launch_backward_rt<RT, LT, MODE>(P, grid, smem, want_sdf, want_pose, s)
    SDFR_DISPATCH_RT_LT(P.grid.R, skewed, SDFR_CALL);
#undef SDFR_CALL
  }
  return check_launch("sdfr_backward_kernel");
}

int check_backward_outputs(unsigned flags, const float* gs, long long gs_stride, const float* gp,
                           const float* gq, const float* gi) {
  if (flags & ~(SDFR_GRAD_ALL | SDFR_SDF_GRAD_EXACT | SDFR_ZERO_GRADS))
    return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (gs_stride < 0) return fail(SDFR_E_SHAPE, "negative grad_sdf_stride");
  if (((flags & SDFR_GRAD_SDF) && !gs) || ((flags & SDFR_GRAD_POSITION) && !gp) ||
      ((flags & SDFR_GRAD_ORIENTATION) && !gq) || ((flags & SDFR_GRAD_INV_SCALE) && !gi))
    return fail(SDFR_E_NULL, "NULL gradient buffer for a requested gradient");
  return 0;
}

int zero_grads(unsigned flags, int R, int batch, float* gs, long long gs_stride, float* gp,
               float* gq, float* gi, cudaStream_t s) {
  if (!(flags & SDFR_ZERO_GRADS)) return 0;
  int rc = 0;
  const size_t grid_elems = (size_t)R * R * R;
  if (flags & SDFR_GRAD_SDF) {
    if (gs_stride == 0 || (size_t)gs_stride == grid_elems) {
      const size_t n = gs_stride == 0 ? grid_elems : grid_elems * batch;
      rc = zero_async(gs, n * sizeof(float), s);
    } else {
      for (int b = 0; b < batch && rc == 0; ++b)
        rc = zero_async(gs + (size_t)b * gs_stride, grid_elems * sizeof(float), s);
    }
  }
  if (rc == 0 && (flags & (SDFR_GRAD_POSITION | SDFR_GRAD_ORIENTATION | SDFR_GRAD_INV_SCALE))) {
    /* the three small outputs in ONE launch instead of three memset nodes */
    const int na = (flags & SDFR_GRAD_POSITION) ? 3 * batch : 0;
    const int nb = (flags & SDFR_GRAD_ORIENTATION) ? 4 * batch : 0;
    const int nc = (flags & SDFR_GRAD_INV_SCALE) ? batch : 0;
    const int n = na + nb + nc;
    sdfr_zero_small_kernel<<<n > 4096 ? 16 : 1, 256, 0, s>>>(gp, na, gq, nb, gi, nc);
    rc = check_launch("sdfr_zero_small_kernel");
  }
  return rc;
}

Pose make_pose(const float* pos, const float* quat, const float* inv_scale, const sdfr_cell_bounds* bounds,
               long long sdf_stride, int R, float threshold) {
  Pose p;
  p.position = pos;
  p.orientation = quat;
  p.inv_scale = inv_scale;
  p.bounds = reinterpret_cast<const CellBounds*>(bounds);
  p.bounds_stride = sdf_stride != 0 ? 1 : 0; /* one entry per grid */
  p.R = R;
  p.threshold = threshold;
  return p;
}

FwdParams fwd_params(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                     const float* quat, const float* inv_scale, int W, int H, float cx, float cy,
                     float fx, float fy, float threshold, float* depth,
                     const sdfr_cell_bounds* bounds = nullptr) {
  FwdParams P;
  memset(&P, 0, sizeof(P));
  P.sdf = sdf;
  P.sdf_stride = sdf_stride;
  P.pose = make_pose(pos, quat, inv_scale, bounds, sdf_stride, R, threshold);
  P.grid = make_grid(R, layout);
  P.cam = Camera{W, H, cx, cy, fx, fy};
  P.threshold = threshold;
  P.depth = depth;
  return P;
}

BwdParams bwd_params(const float* depth, const float* sdf, int R, long long sdf_stride, int layout,
                     const float* pos, const float* quat, const float* inv_scale, int W, int H,
                     float cx, float cy, float fx, float fy, float* gs, long long gs_stride,
                     float* gp, float* gq, float* gi, unsigned flags,
                     const sdfr_cell_bounds* bounds = nullptr, float threshold = 0.0f) {
  BwdParams P;
  memset(&P, 0, sizeof(P));
  P.depth = depth;
  P.sdf = sdf;
  P.sdf_stride = sdf_stride;
  P.pose = make_pose(pos, quat, inv_scale, bounds, sdf_stride, R, threshold);
  P.grid = make_grid(R, layout);
  P.cam = Camera{W, H, cx, cy, fx, fy};
  P.grad_sdf = gs;
  P.grad_sdf_stride = gs_stride;
  P.grad_position = gp;
  P.grad_orientation = gq;
  P.grad_inv_scale = gi;
  P.flags = flags;
  return P;
}

#if SDFR_IN_PART(4)
#include "sdfr_points.cuh"
#include "sdfr_decoder.cuh"
#include "sdfr_step.cuh"
#endif

}  // namespace

extern "C" {

#if SDFR_IN_PART(1)
int sdfr_abi_version(void) { return SDFR_ABI_VERSION; }
const char* sdfr_last_error(void) { return g_err; }
const char* sdfr_build_info(void) {
  return "libsdfrender sm_100a; persistent CTAs per hypothesis, tile 32x8 (8 warps of 8x4 px); fp32; nvcc " __DATE__;
}
int sdfr_max_steps(void) { return sdfr::kMaxSteps; }

#endif
#if SDFR_IN_PART(1)
int sdfr_forward(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                 const float* quat, const float* inv_scale, int batch, int W, int H, float cx,
                 float cy, float fx, float fy, float threshold, float* depth,
                 const sdfr_cell_bounds* bounds, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H)) return rc;
  if (batch == 0 || W == 0 || H == 0) return 0;
  if (!depth) return fail(SDFR_E_NULL, "depth is NULL");
  FwdParams P = fwd_params(sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           threshold, depth, bounds);
  return launch_forward<0, false>(P, batch, (cudaStream_t)stream);
}

#endif
#if SDFR_IN_PART(1)
int sdfr_forward_stats(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                       const float* quat, const float* inv_scale, int batch, int W, int H,
                       float cx, float cy, float fx, float fy, float threshold, float* depth,
                       unsigned long long* stats, const sdfr_cell_bounds* bounds, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H)) return rc;
  if (batch == 0 || W == 0 || H == 0) return 0;
  if (!depth || !stats) return fail(SDFR_E_NULL, "depth or stats is NULL");
  FwdParams P = fwd_params(sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           threshold, depth, bounds);
  P.stats = stats;
  return launch_forward<0, true>(P, batch, (cudaStream_t)stream);
}

#endif
#if SDFR_IN_PART(3)
int sdfr_backward(const float* grad_depth, const float* depth, const float* sdf, int R,
                  long long sdf_stride, int layout, const float* pos, const float* quat,
                  const float* inv_scale, int batch, int W, int H, float cx, float cy, float fx,
                  float fy, float* gs, long long gs_stride, float* gp, float* gq, float* gi,
                  unsigned flags, const sdfr_cell_bounds* bounds, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H)) return rc;
  if (int rc = check_backward_outputs(flags, gs, gs_stride, gp, gq, gi)) return rc;
  if (batch == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const bool empty = W == 0 || H == 0;
  if (int rc = zero_grads(empty ? flags : flags & ~SDFR_GRAD_SDF, R, batch, gs, gs_stride, gp, gq,
                          gi, s))
    return rc;
  if (empty) return 0;
  if (!grad_depth || !depth) return fail(SDFR_E_NULL, "grad_depth or depth is NULL");
  BwdParams P = bwd_params(depth, sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           gs, gs_stride, gp, gq, gi, flags, bounds);
  P.grad_depth = grad_depth;
  return launch_backward<0>(P, batch, (flags & SDFR_ZERO_GRADS) != 0, s);
}

#endif
#if SDFR_IN_PART(1)
int sdfr_compare_forward(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                         const float* quat, const float* inv_scale, int batch, int W, int H,
                         float cx, float cy, float fx, float fy, float threshold,
                         const float* depth_obs, long long obs_stride, float* depth,
                         float* loss_sum, float* n_overlap, unsigned flags,
                         const sdfr_cell_bounds* bounds, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H)) return rc;
  if (flags & ~SDFR_ZERO_GRADS) return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (obs_stride < 0) return fail(SDFR_E_SHAPE, "negative obs_stride");
  if (batch == 0) return 0;
  if (!loss_sum || !n_overlap) return fail(SDFR_E_NULL, "loss_sum or n_overlap is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  if (flags & SDFR_ZERO_GRADS) {
    if (int rc = zero_async(loss_sum, sizeof(float) * batch, s)) return rc;
    if (int rc = zero_async(n_overlap, sizeof(float) * batch, s)) return rc;
  }
  if (W == 0 || H == 0) return 0;
  if (!depth || !depth_obs) return fail(SDFR_E_NULL, "depth or depth_obs is NULL");
  FwdParams P = fwd_params(sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           threshold, depth, bounds);
  P.depth_obs = depth_obs;
  P.obs_stride = obs_stride;
  P.loss_sum = loss_sum;
  P.n_overlap = n_overlap;
  return launch_forward<1, false>(P, batch, s);
}

#endif
#if SDFR_IN_PART(3)
int sdfr_compare_backward(const float* depth, const float* depth_obs, long long obs_stride,
                          const float* n_overlap, const float* upstream, const float* sdf, int R,
                          long long sdf_stride, int layout, const float* pos, const float* quat,
                          const float* inv_scale, int batch, int W, int H, float cx, float cy,
                          float fx, float fy, float* gs, long long gs_stride, float* gp,
                          float* gq, float* gi, unsigned flags, const sdfr_cell_bounds* bounds,
                          void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H)) return rc;
  if (int rc = check_backward_outputs(flags, gs, gs_stride, gp, gq, gi)) return rc;
  if (obs_stride < 0) return fail(SDFR_E_SHAPE, "negative obs_stride");
  if (batch == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const bool empty = W == 0 || H == 0;
  if (int rc = zero_grads(empty ? flags : flags & ~SDFR_GRAD_SDF, R, batch, gs, gs_stride, gp, gq,
                          gi, s))
    return rc;
  if (empty) return 0;
  if (!depth || !depth_obs || !n_overlap)
    return fail(SDFR_E_NULL, "depth, depth_obs or n_overlap is NULL");
  BwdParams P = bwd_params(depth, sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           gs, gs_stride, gp, gq, gi, flags, bounds);
  P.depth_obs = depth_obs;
  P.obs_stride = obs_stride;
  P.n_overlap = n_overlap;
  P.upstream = upstream;
  return launch_backward<1>(P, batch, (flags & SDFR_ZERO_GRADS) != 0, s);
}

#endif
#if SDFR_IN_PART(2)
static int compare_fused_impl(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                              const float* quat, const float* inv_scale, int batch, int W, int H,
                              float cx, float cy, float fx, float fy, float threshold,
                              const float* depth_obs, long long obs_stride, float* depth,
                              float* loss_sum, float* n_overlap, float rel_threshold, float* n_inlier,
                              float* gs, long long gs_stride, float* gp, float* gq, float* gi,
                              unsigned flags, const sdfr_cell_bounds* bounds, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H)) return rc;
  if (int rc = check_backward_outputs(flags, gs, gs_stride, gp, gq, gi)) return rc;
  if (obs_stride < 0) return fail(SDFR_E_SHAPE, "negative obs_stride");
  if ((flags & SDFR_GRAD_SDF) && gs_stride == 0 && batch > 1)
    return fail(SDFR_E_SHAPE,
                "fused compare needs one grad_sdf grid per hypothesis (the deferred 1/n_overlap "
                "differs per hypothesis); use sdfr_compare_forward + sdfr_compare_backward");
  if (batch == 0) return 0;
  if (!loss_sum || !n_overlap) return fail(SDFR_E_NULL, "loss_sum or n_overlap is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  if (flags & SDFR_ZERO_GRADS) {
    /* the gradient grids by memset, every small buffer (sums and pose gradients) in one launch */
    if (int rc = zero_grads(flags & ~(SDFR_GRAD_POSITION | SDFR_GRAD_ORIENTATION | SDFR_GRAD_INV_SCALE), R, batch,
                            gs, gs_stride, gp, gq, gi, s))
      return rc;
    const int na = (flags & SDFR_GRAD_POSITION) ? 3 * batch : 0;
    const int nb = (flags & SDFR_GRAD_ORIENTATION) ? 4 * batch : 0;
    const int nc = (flags & SDFR_GRAD_INV_SCALE) ? batch : 0;
    sdfr_zero_sums_and_small_kernel<<<batch > 512 ? 16 : 1, 256, 0, s>>>(loss_sum, n_overlap, n_inlier, batch, gp,
                                                                       na, gq, nb, gi, nc);
    if (int rc = check_launch("sdfr_zero_sums_and_small_kernel")) return rc;
  }
  if (W == 0 || H == 0) return 0;
  if (!depth || !depth_obs) return fail(SDFR_E_NULL, "depth or depth_obs is NULL");
  FwdParams P = fwd_params(sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           threshold, depth, bounds);
  P.depth_obs = depth_obs;
  P.obs_stride = obs_stride;
  P.loss_sum = loss_sum;
  P.n_overlap = n_overlap;
  P.n_inlier = n_inlier;
  P.inlier_threshold = rel_threshold;
  P.grad_sdf = gs;
  P.grad_sdf_stride = gs_stride;
  P.grad_position = gp;
  P.grad_orientation = gq;
  P.grad_inv_scale = gi;
  P.flags = flags;
  return launch_forward<2, false>(P, batch, s);
}

int sdfr_compare_fused(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                       const float* quat, const float* inv_scale, int batch, int W, int H,
                       float cx, float cy, float fx, float fy, float threshold,
                       const float* depth_obs, long long obs_stride, float* depth,
                       float* loss_sum, float* n_overlap, float* gs, long long gs_stride,
                       float* gp, float* gq, float* gi, unsigned flags,
                       const sdfr_cell_bounds* bounds, void* stream) {
  return compare_fused_impl(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H, cx, cy, fx, fy,
                            threshold, depth_obs, obs_stride, depth, loss_sum, n_overlap, 0.0f, nullptr,
                            gs, gs_stride, gp, gq, gi, flags, bounds, stream);
}

int sdfr_compare_fused_inliers(const float* sdf, int R, long long sdf_stride, int layout,
                               const float* pos, const float* quat, const float* inv_scale, int batch,
                               int W, int H, float cx, float cy, float fx, float fy, float threshold,
                               const float* depth_obs, long long obs_stride, float* depth,
                               float* loss_sum, float* n_overlap, float rel_threshold, float* n_inlier,
                               float* gs, long long gs_stride, float* gp, float* gq, float* gi,
                               unsigned flags, const sdfr_cell_bounds* bounds, void* stream) {
  if (batch > 0 && !n_inlier) return fail(SDFR_E_NULL, "n_inlier is NULL");
  if (!(rel_threshold <= 1.0f))
    return fail(SDFR_E_SHAPE, "fused inlier count: rel_threshold <= 1 expected (a missed pixel has "
                              "relative error 1; use sdfr_inlier_count for larger thresholds)");
  return compare_fused_impl(sdf, R, sdf_stride, layout, pos, quat, inv_scale, batch, W, H, cx, cy, fx, fy,
                            threshold, depth_obs, obs_stride, depth, loss_sum, n_overlap, rel_threshold,
                            n_inlier, gs, gs_stride, gp, gq, gi, flags, bounds, stream);
}

#endif
#if SDFR_IN_PART(3)
int sdfr_scale_grads(const float* n_overlap, const float* upstream, int R, int batch, float* gs,
                     long long gs_stride, float* gp, float* gq, float* gi, unsigned flags,
                     const sdfr_cell_bounds* bounds, long long bounds_stride, void* stream) {
  if (batch < 0) return fail(SDFR_E_SHAPE, "negative batch");
  if (R < 2 || R > 1024) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (int rc = check_backward_outputs(flags & ~SDFR_ZERO_GRADS, gs, gs_stride, gp, gq, gi)) return rc;
  if (batch == 0 || !(flags & SDFR_GRAD_ALL)) return 0;
  if (!n_overlap) return fail(SDFR_E_NULL, "n_overlap is NULL");
  if ((flags & SDFR_GRAD_SDF) && gs_stride == 0 && batch > 1)
    return fail(SDFR_E_SHAPE, "a shared grad_sdf grid cannot be scaled per hypothesis");
  if (bounds_stride != 0 && bounds_stride != 1) return fail(SDFR_E_SHAPE, "bounds_stride must be 0 (one shared grid) or 1");
  const CellBounds* cb = reinterpret_cast<const CellBounds*>(bounds);
  const long long elems = (long long)R * R * R;
  const int gx = (flags & SDFR_GRAD_SDF) ? (int)((elems / 4 + 2047) / 2048 < 1 ? 1 : (elems / 4 + 2047) / 2048) : 1;
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    const int nz = batch - z0 < 65535 ? batch - z0 : 65535;
    sdfr_scale_grads_kernel<<<dim3(gx, nz), 256, 0, (cudaStream_t)stream>>>(
        n_overlap + z0, upstream ? upstream + z0 : nullptr, elems,
        gs ? gs + (size_t)z0 * gs_stride : nullptr, gs_stride, gp ? gp + 3 * (size_t)z0 : nullptr,
        gq ? gq + 4 * (size_t)z0 : nullptr, gi ? gi + z0 : nullptr, flags,
        cb ? cb + (size_t)z0 * bounds_stride : nullptr, (int)bounds_stride, R);
  }
  return check_launch("sdfr_scale_grads_kernel");
}

#endif
#if SDFR_IN_PART(3)
int sdfr_forward_composite(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                           const float* quat, const float* inv_scale, int n_objects, int W,
                           int H, float cx, float cy, float fx, float fy, float threshold,
                           float* depth, int* winner, const sdfr_cell_bounds* bounds, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, n_objects, W, H)) return rc;
  if (W == 0 || H == 0) return 0;
  if (!depth || !winner) return fail(SDFR_E_NULL, "depth or winner is NULL");
  FwdParams P = fwd_params(sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           threshold, depth, bounds);
  const bool skewed = P.grid.py != P.grid.R;
#define SDFR_CALL(RT, LT) \
  sdfr_forward_composite_kernel<RT, LT><<<tile_grid(W, H, 1), kThreads, 0, (cudaStream_t)stream>>>(P, n_objects, winner)
  SDFR_DISPATCH_RT_LT(R, skewed, SDFR_CALL);
#undef SDFR_CALL
  return check_launch("sdfr_forward_composite_kernel");
}

int sdfr_backward_composite(const float* grad_depth, const float* depth, const int* winner,
                            const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                            const float* quat, const float* inv_scale, int n_objects, int W,
                            int H, float cx, float cy, float fx, float fy, float* gs,
                            long long gs_stride, float* gp, float* gq, float* gi, unsigned flags,
                            void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, inv_scale, n_objects, W, H)) return rc;
  if (int rc = check_backward_outputs(flags, gs, gs_stride, gp, gq, gi)) return rc;
  if (n_objects == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (int rc = zero_grads(flags, R, n_objects, gs, gs_stride, gp, gq, gi, s)) return rc;
  if (W == 0 || H == 0) return 0;
  if (!grad_depth || !depth || !winner)
    return fail(SDFR_E_NULL, "grad_depth, depth or winner is NULL");
  BwdParams P = bwd_params(depth, sdf, R, sdf_stride, layout, pos, quat, inv_scale, W, H, cx, cy, fx, fy,
                           gs, gs_stride, gp, gq, gi, flags);
  P.grad_depth = grad_depth;
  P.winner = winner;
  P.n_objects = n_objects;
  const bool want_sdf = (flags & SDFR_GRAD_SDF) != 0;
  const bool want_pose =
      (flags & (SDFR_GRAD_POSITION | SDFR_GRAD_ORIENTATION | SDFR_GRAD_INV_SCALE)) != 0;
  if (!want_sdf && !want_pose) return 0;
  const dim3 grid = tile_grid(W, H, 1);
  const bool skewed = P.grid.py != P.grid.R;
#define SDFR_CALL(RT, LT)                                                                         \
  do {                                                                                            \
    if (want_sdf && want_pose) sdfr_backward_composite_kernel<RT, LT, true, true><<<grid, kThreads, 0, s>>>(P);  \
    else if (want_sdf) sdfr_backward_composite_kernel<RT, LT, true, false><<<grid, kThreads, 0, s>>>(P);         \
    else sdfr_backward_composite_kernel<RT, LT, false, true><<<grid, kThreads, 0, s>>>(P);                       \
  } while (0)
  SDFR_DISPATCH_RT_LT(R, skewed, SDFR_CALL);
#undef SDFR_CALL
  return check_launch("sdfr_backward_composite_kernel");
}

static int launch_bounds_scan(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                              const float* inv_scale, int batch, float threshold, sdfr_cell_bounds* bounds,
                              float* skewed, long long skewed_stride, cudaStream_t s) {
  const int n_grids = sdf_stride == 0 ? 1 : batch;
  const Grid G = make_grid(R, layout);
  const Grid GS = make_grid(R, kLayoutSkewed);
  CellBounds* out = reinterpret_cast<CellBounds*>(bounds);
  sdfr_bounds_init_kernel<<<n_grids, n_grids == 1 ? 256 : 32, 0, s>>>(pos, inv_scale, batch, n_grids, threshold, out);
  for (int z0 = 0; z0 < n_grids; z0 += 65535) {
    const int nz = n_grids - z0 < 65535 ? n_grids - z0 : 65535;
    const dim3 grid(R, nz); /* one CTA per voxel layer and grid */
    if (skewed)
      sdfr_bounds_scan_kernel<true><<<grid, 256, 0, s>>>(sdf + (size_t)z0 * sdf_stride, sdf_stride, R, G.py, G.px,
                                                         out + z0, skewed + (size_t)z0 * skewed_stride,
                                                         skewed_stride, GS.py, GS.px);
    else
      sdfr_bounds_scan_kernel<false><<<grid, 256, 0, s>>>(sdf + (size_t)z0 * sdf_stride, sdf_stride, R, G.py, G.px,
                                                          out + z0, nullptr, 0, 0, 0);
  }
  return check_launch("sdfr_bounds_scan_kernel");
}

int sdfr_grid_bounds(const float* sdf, int R, long long sdf_stride, int layout, const float* pos,
                     const float* inv_scale, int batch, float threshold, sdfr_cell_bounds* bounds,
                     void* stream) {
  if (layout != SDFR_LAYOUT_DENSE && layout != SDFR_LAYOUT_SKEWED) return fail(SDFR_E_FLAGS, "unknown sdf_layout");
  if (R < 2 || R > 1024) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (batch < 0 || sdf_stride < 0) return fail(SDFR_E_SHAPE, "negative batch or sdf_stride");
  if (!(threshold >= 0.0f)) return fail(SDFR_E_SHAPE, "threshold must be >= 0");
  if (batch == 0) return 0;
  if (!sdf || !pos || !inv_scale || !bounds) return fail(SDFR_E_NULL, "grid bounds: NULL pointer");
  return launch_bounds_scan(sdf, R, sdf_stride, layout, pos, inv_scale, batch, threshold, bounds, nullptr, 0,
                            (cudaStream_t)stream);
}

int sdfr_grid_slab_minima(const float* sdf, int R, long long sdf_stride, int layout, int n_grids,
                          float* minima, void* stream) {
  if (layout != SDFR_LAYOUT_DENSE && layout != SDFR_LAYOUT_SKEWED) return fail(SDFR_E_FLAGS, "unknown sdf_layout");
  if (R < 2 || R > kSlabMaxR) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (n_grids < 0 || sdf_stride < 0) return fail(SDFR_E_SHAPE, "negative n_grids or sdf_stride");
  if (n_grids == 0) return 0;
  if (!sdf || !minima) return fail(SDFR_E_NULL, "slab minima: NULL pointer");
  const Grid G = make_grid(R, layout);
  cudaStream_t s = (cudaStream_t)stream;
  const long long total = (long long)n_grids * 3 * R;
  sdfr_fill_kernel<<<(int)((total + 255) / 256 < 1024 ? (total + 255) / 256 : 1024), 256, 0, s>>>(minima, total, 3.0e38f);
  for (int z0 = 0; z0 < n_grids; z0 += 65535) {
    const int nz = n_grids - z0 < 65535 ? n_grids - z0 : 65535;
    sdfr_slab_minima_kernel<<<dim3(R, nz), 256, 0, s>>>(sdf + (size_t)z0 * sdf_stride, sdf_stride, R, G.py, G.px,
                                                        minima + (size_t)z0 * 3 * R);
  }
  return check_launch("sdfr_slab_minima_kernel");
}

int sdfr_bounds_from_minima(const float* minima, int R, int n_grids, const float* pos, const float* inv_scale,
                            int batch, float threshold, sdfr_cell_bounds* bounds, void* stream) {
  if (R < 2 || R > kSlabMaxR) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (batch < 0 || n_grids < 0) return fail(SDFR_E_SHAPE, "negative batch or n_grids");
  if (!(threshold >= 0.0f)) return fail(SDFR_E_SHAPE, "threshold must be >= 0");
  if (batch == 0 || n_grids == 0) return 0;
  if (n_grids != 1 && n_grids != batch)
    return fail(SDFR_E_SHAPE, "bounds from minima: one grid per hypothesis or one shared grid expected");
  if (!minima || !pos || !inv_scale || !bounds) return fail(SDFR_E_NULL, "bounds from minima: NULL pointer");
  sdfr_bounds_from_minima_kernel<<<n_grids, 256, 0, (cudaStream_t)stream>>>(
      minima, R, pos, inv_scale, batch, n_grids, threshold, reinterpret_cast<CellBounds*>(bounds));
  return check_launch("sdfr_bounds_from_minima_kernel");
}

int sdfr_skew_grids_bounds(const float* sdf, int R, long long sdf_stride, int batch, float* skewed,
                           long long skewed_stride, const float* pos, const float* inv_scale, float threshold,
                           sdfr_cell_bounds* bounds, void* stream) {
  if (R < 2 || R > 1024) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (batch < 0 || sdf_stride < 0) return fail(SDFR_E_SHAPE, "negative batch or sdf_stride");
  if (!(threshold >= 0.0f)) return fail(SDFR_E_SHAPE, "threshold must be >= 0");
  if (batch == 0) return 0;
  if (!sdf || !skewed || !pos || !inv_scale || !bounds) return fail(SDFR_E_NULL, "skew + bounds: NULL pointer");
  const Grid G = make_grid(R, kLayoutSkewed);
  if (skewed_stride < (long long)R * G.px)
    return fail(SDFR_E_SHAPE, "skewed_stride smaller than sdfr_skewed_pitches' elems");
  if (sdf_stride == 0 && batch > 1) skewed_stride = 0; /* one shared grid: one skewed copy */
  return launch_bounds_scan(sdf, R, sdf_stride, SDFR_LAYOUT_DENSE, pos, inv_scale, batch, threshold, bounds, skewed,
                            skewed_stride, (cudaStream_t)stream);
}

int sdfr_skewed_pitches(int R, int* pitch_y, int* pitch_x, long long* elems) {
  if (R < 2 || R > 1024) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  const Grid G = make_grid(R, kLayoutSkewed);
  if (pitch_y) *pitch_y = G.py;
  if (pitch_x) *pitch_x = G.px;
  if (elems) *elems = (long long)R * G.px;
  return 0;
}

int sdfr_skew_grids(const float* sdf, int R, long long sdf_stride, int batch, float* skewed,
                    long long skewed_stride, void* stream) {
  if (R < 2 || R > 1024) return fail(SDFR_E_SHAPE, "resolution must be in [2, 1024]");
  if (batch < 0 || sdf_stride < 0) return fail(SDFR_E_SHAPE, "negative batch or sdf_stride");
  if (batch == 0) return 0;
  if (!sdf || !skewed) return fail(SDFR_E_NULL, "NULL grid pointer");
  const Grid G = make_grid(R, kLayoutSkewed);
  if (skewed_stride < (long long)R * G.px)
    return fail(SDFR_E_SHAPE, "skewed_stride smaller than sdfr_skewed_pitches' elems");
  const long long work = ((long long)R * R * R + 3) / 4;
  int gx = (int)((work + 255) / 256 < 1024 ? (work + 255) / 256 : 1024);
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    const int nz = batch - z0 < 65535 ? batch - z0 : 65535;
    sdfr_skew_kernel<<<dim3(gx, nz), 256, 0, (cudaStream_t)stream>>>(
        sdf + (size_t)z0 * sdf_stride, sdf_stride, skewed + (size_t)z0 * skewed_stride,
        skewed_stride, R, G.py, G.px);
  }
  return check_launch("sdfr_skew_kernel");
}

#endif
#if SDFR_IN_PART(4)
int sdfr_point_loss_forward(const float* points, long long points_stride, int n_points,
                            const float* sdf, int R, long long sdf_stride, int layout,
                            const float* pos, const float* quat, const float* scale, int batch,
                            float* loss_sum, unsigned flags, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, scale, batch, 1, 1)) return rc;
  if (flags & ~SDFR_ZERO_GRADS) return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (n_points < 0 || points_stride < 0) return fail(SDFR_E_SHAPE, "negative n_points or stride");
  if (batch == 0) return 0;
  if (!loss_sum) return fail(SDFR_E_NULL, "loss_sum is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  if (flags & SDFR_ZERO_GRADS)
    if (int rc = zero_async(loss_sum, sizeof(float) * batch, s)) return rc;
  if (n_points == 0) return 0;
  if (!points) return fail(SDFR_E_NULL, "points is NULL");
  PointParams P;
  memset(&P, 0, sizeof(P));
  P.points = points; P.points_stride = points_stride; P.n_points = n_points;
  P.sdf = sdf; P.sdf_stride = sdf_stride; P.grid = make_grid(R, layout);
  P.position = pos; P.orientation = quat; P.scale = scale;
  P.loss_sum = loss_sum;
  return launch_point_loss<false>(P, batch, s);
}

int sdfr_point_loss_backward(const float* points, long long points_stride, int n_points,
                             const float* sdf, int R, long long sdf_stride, int layout,
                             const float* pos, const float* quat, const float* scale, int batch,
                             const float* upstream, float* gs, long long gs_stride, float* gp,
                             float* gq, float* gscale, unsigned flags, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, scale, batch, 1, 1)) return rc;
  if (flags & SDFR_SDF_GRAD_EXACT) return fail(SDFR_E_FLAGS, "the point loss has one weight list");
  if (int rc = check_backward_outputs(flags, gs, gs_stride, gp, gq, gscale)) return rc;
  if (n_points < 0 || points_stride < 0) return fail(SDFR_E_SHAPE, "negative n_points or stride");
  if (batch == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (int rc = zero_grads(flags, R, batch, gs, gs_stride, gp, gq, gscale, s)) return rc;
  if (n_points == 0) return 0;
  if (!points) return fail(SDFR_E_NULL, "points is NULL");
  PointParams P;
  memset(&P, 0, sizeof(P));
  P.points = points; P.points_stride = points_stride; P.n_points = n_points;
  P.sdf = sdf; P.sdf_stride = sdf_stride; P.grid = make_grid(R, layout);
  P.position = pos; P.orientation = quat; P.scale = scale;
  P.upstream = upstream;
  P.grad_sdf = gs; P.grad_sdf_stride = gs_stride;
  P.grad_position = gp; P.grad_orientation = gq; P.grad_scale = gscale;
  P.flags = flags;
  return launch_point_loss<true>(P, batch, s);
}

int sdfr_point_loss_fused(const float* points, long long points_stride, int n_points,
                          const float* sdf, int R, long long sdf_stride, int layout,
                          const float* pos, const float* quat, const float* scale, int batch,
                          const float* upstream, float* loss_sum, float* gs, long long gs_stride,
                          float* gp, float* gq, float* gscale, unsigned flags, void* stream) {
  if (int rc = check_common(sdf, R, sdf_stride, layout, pos, quat, scale, batch, 1, 1)) return rc;
  if (flags & SDFR_SDF_GRAD_EXACT) return fail(SDFR_E_FLAGS, "the point loss has one weight list");
  if (int rc = check_backward_outputs(flags & ~SDFR_LOSS_WEIGHTED, gs, gs_stride, gp, gq, gscale)) return rc;
  if (n_points < 0 || points_stride < 0) return fail(SDFR_E_SHAPE, "negative n_points or stride");
  if (batch == 0) return 0;
  if (!loss_sum) return fail(SDFR_E_NULL, "loss_sum is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  if (flags & SDFR_ZERO_GRADS)
    if (int rc = zero_async(loss_sum, sizeof(float) * batch, s)) return rc;
  if (int rc = zero_grads(flags, R, batch, gs, gs_stride, gp, gq, gscale, s)) return rc;
  if (n_points == 0) return 0;
  if (!points) return fail(SDFR_E_NULL, "points is NULL");
  PointParams P;
  memset(&P, 0, sizeof(P));
  P.points = points; P.points_stride = points_stride; P.n_points = n_points;
  P.sdf = sdf; P.sdf_stride = sdf_stride; P.grid = make_grid(R, layout);
  P.position = pos; P.orientation = quat; P.scale = scale;
  P.upstream = upstream;
  P.loss_sum = loss_sum;
  P.grad_sdf = gs; P.grad_sdf_stride = gs_stride;
  P.grad_position = gp; P.grad_orientation = gq; P.grad_scale = gscale;
  P.flags = flags;
  return launch_point_loss<true, true>(P, batch, s);
}

int sdfr_hypothesis_step(float* position, float* orientation, float* scale, float* latent,
                         int latent_size, int batch, float* loss_sum, float* n_overlap,
                         float* gr_position, float* gr_orientation, float* gr_inv_scale,
                         float depth_weight, float* point_sum, float point_weight,
                         float* g2_position, float* g2_orientation, float* g2_scale,
                         float* g_latent, float* g_orientation_raw, float* loss_extra, float* exp_avg,
                         float* exp_avg_sq, int* step, const float* lr, float beta1, float beta2, float eps,
                         float* unit_orientation, float* inv_scale, float* loss, unsigned flags,
                         void* stream) {
  if (flags & ~(SDFR_STEP_CLEAR_INPUTS | SDFR_STEP_NO_UPDATE)) return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (batch < 0 || latent_size < 0 || latent_size > kStepMaxLatent)
    return fail(SDFR_E_SHAPE, "hypothesis step: batch >= 0 and 0 <= latent_size <= 64 expected");
  if (batch == 0) return 0;
  if (!position || !orientation || !scale) return fail(SDFR_E_NULL, "hypothesis step: NULL parameter pointer");
  const bool update = !(flags & SDFR_STEP_NO_UPDATE);
  if (update && (!exp_avg || !exp_avg_sq || !step || !lr))
    return fail(SDFR_E_NULL, "hypothesis step: NULL optimiser state or learning rates");
  if (loss_sum && !n_overlap) return fail(SDFR_E_NULL, "hypothesis step: loss_sum without n_overlap");
  if ((gr_position || gr_orientation || gr_inv_scale) && !n_overlap)
    return fail(SDFR_E_NULL, "hypothesis step: raw render gradients without n_overlap");
  StepParams P;
  memset(&P, 0, sizeof(P));
  P.position = position; P.orientation = orientation; P.scale = scale;
  P.latent = latent_size > 0 ? latent : nullptr;
  P.latent_size = (latent && g_latent) ? latent_size : 0;
  P.state_stride = 8 + latent_size;
  P.batch = batch;
  P.loss_sum = loss_sum; P.n_overlap = n_overlap;
  P.gr_position = gr_position; P.gr_orientation = gr_orientation; P.gr_inv_scale = gr_inv_scale;
  P.depth_weight = depth_weight;
  P.point_sum = point_sum; P.point_weight = point_weight;
  P.g2_position = g2_position; P.g2_orientation = g2_orientation; P.g2_scale = g2_scale;
  P.g_latent = P.latent_size > 0 ? g_latent : nullptr;
  P.g_orientation_raw = g_orientation_raw; P.loss_extra = loss_extra;
  P.exp_avg = exp_avg; P.exp_avg_sq = exp_avg_sq; P.step = step;
  if (lr) for (int i = 0; i < 4; ++i) P.lr[i] = lr[i];
  P.beta1 = beta1; P.beta2 = beta2; P.eps = eps;
  P.unit_orientation = unit_orientation; P.inv_scale = inv_scale; P.loss = loss;
  P.flags = flags;
  sdfr_hypothesis_step_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(P);
  return check_launch("sdfr_hypothesis_step_kernel");
}

static int view_check(int n_views, int batch) {
  if (n_views < 0 || batch < 0 || (long long)n_views * batch > (1ll << 30))
    return fail(SDFR_E_SHAPE, "views: n_views >= 0 and batch >= 0 expected");
  return 0;
}

int sdfr_view_poses(const float* position, const float* unit_orientation, const float* inv_scale,
                    const float* cam_position, const float* cam_orientation, int n_views, int batch,
                    float* position_c, float* orientation_c, float* inv_scale_c, void* stream) {
  if (int rc = view_check(n_views, batch)) return rc;
  if (n_views == 0 || batch == 0) return 0;
  if (!position || !unit_orientation || !inv_scale || !cam_position || !cam_orientation || !position_c ||
      !orientation_c || !inv_scale_c)
    return fail(SDFR_E_NULL, "view poses: NULL pointer");
  ViewParams P;
  memset(&P, 0, sizeof(P));
  P.position = position; P.unit_orientation = unit_orientation; P.inv_scale = inv_scale;
  P.cam_position = cam_position; P.cam_orientation = cam_orientation;
  P.n_views = n_views; P.batch = batch;
  P.position_c = position_c; P.orientation_c = orientation_c; P.inv_scale_c = inv_scale_c;
  sdfr_view_poses_kernel<<<(n_views * batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(P);
  return check_launch("sdfr_view_poses_kernel");
}

int sdfr_views_pull_back(const float* cam_orientation, const float* scale, int n_views, int batch,
                         float* gr_position, float* gr_orientation, float* gr_inv_scale, float* g2_position,
                         float* g2_orientation, float* g2_scale, float* loss_sum, float* n_overlap,
                         float depth_weight, float* point_sum, float* g_position, float* g_orientation,
                         float* g_scale, float* loss, unsigned flags, void* stream) {
  if (int rc = view_check(n_views, batch)) return rc;
  if (flags & ~SDFR_STEP_CLEAR_INPUTS) return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (batch == 0) return 0;
  if (!cam_orientation || !scale || !g_position || !g_orientation || !g_scale || !loss)
    return fail(SDFR_E_NULL, "views pull back: NULL pointer");
  if ((loss_sum == nullptr) != (n_overlap == nullptr))
    return fail(SDFR_E_NULL, "views pull back: loss_sum and n_overlap go together");
  ViewParams P;
  memset(&P, 0, sizeof(P));
  P.cam_orientation = cam_orientation; P.scale = scale; P.n_views = n_views; P.batch = batch;
  P.gr_position = gr_position; P.gr_orientation = gr_orientation; P.gr_inv_scale = gr_inv_scale;
  P.g2_position = g2_position; P.g2_orientation = g2_orientation; P.g2_scale = g2_scale;
  P.loss_sum = loss_sum; P.n_overlap = n_overlap; P.depth_weight = depth_weight; P.point_sum = point_sum;
  P.g_position = g_position; P.g_orientation = g_orientation; P.g_scale = g_scale; P.loss = loss;
  P.flags = flags;
  sdfr_views_pull_back_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(P);
  return check_launch("sdfr_views_pull_back_kernel");
}

int sdfr_point_constraint(const float* orientation, int batch, const float* source, const float* target,
                          float weight, float* g_orientation_raw, float* loss, void* stream) {
  if (batch < 0) return fail(SDFR_E_SHAPE, "point constraint: batch >= 0 expected");
  if (batch == 0) return 0;
  if (!orientation || !source || !target) return fail(SDFR_E_NULL, "point constraint: NULL pointer");
  ConstraintParams P;
  memset(&P, 0, sizeof(P));
  P.orientation = orientation; P.batch = batch; P.weight = weight;
  for (int k = 0; k < 3; ++k) { P.source[k] = source[k]; P.target[k] = target[k]; }
  P.g_orientation_raw = g_orientation_raw; P.loss = loss;
  sdfr_point_constraint_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(P);
  return check_launch("sdfr_point_constraint_kernel");
}

int sdfr_inlier_count(const float* depth, const float* depth_obs, long long obs_stride, int batch,
                      int width, int height, float rel_threshold, float* n_inlier, float* n_valid,
                      unsigned flags, void* stream) {
  if (flags & ~SDFR_ZERO_GRADS) return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (batch < 0 || width < 1 || height < 1 || obs_stride < 0 || (long long)width * height > (1ll << 30))
    return fail(SDFR_E_SHAPE, "inlier count: batch >= 0, a non-empty image and obs_stride >= 0 expected");
  if (batch == 0) return 0;
  if (!depth || !depth_obs || !n_inlier || !n_valid) return fail(SDFR_E_NULL, "inlier count: NULL pointer");
  cudaStream_t s = (cudaStream_t)stream;
  if (flags & SDFR_ZERO_GRADS) {
    if (int rc = zero_async(n_inlier, sizeof(float) * batch, s)) return rc;
    if (int rc = zero_async(n_valid, sizeof(float) * batch, s)) return rc;
  }
  InlierParams P;
  memset(&P, 0, sizeof(P));
  P.depth = depth; P.obs = depth_obs; P.obs_stride = obs_stride;
  P.pixels = width * height; P.threshold = rel_threshold;
  P.n_inlier = n_inlier; P.n_valid = n_valid;
  const bool vec = (P.pixels % 4 == 0) && (obs_stride % 4 == 0) &&
                   ((reinterpret_cast<uintptr_t>(depth) | reinterpret_cast<uintptr_t>(depth_obs)) & 15) == 0;
  int gx = ((vec ? P.pixels / 4 : P.pixels) + 1023) / 1024; /* ~4 loads per thread */
  gx = gx < 1 ? 1 : (gx > 256 ? 256 : gx);
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid(gx, batch - z0 < 65535 ? batch - z0 : 65535);
    if (vec) sdfr_inlier_count_kernel<true><<<grid, 256, 0, s>>>(P);
    else sdfr_inlier_count_kernel<false><<<grid, 256, 0, s>>>(P);
  }
  return check_launch("sdfr_inlier_count_kernel");
}

int sdfr_track_best(float* n_inlier, float* n_valid, const float* position, const float* orientation,
                    const float* scale, const float* latent, int latent_size, int batch,
                    const int* step, float* ratio, float* best_ratio, int* best_iteration,
                    float* best_position, float* best_orientation, float* best_scale,
                    float* best_latent, unsigned flags, void* stream) {
  if (flags & ~(SDFR_STEP_CLEAR_INPUTS | SDFR_TRACK_KEEP_VALID)) return fail(SDFR_E_FLAGS, "unknown flag bits");
  if (batch < 0 || latent_size < 0) return fail(SDFR_E_SHAPE, "track best: batch >= 0 and latent_size >= 0 expected");
  if (batch == 0) return 0;
  if (!n_inlier || !n_valid || !position || !orientation || !scale || !best_ratio || !best_iteration ||
      !best_position || !best_orientation || !best_scale)
    return fail(SDFR_E_NULL, "track best: NULL pointer");
  TrackParams P;
  memset(&P, 0, sizeof(P));
  P.n_inlier = n_inlier; P.n_valid = n_valid;
  P.position = position; P.orientation = orientation; P.scale = scale;
  P.latent = latent_size > 0 ? latent : nullptr;
  P.latent_size = latent_size; P.batch = batch; P.step = step; P.ratio = ratio;
  P.best_ratio = best_ratio; P.best_iteration = best_iteration;
  P.best_position = best_position; P.best_orientation = best_orientation; P.best_scale = best_scale;
  P.best_latent = best_latent;
  P.flags = flags;
  sdfr_track_best_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(P);
  return check_launch("sdfr_track_best_kernel");
}

int sdfr_decoder_tail_forward(const float* x, int channels, int in_size, const float* weight,
                              const float* bias, const float* base, int batch, int R, float* sdf,
                              long long sdf_stride, int layout, void* stream) {
  if (int rc = tail_check(channels, in_size, R, batch)) return rc;
  if (layout != SDFR_LAYOUT_DENSE && layout != SDFR_LAYOUT_SKEWED)
    return fail(SDFR_E_FLAGS, "unknown sdf_layout");
  if (batch == 0) return 0;
  if (!x || !weight || !sdf) return fail(SDFR_E_NULL, "decoder tail: x, weight or sdf is NULL");
  const Grid G = make_grid(R, layout);
  if (sdf_stride < (long long)R * G.px)
    return fail(SDFR_E_SHAPE, "decoder tail: sdf_stride smaller than one grid in this layout");
  TailParams P;
  memset(&P, 0, sizeof(P));
  P.x = x; P.weight = weight; P.bias = bias; P.base = base;
  P.C = channels; P.S = in_size; P.R = R;
  P.out = sdf; P.out_stride = sdf_stride; P.py = G.py; P.px = G.px;
  return launch_tail_forward(P, batch, (cudaStream_t)stream);
}

int sdfr_decoder_tail_forward_bounds(const float* x, int channels, int in_size, const float* weight,
                                     const float* bias, const float* base, int batch, int R, float* sdf,
                                     long long sdf_stride, int layout, const float* position,
                                     const float* inv_scale, float threshold, sdfr_cell_bounds* bounds,
                                     void* stream) {
  if (int rc = tail_check(channels, in_size, R, batch)) return rc;
  if (layout != SDFR_LAYOUT_DENSE && layout != SDFR_LAYOUT_SKEWED)
    return fail(SDFR_E_FLAGS, "unknown sdf_layout");
  if (!(threshold >= 0.0f)) return fail(SDFR_E_SHAPE, "threshold must be >= 0");
  if (batch == 0) return 0;
  if (!x || !weight || !sdf || !position || !inv_scale || !bounds)
    return fail(SDFR_E_NULL, "decoder tail + bounds: NULL pointer");
  const Grid G = make_grid(R, layout);
  if (sdf_stride < (long long)R * G.px)
    return fail(SDFR_E_SHAPE, "decoder tail: sdf_stride smaller than one grid in this layout");
  CellBounds* out = reinterpret_cast<CellBounds*>(bounds);
  sdfr_bounds_init_kernel<<<batch, 32, 0, (cudaStream_t)stream>>>(position, inv_scale, batch, batch, threshold, out);
  TailParams P;
  memset(&P, 0, sizeof(P));
  P.x = x; P.weight = weight; P.bias = bias; P.base = base;
  P.C = channels; P.S = in_size; P.R = R;
  P.out = sdf; P.out_stride = sdf_stride; P.py = G.py; P.px = G.px;
  P.bounds = out;
  return launch_tail_forward(P, batch, (cudaStream_t)stream);
}

int sdfr_decoder_tail_backward(const float* grad_sdf, long long grad_sdf_stride,
                               const float* n_overlap, const float* upstream,
                               const float* grad_sdf_extra, long long extra_stride,
                               const float* weight, int channels, int in_size, int batch, int R,
                               float* grad_x, void* stream) {
  if (int rc = tail_check(channels, in_size, R, batch)) return rc;
  if (grad_sdf_stride < 0 || extra_stride < 0) return fail(SDFR_E_SHAPE, "negative gradient stride");
  if (batch == 0) return 0;
  if (!grad_sdf || !weight || !grad_x)
    return fail(SDFR_E_NULL, "decoder tail: grad_sdf, weight or grad_x is NULL");
  TailParams P;
  memset(&P, 0, sizeof(P));
  P.weight = weight;
  P.C = channels; P.S = in_size; P.R = R;
  P.g_main = grad_sdf; P.g_main_stride = grad_sdf_stride;
  P.n_overlap = n_overlap; P.upstream = upstream;
  P.g_extra = grad_sdf_extra; P.g_extra_stride = extra_stride;
  P.g_x = grad_x;
  return launch_tail_backward(P, batch, (cudaStream_t)stream);
}

int sdfr_upsample3d_forward(const float* x, int n_volumes, int in_size, int out_size, float* y,
                            void* stream) {
  if (int rc = tail_check(1, in_size, out_size, n_volumes)) return rc;
  if (n_volumes == 0) return 0;
  if (!x || !y) return fail(SDFR_E_NULL, "upsample3d: x or y is NULL");
  TailParams P;
  memset(&P, 0, sizeof(P));
  P.x = x; P.C = 1; P.S = in_size; P.R = out_size;
  P.out = y; P.out_stride = (long long)out_size * out_size * out_size;
  P.py = out_size; P.px = out_size * out_size;
  return launch_tail_forward(P, n_volumes, (cudaStream_t)stream);
}

int sdfr_upsample3d_backward(const float* grad_y, int n_volumes, int in_size, int out_size,
                             float* grad_x, void* stream) {
  if (int rc = tail_check(1, in_size, out_size, n_volumes)) return rc;
  if (n_volumes == 0) return 0;
  if (!grad_y || !grad_x) return fail(SDFR_E_NULL, "upsample3d: grad_y or grad_x is NULL");
  TailParams P;
  memset(&P, 0, sizeof(P));
  P.C = 1; P.S = in_size; P.R = out_size;
  P.g_main = grad_y; P.g_main_stride = (long long)out_size * out_size * out_size;
  P.g_x = grad_x;
  return launch_tail_backward(P, n_volumes, (cudaStream_t)stream);
}

#endif
#if SDFR_IN_PART(4)
static int conv3_check(int batch, int ci, int co, int in_size, int k) {
  if (k != 3) return fail(SDFR_E_SHAPE, "conv3d: only kernel_size 3 is implemented (every reference decoder trunk uses 3)");
  if (batch < 0 || ci < 1 || ci > 4096 || co < 1 || co > 4096)
    return fail(SDFR_E_SHAPE, "conv3d: bad batch or channel count");
  if (in_size < k || in_size > 512) return fail(SDFR_E_SHAPE, "conv3d: in_size must be in [3, 512]");
  return 0;
}

int sdfr_conv3d_forward(const float* x, int batch, int in_channels, int in_size, const float* weight,
                        const float* bias, int out_channels, int kernel_size, int relu, float* y,
                        void* stream) {
  if (int rc = conv3_check(batch, in_channels, out_channels, in_size, kernel_size)) return rc;
  if (out_channels != 4 && out_channels != 8 && out_channels != 16 && out_channels != 32)
    return fail(SDFR_E_SHAPE, "conv3d forward: out_channels must be 4, 8, 16 or 32");
  if (batch == 0) return 0;
  if (!x || !weight || !y) return fail(SDFR_E_NULL, "conv3d: x, weight or y is NULL");
  ConvParams P;
  memset(&P, 0, sizeof(P));
  P.in = x; P.w = weight; P.bias = bias; P.out = y;
  P.CI = in_channels; P.n_in = in_size; P.n_out = in_size - kernel_size + 1; P.relu = relu != 0;
  return launch_conv3<false>(P, out_channels, batch, (cudaStream_t)stream);
}

int sdfr_conv3d_backward_data(const float* grad_y, const float* y, int batch, int in_channels,
                              int in_size, const float* weight, int out_channels, int kernel_size,
                              float* grad_x, void* stream) {
  if (int rc = conv3_check(batch, in_channels, out_channels, in_size, kernel_size)) return rc;
  if (in_channels != 4 && in_channels != 8 && in_channels != 16 && in_channels != 32)
    return fail(SDFR_E_SHAPE, "conv3d backward: in_channels must be 4, 8, 16 or 32");
  if (batch == 0) return 0;
  if (!grad_y || !weight || !grad_x) return fail(SDFR_E_NULL, "conv3d: grad_y, weight or grad_x is NULL");
  ConvParams P;
  memset(&P, 0, sizeof(P));
  P.in = grad_y; P.mask = y; P.w = weight; P.out = grad_x;
  P.CI = out_channels; /* the transposed convolution reads the layer's OUTPUT channels */
  P.n_in = in_size - kernel_size + 1; P.n_out = in_size;
  return launch_conv3<true>(P, in_channels, batch, (cudaStream_t)stream);
}

static int points_check(int n_instances, int width, int height) {
  if (n_instances < 0 || width < 1 || height < 1 || (long long)width * height > (1ll << 30))
    return fail(SDFR_E_SHAPE, "depth to points: n_instances >= 0 and a non-empty image of at most 2^30 pixels expected");
  return 0;
}

int sdfr_depth_to_points_scratch(int n_instances, int width, int height, long long* bytes) {
  if (int rc = points_check(n_instances, width, height)) return rc;
  if (!bytes) return fail(SDFR_E_NULL, "depth to points scratch: bytes is NULL");
  const long long n_tiles = ((long long)width * height + kPtsTile - 1) / kPtsTile;
  *bytes = (long long)sizeof(int) * n_instances * n_tiles;
  return 0;
}

int sdfr_depth_to_points(const float* depth, long long depth_stride, const unsigned char* mask, int n_instances,
                         int width, int height, float far_field, float fx, float fy, float cx, float cy,
                         float* masked_depth, float* points, int capacity, long long* counts, void* scratch,
                         void* stream) {
  if (int rc = points_check(n_instances, width, height)) return rc;
  if (depth_stride < 0 || capacity < 0) return fail(SDFR_E_SHAPE, "depth to points: depth_stride >= 0 and capacity >= 0 expected");
  if (n_instances == 0) return 0;
  if (!depth || !counts || !scratch) return fail(SDFR_E_NULL, "depth to points: depth, counts or scratch is NULL");
  if (!points && capacity > 0) return fail(SDFR_E_NULL, "depth to points: points is NULL but capacity > 0");
  ExtractParams P;
  memset(&P, 0, sizeof(P));
  P.depth = depth; P.depth_stride = depth_stride; P.mask = mask; P.far_field = far_field;
  /* torch's CUDA division of a tensor by a Python scalar multiplies by the reciprocal rounded to fp32 */
  P.cx = cx; P.cy = cy; P.inv_fx = 1.0f / fx; P.inv_fy = 1.0f / fy;
  P.width = width; P.n_pixels = width * height; P.n_tiles = (P.n_pixels + kPtsTile - 1) / kPtsTile;
  P.capacity = capacity; P.masked_depth = masked_depth; P.points = capacity > 0 ? points : nullptr;
  P.counts = counts; P.tile_offsets = static_cast<int*>(scratch);
  return launch_depth_to_points(P, n_instances, (cudaStream_t)stream);
}

#endif
}  // extern "C"
