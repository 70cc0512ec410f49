/*
 * sdfr_points.cuh -- point-cloud loss of the render-and-compare loop as sm_100a kernels.
 * Included by sdfrender.cu inside its anonymous namespace (one translation unit, shared error
 * state and launch helpers).
 *
 * Replaces, batched over hypotheses and without host synchronisation, the caller-side helper
 *   sdfest/estimation/losses.py:32-135   pc_loss(points, position, orientation, scale, sdf)
 * as it is used by estimation/simple_setup.py:134-144:  loss_pc = mean_m | pc_loss(...)[m] |.
 * Per hypothesis b and observed point p_m (camera frame):
 *   q   = orientation_b / |orientation_b|                      (losses.py:56, "to get
 *                                                                normalization gradients")
 *   x   = Rm(q) (p_m - position_b) / scale_b                   (losses.py:57-81; Rm = R(q)^T)
 *   c   = floor((x + 1)(R - 1)/2); outside if any c < 0 or c > R-2; c clipped to [0, R-2]
 *   u   = (x - (c h - 1)) / h,  h = 2/(R-1)                     (losses.py:84-104)
 *   val = outside ? 0 : trilerp(sdf_b, c, u) * scale_b          (losses.py:107-135)
 * forward:  loss_sum[b] += sum_m |val|      (the caller divides by the number of points)
 * backward: gradients of  sum_b upstream[b] * loss_sum[b]  w.r.t. sdf (true trilinear weights),
 *           position, the UN-normalised orientation, and scale -- recomputing the interpolation
 *           instead of saving per-point state (M x B x 12 floats).
 *
 * The same 8-corner gather as the renderer (sdfr_core.cuh gather<>), either SDF layout.  Pose
 * gradients: registers -> warp shuffle -> shared -> <= 8 atomics per CTA; SDF gradients:
 * fire-and-forget RED.ADD.F32.
 */
#ifndef SDFR_POINTS_CUH_
#define SDFR_POINTS_CUH_

struct PointParams {
  const float* __restrict__ points;  // [M,3] (or [B,M,3] with points_stride = 3M)
  long long points_stride;
  int n_points;
  const float* __restrict__ sdf;
  long long sdf_stride;
  Grid grid;
  const float* __restrict__ position;     // [B,3]
  const float* __restrict__ orientation;  // [B,4] x,y,z,w, any non-zero length
  const float* __restrict__ scale;        // [B]
  float* __restrict__ loss_sum;           // [B]  (forward)
  const float* __restrict__ upstream;     // [B] or NULL (= 1)  (backward)
  float* __restrict__ grad_sdf;
  long long grad_sdf_stride;
  float* __restrict__ grad_position;
  float* __restrict__ grad_orientation;
  float* __restrict__ grad_scale;
  unsigned flags;
  int z_offset;
};

template <bool BACKWARD, bool WANT_SDF, bool WANT_POSE, bool WITH_LOSS = false>
__global__ void __launch_bounds__(256)
sdfr_point_loss_kernel(const __grid_constant__ PointParams P) {
  __shared__ float red[8][9];
  const int b = blockIdx.y + P.z_offset;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Grid& G = P.grid;

  /* per-hypothesis constants, in registers of every thread */
  const float o0 = __ldg(P.orientation + 4 * b + 0), o1 = __ldg(P.orientation + 4 * b + 1);
  const float o2 = __ldg(P.orientation + 4 * b + 2), o3 = __ldg(P.orientation + 4 * b + 3);
  const float qn = sqrtf(o0 * o0 + o1 * o1 + o2 * o2 + o3 * o3);
  const float qx = o0 / qn, qy = o1 / qn, qz = o2 / qn, qw = o3 / qn;
  /* losses.py:61-75 (rotation of the conjugate: camera -> object) */
  const float r00 = 1 - 2 * (qy * qy + qz * qz), r01 = 2 * (qx * qy + qz * qw), r02 = 2 * (qx * qz - qw * qy);
  const float r10 = 2 * (qx * qy - qz * qw), r11 = 1 - 2 * (qx * qx + qz * qz), r12 = 2 * (qy * qz + qw * qx);
  const float r20 = 2 * (qx * qz + qw * qy), r21 = 2 * (qy * qz - qw * qx), r22 = 1 - 2 * (qx * qx + qy * qy);
  const float tx = __ldg(P.position + 3 * b + 0), ty = __ldg(P.position + 3 * b + 1);
  const float tz = __ldg(P.position + 3 * b + 2);
  const float s = __ldg(P.scale + b);
  /* one reciprocal per hypothesis instead of nine IEEE divisions per point (1 ulp per quotient;
   * the reference evaluates obj / scale and offsets / grid_size in torch, losses.py:81, 104) */
  const float rs = 1.0f / s, rh = 1.0f / G.h;
  const float up = BACKWARD ? (P.upstream ? __ldg(P.upstream + b) : 1.0f) : 0.0f;
  const float* __restrict__ pts = P.points + (size_t)b * P.points_stride;
  const float* __restrict__ grid = P.sdf + (size_t)b * P.sdf_stride;
  float* __restrict__ gsdf = (BACKWARD && WANT_SDF) ? P.grad_sdf + (size_t)b * P.grad_sdf_stride : nullptr;
  const float half_rm1 = G.Rm1f * 0.5f;
  const float rm2f = (float)G.Rm2;

  float acc[9]; /* forward: [0] = sum |val|;  backward: g_t (3), g_q (4), g_s (1), [8] = sum |val| (WITH_LOSS) */
#pragma unroll
  for (int i = 0; i < 9; ++i) acc[i] = 0.0f;

  /* The trip count is uniform over the CTA so that all 32 lanes reach the warp-aggregated scatter:
   * observed points come in scan order, neighbouring lanes mostly fall into the same grid cell, and
   * their 8 corner contributions merge inside the warp before any RED is issued (sdfrender.cu
   * scatter_sdf_warp; the first version issued 8 REDs per point, 76 us for 64 x 20 k points). */
  for (int m0 = blockIdx.x * blockDim.x; m0 < P.n_points; m0 += gridDim.x * blockDim.x) {
    const int m = m0 + threadIdx.x;
    bool has = false;
    PixelGrad pg;
    pg.base = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) pg.w[i] = 0.0f;
    if (m < P.n_points) {
      const float dx = __ldg(pts + 3 * m + 0) - tx, dy = __ldg(pts + 3 * m + 1) - ty;
      const float dz = __ldg(pts + 3 * m + 2) - tz;
      const float x0 = (r00 * dx + r01 * dy + r02 * dz) * rs;
      const float x1 = (r10 * dx + r11 * dy + r12 * dz) * rs;
      const float x2 = (r20 * dx + r21 * dy + r22 * dz) * rs;
      const float f0 = floorf((x0 + 1.0f) * half_rm1), f1 = floorf((x1 + 1.0f) * half_rm1);
      const float f2 = floorf((x2 + 1.0f) * half_rm1);
      const bool outside = fminf(f0, fminf(f1, f2)) < 0.0f || fmaxf(f0, fmaxf(f1, f2)) > rm2f;
      if (!(outside || !(f0 == f0) || !(f1 == f1) || !(f2 == f2))) { /* else contributes 0 */
        const int ix = (int)f0, iy = (int)f1, iz = (int)f2;
        const float u0 = (x0 - (f0 * G.h - 1.0f)) * rh, u1 = (x1 - (f1 * G.h - 1.0f)) * rh;
        const float u2 = (x2 - (f2 * G.h - 1.0f)) * rh;
        const Corners k = gather<0>(grid, G, ix, iy, iz);
        /* losses.py:107-131: x first, then y, then z */
        const float a0 = k.c000 * (1 - u0) + k.c100 * u0; /* y0 z0 */
        const float a2 = k.c010 * (1 - u0) + k.c110 * u0; /* y1 z0 */
        const float a1 = k.c001 * (1 - u0) + k.c101 * u0; /* y0 z1 */
        const float a3 = k.c011 * (1 - u0) + k.c111 * u0; /* y1 z1 */
        const float b0 = a0 * (1 - u1) + a2 * u1, b1 = a1 * (1 - u1) + a3 * u1;
        const float v = b0 * (1 - u2) + b1 * u2;
        const float val = v * s;
        if (!BACKWARD) acc[0] += fabsf(val);
        if (WITH_LOSS) acc[8] += fabsf(val);
        if (BACKWARD && val != 0.0f) { /* d|.|/d. = 0 at 0, as torch.abs */
          const float g = val > 0.0f ? up : -up; /* d L / d val */
          if (WANT_SDF) {
            const float gs_ = g * s;
            const float wx0 = (1 - u0) * gs_, wx1 = u0 * gs_;
            has = true;
            pg.base = (ix * G.R + iy) * G.R + iz;
            pg.w[0] = wx0 * (1 - u1) * (1 - u2);
            pg.w[1] = wx0 * (1 - u1) * u2;
            pg.w[2] = wx0 * u1 * (1 - u2);
            pg.w[3] = wx0 * u1 * u2;
            pg.w[4] = wx1 * (1 - u1) * (1 - u2);
            pg.w[5] = wx1 * (1 - u1) * u2;
            pg.w[6] = wx1 * u1 * (1 - u2);
            pg.w[7] = wx1 * u1 * u2;
          }
          if (WANT_POSE) {
            const float dv0 = ((k.c100 - k.c000) * (1 - u1) + (k.c110 - k.c010) * u1) * (1 - u2) +
                              ((k.c101 - k.c001) * (1 - u1) + (k.c111 - k.c011) * u1) * u2;
            const float dv1 = (a2 - a0) * (1 - u2) + (a3 - a1) * u2;
            const float dv2 = b1 - b0;
            /* dL/dx = g * s * dv/du / h ;  x = Rm d / s */
            const float c0 = g * s * rh;
            const float gx0 = c0 * dv0, gx1 = c0 * dv1, gx2 = c0 * dv2;
            const float gy0 = gx0 * rs, gy1 = gx1 * rs, gy2 = gx2 * rs; /* dL/d(Rm d) */
            /* position: d = p - t */
            acc[0] -= r00 * gy0 + r10 * gy1 + r20 * gy2;
            acc[1] -= r01 * gy0 + r11 * gy1 + r21 * gy2;
            acc[2] -= r02 * gy0 + r12 * gy1 + r22 * gy2;
            /* scale: val = v s, dx/ds = -x/s */
            acc[7] += g * v - (gx0 * x0 + gx1 * x1 + gx2 * x2) * rs;
            /* unit quaternion: dL/dq_k = gy . (dRm/dq_k d) */
            acc[3] += gy0 * (2 * qy * dy + 2 * qz * dz) + gy1 * (2 * qy * dx - 4 * qx * dy + 2 * qw * dz) +
                      gy2 * (2 * qz * dx - 2 * qw * dy - 4 * qx * dz);
            acc[4] += gy0 * (-4 * qy * dx + 2 * qx * dy - 2 * qw * dz) + gy1 * (2 * qx * dx + 2 * qz * dz) +
                      gy2 * (2 * qw * dx + 2 * qz * dy - 4 * qy * dz);
            acc[5] += gy0 * (-4 * qz * dx + 2 * qw * dy + 2 * qx * dz) +
                      gy1 * (-2 * qw * dx - 4 * qz * dy + 2 * qy * dz) + gy2 * (2 * qx * dx + 2 * qy * dy);
            acc[6] += gy0 * (2 * qz * dy - 2 * qy * dz) + gy1 * (-2 * qz * dx + 2 * qx * dz) +
                      gy2 * (2 * qy * dx - 2 * qx * dy);
          }
        }
      }
    }
    if (BACKWARD && WANT_SDF) scatter_sdf_warp<0>(gsdf, G, pg.base, pg.w, has, lane);
  }

  /* CTA reduction: one value (forward) or eight (backward) */
  constexpr int NV = BACKWARD ? (WITH_LOSS ? 9 : 8) : 1;
  if constexpr (!BACKWARD || WANT_POSE || WITH_LOSS) {
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = warp_sum(acc[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) red[warp][i] = acc[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t[9];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float v = 0.0f;
      for (int w = 0; w < 8; ++w) v += red[w][i];
      t[i] = v;
    }
    if (!BACKWARD) {
      if (t[0] != 0.0f) atomicAdd(P.loss_sum + b, t[0]);
    } else {
      if (WITH_LOSS && t[8] != 0.0f)
        atomicAdd(P.loss_sum + b, (P.flags & SDFR_LOSS_WEIGHTED) ? up * t[8] : t[8]);
      if (P.flags & SDFR_GRAD_POSITION) {
        if (t[0] != 0.0f) atomicAdd(P.grad_position + 3 * b + 0, t[0]);
        if (t[1] != 0.0f) atomicAdd(P.grad_position + 3 * b + 1, t[1]);
        if (t[2] != 0.0f) atomicAdd(P.grad_position + 3 * b + 2, t[2]);
      }
      if (P.flags & SDFR_GRAD_ORIENTATION) {
        /* through q = o/|o|:  dL/do = (g - q (q.g)) / |o|   (linear, applied to the CTA sum) */
        const float dot = qx * t[3] + qy * t[4] + qz * t[5] + qw * t[6];
        const float g0 = (t[3] - qx * dot) / qn, g1 = (t[4] - qy * dot) / qn;
        const float g2 = (t[5] - qz * dot) / qn, g3 = (t[6] - qw * dot) / qn;
        if (g0 != 0.0f) atomicAdd(P.grad_orientation + 4 * b + 0, g0);
        if (g1 != 0.0f) atomicAdd(P.grad_orientation + 4 * b + 1, g1);
        if (g2 != 0.0f) atomicAdd(P.grad_orientation + 4 * b + 2, g2);
        if (g3 != 0.0f) atomicAdd(P.grad_orientation + 4 * b + 3, g3);
      }
      if ((P.flags & SDFR_GRAD_INV_SCALE) && t[7] != 0.0f) atomicAdd(P.grad_scale + b, t[7]);
    }
  }
  }
}

template <bool BACKWARD, bool WITH_LOSS = false>
int launch_point_loss(PointParams P, int batch, cudaStream_t s) {
  /* ~4 points per thread: the per-thread prologue (rotation matrix, reciprocals) and the CTA
   * reduction of the eight pose gradients cost about half as much as one point */
  int gx = (P.n_points + 1023) / 1024;
  if ((long)gx * batch < 592) gx = (P.n_points + 255) / 256; /* few hypotheses: keep the SMs busy */
  gx = gx < 1 ? 1 : (gx > 512 ? 512 : gx);
  const bool want_sdf = (P.flags & SDFR_GRAD_SDF) != 0;
  const bool want_pose =
      (P.flags & (SDFR_GRAD_POSITION | SDFR_GRAD_ORIENTATION | SDFR_GRAD_INV_SCALE)) != 0;
  if (BACKWARD && !WITH_LOSS && !want_sdf && !want_pose) return 0;
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid(gx, batch - z0 < 65535 ? batch - z0 : 65535);
    if (!BACKWARD || (!want_sdf && !want_pose))
      sdfr_point_loss_kernel<false, false, false><<<grid, 256, 0, s>>>(P);
    else if (want_sdf && want_pose)
      sdfr_point_loss_kernel<true, true, true, WITH_LOSS><<<grid, 256, 0, s>>>(P);
    else if (want_sdf)
      sdfr_point_loss_kernel<true, true, false, WITH_LOSS><<<grid, 256, 0, s>>>(P);
    else
      sdfr_point_loss_kernel<true, false, true, WITH_LOSS><<<grid, 256, 0, s>>>(P);
  }
  return check_launch("sdfr_point_loss_kernel");
}

/*
 * Observed point clouds of K object instances (sdfr_depth_to_points): an ordered compaction of the
 * selected pixels of every instance, in row-major pixel order (the order of torch.nonzero), so that the
 * clouds are the ones losses.depth_to_pointcloud builds, bit for bit.
 *   1. sdfr_points_count_kernel: per (instance, tile of kPtsTile pixels) the number of selected pixels
 *      (and the masked depth, when asked for);
 *   2. sdfr_points_scan_kernel: one CTA per instance scans its tile counts into tile offsets (exclusive)
 *      and writes the instance's true count;
 *   3. sdfr_points_write_kernel: each tile is selected again, a CTA prefix sum gives every selected
 *      pixel its row, and rows below the capacity are written; extra CTAs fill rows [count, capacity)
 *      with the padding coordinate.
 * Each thread owns kPtsPerThread consecutive pixels, so thread order is pixel order.
 */
constexpr int kPtsThreads = 256;
constexpr int kPtsPerThread = 4;
constexpr int kPtsTile = kPtsThreads * kPtsPerThread;
constexpr float kPadCoordinate = 1.0e6f; /* losses.PAD_COORDINATE */

struct ExtractParams {
  const float* __restrict__ depth;  // [H,W] (depth_stride 0) or [K,H,W]
  long long depth_stride;
  const unsigned char* __restrict__ mask;  // [K,H,W] or NULL (= depth != 0)
  float far_field;
  float cx, cy, inv_fx, inv_fy;
  int width, n_pixels, n_tiles, capacity;
  float* __restrict__ masked_depth;  // [K,H,W] or NULL
  float* __restrict__ points;        // [K,capacity,3]
  long long* __restrict__ counts;    // [K]
  int* __restrict__ tile_offsets;    // [K,n_tiles] scratch: tile counts, then exclusive offsets
  int z_offset;
};

/* The masked depth of this thread's pixels (as SDFPipeline._preprocess_depth: 0 outside the mask and
 * beyond the far field) and a bit per selected pixel (masked depth != 0; NaN is selected, as by
 * torch.nonzero). */
__device__ __forceinline__ unsigned select_pixels(const ExtractParams& P, int k, int p0, float v[kPtsPerThread]) {
  const float* __restrict__ d = P.depth + (size_t)k * P.depth_stride;
  const unsigned char* __restrict__ m = P.mask ? P.mask + (size_t)k * P.n_pixels : nullptr;
  unsigned bits = 0;
#pragma unroll
  for (int i = 0; i < kPtsPerThread; ++i) {
    const int p = p0 + i;
    float x = 0.0f;
    if (p < P.n_pixels) {
      x = __ldg(d + p);
      if (m && !__ldg(m + p)) x = 0.0f;
      if (x > P.far_field) x = 0.0f;
    }
    v[i] = x;
    if (x != 0.0f) bits |= 1u << i;
  }
  return bits;
}

/* exclusive prefix of `x` over the CTA's threads, and the CTA total */
__device__ __forceinline__ int cta_exclusive_scan(int x, int* total) {
  __shared__ int warp_tot[kPtsThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < kPtsThreads / 32; ++w) {
    const int t = warp_tot[w];
    before += w < warp ? t : 0;
    all += t;
  }
  __syncthreads(); /* warp_tot may be reused by the caller's next scan */
  *total = all;
  return before + incl - x;
}

__global__ void __launch_bounds__(kPtsThreads) sdfr_points_count_kernel(const __grid_constant__ ExtractParams P) {
  const int k = blockIdx.y + P.z_offset;
  const int p0 = blockIdx.x * kPtsTile + threadIdx.x * kPtsPerThread;
  float v[kPtsPerThread];
  const unsigned bits = select_pixels(P, k, p0, v);
  if (P.masked_depth) {
    float* __restrict__ out = P.masked_depth + (size_t)k * P.n_pixels;
#pragma unroll
    for (int i = 0; i < kPtsPerThread; ++i)
      if (p0 + i < P.n_pixels) out[p0 + i] = v[i];
  }
  int total;
  cta_exclusive_scan(__popc(bits), &total);
  if (threadIdx.x == 0) P.tile_offsets[(size_t)k * P.n_tiles + blockIdx.x] = total;
}

/* one CTA per instance: tile counts -> exclusive tile offsets, counts[k] = the instance's total */
__global__ void __launch_bounds__(kPtsThreads) sdfr_points_scan_kernel(const __grid_constant__ ExtractParams P) {
  const int k = blockIdx.x;
  int* __restrict__ t = P.tile_offsets + (size_t)k * P.n_tiles;
  int carry = 0;
  for (int i0 = 0; i0 < P.n_tiles; i0 += kPtsThreads) {
    const int i = i0 + threadIdx.x;
    const int c = i < P.n_tiles ? t[i] : 0;
    int total;
    const int before = cta_exclusive_scan(c, &total);
    if (i < P.n_tiles) t[i] = carry + before;
    carry += total;
  }
  if (threadIdx.x == 0) P.counts[k] = carry;
}

__global__ void __launch_bounds__(kPtsThreads) sdfr_points_write_kernel(const __grid_constant__ ExtractParams P) {
  const int k = blockIdx.y + P.z_offset;
  float* __restrict__ out = P.points + (size_t)k * P.capacity * 3;
  if ((int)blockIdx.x >= P.n_tiles) { /* padding rows [count, capacity) */
    const long long n = P.counts[k];
    const int r = ((int)blockIdx.x - P.n_tiles) * kPtsThreads + threadIdx.x;
    if (r < P.capacity && r >= n) {
      out[3 * (size_t)r + 0] = kPadCoordinate;
      out[3 * (size_t)r + 1] = kPadCoordinate;
      out[3 * (size_t)r + 2] = kPadCoordinate;
    }
    return;
  }
  const int p0 = blockIdx.x * kPtsTile + threadIdx.x * kPtsPerThread;
  float v[kPtsPerThread];
  const unsigned bits = select_pixels(P, k, p0, v);
  int total;
  int row = P.tile_offsets[(size_t)k * P.n_tiles + blockIdx.x] + cta_exclusive_scan(__popc(bits), &total);
#pragma unroll
  for (int i = 0; i < kPtsPerThread; ++i) {
    if (!(bits & (1u << i))) continue;
    if (row < P.capacity) {
      /* losses.depth_to_pointcloud: torch evaluates (col - cx) * z / fx with the division by a Python
       * scalar as a multiplication by its fp32 reciprocal; explicit roundings keep nvcc from contracting */
      const int p = p0 + i;
      const int r = p / P.width, c = p - r * P.width;
      const float z = v[i];
      out[3 * (size_t)row + 0] = __fmul_rn(__fmul_rn(__fsub_rn((float)c, P.cx), z), P.inv_fx);
      out[3 * (size_t)row + 1] = __fmul_rn(__fmul_rn(-__fsub_rn((float)r, P.cy), z), P.inv_fy);
      out[3 * (size_t)row + 2] = -z;
    }
    ++row;
  }
}

int launch_depth_to_points(ExtractParams P, int n_instances, cudaStream_t s) {
  const int n_pad = P.points ? (P.capacity + kPtsThreads - 1) / kPtsThreads : 0;
  for (int z0 = 0; z0 < n_instances; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid(P.n_tiles, n_instances - z0 < 65535 ? n_instances - z0 : 65535);
    sdfr_points_count_kernel<<<grid, kPtsThreads, 0, s>>>(P);
  }
  P.z_offset = 0;
  sdfr_points_scan_kernel<<<n_instances, kPtsThreads, 0, s>>>(P);
  if (P.points) {
    for (int z0 = 0; z0 < n_instances; z0 += 65535) {
      P.z_offset = z0;
      const dim3 grid(P.n_tiles + n_pad, n_instances - z0 < 65535 ? n_instances - z0 : 65535);
      sdfr_points_write_kernel<<<grid, kPtsThreads, 0, s>>>(P);
    }
  }
  return check_launch("sdfr_depth_to_points");
}

#endif /* SDFR_POINTS_CUH_ */
