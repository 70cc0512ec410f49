/*
 * sdfr_core.cuh -- per-ray arithmetic of the SDF depth renderer (forward sphere trace and
 * analytic backward), shared by every kernel in sdfrender.cu.
 *
 * The arithmetic deliberately keeps the operation order and the float/double mixing of the
 * reference kernels (sdfest/differentiable_renderer/csrc/sdf_renderer_cuda.cu, cited as cu:NNN)
 * so that depth agrees to rounding and sphere-trace termination does not flip; what is NOT
 * kept is the reference's structure: per-hypothesis constants are hoisted into a Frame built
 * once per CTA, voxel indices are 32-bit, the resolution is a run-time value, ray directions
 * come from per-CTA tables, and nothing here touches global memory except the 8 grid gathers.
 *
 * Everything is SDFR_HD (= __host__ __device__ under nvcc) so that tests/host_emul can compile
 * the very same functions with g++ and check them against the oracle without a GPU.  The
 * product never runs the host instantiation.
 */
#ifndef SDFR_CORE_CUH_
#define SDFR_CORE_CUH_

#if defined(__CUDACC__)
#define SDFR_HD __host__ __device__ __forceinline__
#define SDFR_HDC __host__ __device__ constexpr
#else
#define SDFR_HD static inline
#define SDFR_HDC constexpr
#endif

#if defined(__CUDA_ARCH__)
#define SDFR_LDG(p) __ldg(p)
#define SDFR_RSQRT(x) rsqrtf(x)
#define SDFR_FLOOR_TO_INT(x) __float2int_rd(x)
/* individually rounded products / sums: nvcc may not contract these into fma (see frame_pose) */
#define SDFR_MUL(a, b) __fmul_rn((a), (b))
#define SDFR_ADD(a, b) __fadd_rn((a), (b))
#define SDFR_SUB(a, b) __fsub_rn((a), (b))
/* slab quotients: MUFU.RCP + FMUL (2 ulp) instead of the IEEE division sequence (~9 instructions and
 * a slow-path branch, six times per pixel = 7 % of the fused kernel's instructions); |f| <= 1 here, far
 * from __fdividef's 2^126 caveat. */
#define SDFR_SLAB_DIV(a, b) __fdividef((a), (b))
#else
#include <math.h>
#define SDFR_LDG(p) (*(p))
#define SDFR_RSQRT(x) (1.0f / sqrtf(x))
#define SDFR_FLOOR_TO_INT(x) ((int)floorf(x))
#define SDFR_SLAB_DIV(a, b) ((a) / (b))
/* host emulation: a volatile temporary keeps the compiler from contracting under any -ffp-contract */
static inline float sdfr_nc_mul(float a, float b) { volatile float r = a * b; return r; }
static inline float sdfr_nc_add(float a, float b) { volatile float r = a + b; return r; }
static inline float sdfr_nc_sub(float a, float b) { volatile float r = a - b; return r; }
#define SDFR_MUL(a, b) sdfr_nc_mul((a), (b))
#define SDFR_ADD(a, b) sdfr_nc_add((a), (b))
#define SDFR_SUB(a, b) sdfr_nc_sub((a), (b))
#endif

namespace sdfr {

/* sphere-tracing step cap; the reference loop is unbounded (cu:283-293, SURVEY Q5) */
constexpr int kMaxSteps = 4096;

/* Per-grid constants.  h / hinv_fwd / hinv_bwd reproduce cu:229 (2.0/(R-1) narrowed),
 * cu:230 ((R-1)/2.0 narrowed) and cu:327-328 (1./float(2.0/(R-1)) narrowed). */
struct Grid {
  int R, R2, Rm2;
  int py, px; /* element pitch of the SDF array between consecutive y / consecutive x */
  int layout;
  float Rm1f, h, hinv_fwd, hinv_bwd;
};

/*
 * SDF array layouts.  DENSE is the reference's [R][R][R] (z contiguous, cu:13).  SKEWED is a
 * pitched copy, element (x,y,z) at x*pitch_x + y*pitch_y + z with pitch_y = 3, pitch_x = 9
 * (mod 32): the 32 lanes of a warp gather voxels a few cells apart in x and y, which in the dense
 * layout (pitches = 0 mod 32 for R = 32, 64, 128) all sit in the SAME L1 bank and serialise --
 * measured 6 cycles per warp-level load for 6 rows against 2 when the banks differ
 * (scripts/micro/l1_gather.cu, profiles/r01_l1_gather.txt).  With (3, 9) two voxels share a bank
 * only if they are at least (1,3,0) cells apart.
 */
constexpr int kLayoutDense = 0;
constexpr int kLayoutSkewed = 1;

SDFR_HDC int skew_pitch_y(int R) { return R + (((3 - R % 32) + 32) % 32); }
SDFR_HDC int skew_pitch_x(int R) {
  return R * skew_pitch_y(R) + (((9 - (R * skew_pitch_y(R)) % 32) + 32) % 32);
}

SDFR_HD Grid make_grid(int R, int layout = kLayoutDense) {
  Grid G;
  G.R = R;
  G.R2 = R * R;
  G.Rm2 = R - 2;
  G.py = layout == kLayoutSkewed ? skew_pitch_y(R) : R;
  G.px = layout == kLayoutSkewed ? skew_pitch_x(R) : R * R;
  G.layout = layout;
  G.Rm1f = (float)(R - 1);
  G.h = (float)(2.0 / (double)(R - 1));
  G.hinv_fwd = (float)((double)(R - 1) / 2.0);
  G.hinv_bwd = (float)(1.0 / (double)G.h);
  return G;
}

struct Camera {
  int W, H;
  float cx, cy, fx, fy;
};

/* Per-hypothesis constants, built once per CTA. */
struct Frame {
  float r00, r01, r02, r10, r11, r12, r20, r21, r22; /* rotation of q, object -> camera */
  float px, py, pz;                                  /* position */
  float qx, qy, qz, qw;
  float ox, oy, oz;       /* camera centre in the object frame: R^T (0 - p)   (cu:279-281) */
  float e0, e1, e2;       /* box axes . position                               (cu:173)    */
  float inv_scale, scale; /* scale = (float)(1. / inv_scale), a double divide  (cu:259)    */
  int x0, y0, x1, y1;     /* conservative pixel rectangle of the projected box [x0,x1)x[y0,y1) */
  /* Culling box in the object frame (metric units): no ray that misses [blo, bhi] can hit the surface.
   * Without grid bounds it is the reference's box [-scale, scale]^3 (cu:156-194); with the cell bounds
   * of sdfr_grid_bounds it is the part of the grid where the field can fall below the hit threshold.
   * It only decides WHETHER a ray is traced -- the march itself always starts at the reference's box
   * entry, so every traced ray takes the reference's samples. */
  float blo0, blo1, blo2, bhi0, bhi1, bhi2;
};

/* Cell bounds of one grid as sdfr_grid_bounds writes them: first / last cell index per axis whose
 * smallest corner value is below tau, and tau itself.  lo > hi: no such cell, nothing can be hit. */
struct CellBounds {
  int lo[3], hi[3];
  float tau;
  int pad;
};

/* Hit-threshold bound of a hypothesis: a sample can only terminate the march (cu:286, dist <
 * threshold * t with dist = trilinear * scale) where trilinear < threshold * t / scale, and t never
 * exceeds |p| + sqrt(3) scale inside the box; the trilinear value of a cell is never below its
 * smallest corner.  The factor and the offset absorb the rounding of both sides. */
SDFR_HD float hit_tau(const float* pos, float inv_scale, float threshold) {
  /* individually rounded operations: the value is compared for equality / order between the bounds
   * pass, the render kernels and the test oracle (oracle/grid_bounds.py) */
  const float scale = (float)(1. / (double)inv_scale);
  const float n2 = SDFR_ADD(SDFR_ADD(SDFR_MUL(pos[0], pos[0]), SDFR_MUL(pos[1], pos[1])), SDFR_MUL(pos[2], pos[2]));
  const float far = SDFR_ADD(sqrtf(n2), SDFR_MUL(1.7320509f, scale));
  return SDFR_ADD(SDFR_MUL(SDFR_MUL(SDFR_MUL(threshold, far), inv_scale), 1.001f), 1e-5f);
}

/* Rotation entries, position, scale, culling box (everything of Frame except the rectangle).
 * `bounds` (or NULL) are the grid's cell bounds; they are used only when they were computed for a
 * threshold bound at least as large as this hypothesis' (else the reference's box is kept). */
SDFR_HD void frame_pose(Frame& F, const float* pos, const float* quat, const float* inv_scale,
                        const CellBounds* bounds = nullptr, int R = 0, float threshold = 0.0f) {
  const float x = quat[0], y = quat[1], z = quat[2], w = quat[3];
  F.qx = x; F.qy = y; F.qz = z; F.qw = w;
  /* cu:112-121.  Every product and sum is rounded on its own (SDFR_MUL / SDFR_ADD / SDFR_SUB): when
   * nvcc contracts these expressions into fma, the two products of an entry are rounded differently,
   * the matrix drifts from a rotation by ~1 ulp, and so does the object-frame origin R^T(-p) -- an
   * offset common to ALL pixels that the quaternion gradient amplifies by |p| inv_scale (R-1)/2: 1.8 %
   * of the orientation gradient of an object 1.2 m away at 128^3 (host emulation with and without
   * -ffp-contract, DESIGN.md section 2).  Individually rounded, the result stays within 2e-5 of the
   * float64 evaluation; it costs ~60 instructions once per CTA. */
  const float xx = SDFR_MUL(x, x), yy = SDFR_MUL(y, y), zz = SDFR_MUL(z, z);
  const float xy = SDFR_MUL(x, y), xz = SDFR_MUL(x, z), yz = SDFR_MUL(y, z);
  const float wx = SDFR_MUL(w, x), wy = SDFR_MUL(w, y), wz = SDFR_MUL(w, z);
  F.r00 = SDFR_SUB(1.0f, SDFR_MUL(2.0f, SDFR_ADD(yy, zz)));
  F.r01 = SDFR_MUL(2.0f, SDFR_SUB(xy, wz));
  F.r02 = SDFR_MUL(2.0f, SDFR_ADD(xz, wy));
  F.r10 = SDFR_MUL(2.0f, SDFR_ADD(xy, wz));
  F.r11 = SDFR_SUB(1.0f, SDFR_MUL(2.0f, SDFR_ADD(xx, zz)));
  F.r12 = SDFR_MUL(2.0f, SDFR_SUB(yz, wx));
  F.r20 = SDFR_MUL(2.0f, SDFR_SUB(xz, wy));
  F.r21 = SDFR_MUL(2.0f, SDFR_ADD(yz, wx));
  F.r22 = SDFR_SUB(1.0f, SDFR_MUL(2.0f, SDFR_ADD(xx, yy)));
  F.px = pos[0]; F.py = pos[1]; F.pz = pos[2];
  F.inv_scale = inv_scale[0];
  F.scale = (float)(1. / (double)F.inv_scale);
  const float nx = 0.0f - F.px, ny = 0.0f - F.py, nz = 0.0f - F.pz;
  /* conjugate quaternion = transposed matrix */
  F.ox = SDFR_ADD(SDFR_ADD(SDFR_MUL(F.r00, nx), SDFR_MUL(F.r10, ny)), SDFR_MUL(F.r20, nz));
  F.oy = SDFR_ADD(SDFR_ADD(SDFR_MUL(F.r01, nx), SDFR_MUL(F.r11, ny)), SDFR_MUL(F.r21, nz));
  F.oz = SDFR_ADD(SDFR_ADD(SDFR_MUL(F.r02, nx), SDFR_MUL(F.r12, ny)), SDFR_MUL(F.r22, nz));
  F.e0 = SDFR_ADD(SDFR_ADD(SDFR_MUL(F.r00, F.px), SDFR_MUL(F.r10, F.py)), SDFR_MUL(F.r20, F.pz));
  F.e1 = SDFR_ADD(SDFR_ADD(SDFR_MUL(F.r01, F.px), SDFR_MUL(F.r11, F.py)), SDFR_MUL(F.r21, F.pz));
  F.e2 = SDFR_ADD(SDFR_ADD(SDFR_MUL(F.r02, F.px), SDFR_MUL(F.r12, F.py)), SDFR_MUL(F.r22, F.pz));
  F.blo0 = F.blo1 = F.blo2 = -F.scale;
  F.bhi0 = F.bhi1 = F.bhi2 = F.scale;
  if (bounds != nullptr && R >= 2 && hit_tau(pos, F.inv_scale, threshold) <= bounds->tau) {
    /* cell i spans [i h - 1, (i + 1) h - 1]; one cell of margin on either side covers the rounding of
     * the cell lookup and of the slab quotients */
    const float h = 2.0f / (float)(R - 1);
    float lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (bounds->lo[a] > bounds->hi[a]) { /* empty: a box no ray can enter */
        lo[a] = 2.0f; hi[a] = -2.0f;
      } else {
        lo[a] = fmaxf(-1.0f, (float)(bounds->lo[a] - 1) * h - 1.0f);
        hi[a] = fminf(1.0f, (float)(bounds->hi[a] + 2) * h - 1.0f);
      }
    }
    F.blo0 = lo[0] * F.scale; F.blo1 = lo[1] * F.scale; F.blo2 = lo[2] * F.scale;
    F.bhi0 = hi[0] * F.scale; F.bhi1 = hi[1] * F.scale; F.bhi2 = hi[2] * F.scale;
  }
}

SDFR_HD bool frame_box_empty(const Frame& F) { return F.blo0 > F.bhi0 || F.blo1 > F.bhi1 || F.blo2 > F.bhi2; }

/* Pixel coordinates (continuous, pixel-index units) of box corner `k` (bit0 -> x sign, ...);
 * returns false when the corner is not strictly in front of the camera. */
SDFR_HD bool project_corner(const Frame& F, const Camera& cam, int k, float& col, float& row) {
  const float sx = (k & 1) ? F.bhi0 : F.blo0; /* corners of the culling box */
  const float sy = (k & 2) ? F.bhi1 : F.blo1;
  const float sz = (k & 4) ? F.bhi2 : F.blo2;
  const float X = F.px + F.r00 * sx + F.r01 * sy + F.r02 * sz;
  const float Y = F.py + F.r10 * sx + F.r11 * sy + F.r12 * sz;
  const float Z = F.pz + F.r20 * sx + F.r21 * sy + F.r22 * sz;
  if (!(Z < -1e-30f)) return false;
  const float inv = 1.0f / (0.0f - Z);
  col = cam.cx - 0.5f + cam.fx * X * inv;
  row = cam.cy - 0.5f - cam.fy * Y * inv;
  return (col == col) && (row == row);
}

/* Turn min/max projected corner coordinates into a clamped, 1-pixel-padded rectangle. */
SDFR_HD void frame_rect(Frame& F, const Camera& cam, bool all_in_front, float cmin, float cmax,
                        float rmin, float rmax) {
  if (frame_box_empty(F)) { /* nothing can be hit: an empty rectangle, everything is zero-filled */
    F.x0 = F.y0 = F.x1 = F.y1 = 0;
    return;
  }
  if (!all_in_front) {
    F.x0 = 0; F.y0 = 0; F.x1 = cam.W; F.y1 = cam.H;
    return;
  }
  const float big = 1.0e9f;
  cmin = fminf(fmaxf(cmin, -big), big); cmax = fminf(fmaxf(cmax, -big), big);
  rmin = fminf(fmaxf(rmin, -big), big); rmax = fminf(fmaxf(rmax, -big), big);
  int x0 = (int)floorf(cmin) - 1, x1 = (int)ceilf(cmax) + 2;
  int y0 = (int)floorf(rmin) - 1, y1 = (int)ceilf(rmax) + 2;
  F.x0 = x0 < 0 ? 0 : x0; F.y0 = y0 < 0 ? 0 : y0;
  F.x1 = x1 > cam.W ? cam.W : x1; F.y1 = y1 > cam.H ? cam.H : y1;
}

/*
 * Silhouette culling.  The rays that can hit the box are exactly those through the convex hull of
 * the 8 projected corners (perspective projection preserves convexity in front of the camera);
 * the hull is kept as <= kMaxHullEdges half-planes  a*col + b*row + c >= 0  in pixel-index
 * coordinates, pushed outwards by kHullMargin pixels so that rounding can never cull a pixel
 * whose ray the exact slab test (cu:156-194) would accept.  The bounding rectangle alone keeps
 * ~40 % more pixels than the hull for the reference workloads (profiles/r01a_*).
 */
constexpr int kMaxHullEdges = 8;
constexpr float kHullMargin = 1.0f;     /* pixels */
constexpr float kHullCoordMax = 1.0e5f; /* beyond this fp32 pixel coordinates are too coarse */

struct alignas(16) HullEdge {
  float a, b, c, pad;
};

/* pair number L in [0,28) -> corners i < j */
SDFR_HD void hull_pair(int L, int& i, int& j) {
  int rem = L, row = 7;
  i = 0;
  while (rem >= row) {
    rem -= row;
    ++i;
    --row;
  }
  j = i + 1 + rem;
}

/* Normalised line through corners (xi,yi), (xj,yj); false when they (nearly) coincide. */
SDFR_HD bool hull_line(float xi, float yi, float xj, float yj, float& a, float& b, float& c) {
  a = -(yj - yi);
  b = xj - xi;
  const float len2 = a * a + b * b;
  if (!(len2 > 1e-6f)) return false;
  const float rl = SDFR_RSQRT(len2);
  a *= rl;
  b *= rl;
  c = -(a * xi + b * yi);
  return true;
}

/* Given the smallest / largest signed distance of the 8 corners to the line: is it a supporting
 * line of the hull?  Writes the outward-pushed half-plane. */
SDFR_HD bool hull_accept(float a, float b, float c, float smin, float smax, HullEdge& e) {
  const float eps = 1e-3f;
  if (smin >= -eps) {
    e.a = a; e.b = b; e.c = c + kHullMargin; e.pad = 0.0f;
    return true;
  }
  if (smax <= eps) {
    e.a = -a; e.b = -b; e.c = kHullMargin - c; e.pad = 0.0f;
    return true;
  }
  return false;
}

/* Serial hull builder (host emulation and tests; the kernels spread the 28 pairs over lanes).
 * Returns the number of edges written; 0 = no culling possible. */
SDFR_HD int build_hull_serial(const float* cols, const float* rows, bool all_in_front,
                              HullEdge* edges) {
  int n = 0;
  bool sane = all_in_front;
  for (int k = 0; k < 8; ++k)
    sane = sane && fabsf(cols[k]) <= kHullCoordMax && fabsf(rows[k]) <= kHullCoordMax;
  if (sane) {
    for (int L = 0; L < 28 && n < kMaxHullEdges; ++L) {
      int i, j;
      hull_pair(L, i, j);
      float a, b, c;
      if (!hull_line(cols[i], rows[i], cols[j], rows[j], a, b, c)) continue;
      float smin = 1e30f, smax = -1e30f;
      for (int k = 0; k < 8; ++k) {
        const float s = a * cols[k] + b * rows[k] + c;
        smin = fminf(smin, s);
        smax = fmaxf(smax, s);
      }
      if (hull_accept(a, b, c, smin, smax, edges[n])) ++n;
    }
  }
  for (int k = n; k < kMaxHullEdges; ++k) {
    edges[k].a = 0.0f; edges[k].b = 0.0f; edges[k].c = 1.0f; edges[k].pad = 0.0f;
  }
  return n;
}

/* Can any pixel of the w x h pixel block starting at (x0, y0) lie inside half-plane e? */
SDFR_HD bool hull_block_outside(const HullEdge& e, float x0, float y0, float w, float h) {
  const float ex = x0 + (e.a > 0.0f ? w - 1.0f : 0.0f);
  const float ey = y0 + (e.b > 0.0f ? h - 1.0f : 0.0f);
  return e.a * ex + e.b * ey + e.c < 0.0f;
}

/* Un-normalised ray components; evaluated in double then narrowed exactly like cu:146-147. */
SDFR_HD float pixel_dx(int col, float cx, float fx) { return (float)(((double)col + 0.5 - (double)cx) / (double)fx); }
SDFR_HD float pixel_dy(int row, float cy, float fy) { return (float)(-((double)row + 0.5 - (double)cy) / (double)fy); }

struct Ray {
  float dx, dy, dz;    /* unit direction, camera frame */
  float dox, doy, doz; /* same direction in the object frame */
};

/* cu:145-153 and cu:277-278; (ux, uy) = un-normalised components from the CTA tables */
SDFR_HD Ray make_ray(const Frame& F, float ux, float uy) {
  Ray r;
  const float rn = SDFR_RSQRT(ux * ux + uy * uy + 1);
  r.dx = ux * rn;
  r.dy = uy * rn;
  r.dz = -1.0f * rn;
  r.dox = F.r00 * r.dx + F.r10 * r.dy + F.r20 * r.dz;
  r.doy = F.r01 * r.dx + F.r11 * r.dy + F.r21 * r.dz;
  r.doz = F.r02 * r.dx + F.r12 * r.dy + F.r22 * r.dz;
  return r;
}

/* One slab of the ray/box test (cu:171-189); returns false on a miss. */
SDFR_HD bool slab(float e, float f, float scale, float& t_min, float& t_max) {
  /* (double)|f| > 1e-20  <=>  |f| > 1e-20f  (the float just below 1e-20 is the threshold) */
  if (fabsf(f) > 1e-20f) {
    float t1 = SDFR_SLAB_DIV(e + scale, f);
    float t2 = SDFR_SLAB_DIV(e - scale, f);
    if (t1 > t2) {
      const float tmp = t2;
      t2 = t1;
      t1 = tmp;
    }
    t_min = fmaxf(t_min, t1);
    t_max = fminf(t_max, t2);
    if (t_min > t_max || t_max < 0) return false;
  } else if (-e > scale || -e < -scale) {
    return false;
  }
  return true;
}

/* One axis of the culling-box test: the ray's object coordinate is  -e + t f; it lies in [lo, hi] for
 * t between (e + lo)/f and (e + hi)/f. */
SDFR_HD bool cull_slab(float e, float f, float lo, float hi, float& t_lo, float& t_hi) {
  if (fabsf(f) > 1e-20f) {
    const float ta = SDFR_SLAB_DIV(e + lo, f), tb = SDFR_SLAB_DIV(e + hi, f);
    t_lo = fmaxf(t_lo, fminf(ta, tb));
    t_hi = fminf(t_hi, fmaxf(ta, tb));
    return true;
  }
  return !(-e < lo || -e > hi);
}

/* Can the ray enter the culling box at all (anywhere along the line)?  Conservative by the box's
 * one-cell margin; rays that pass are traced exactly as the reference traces them. */
SDFR_HD bool ray_enters_cull_box(const Frame& F, const Ray& r) {
  float t_lo = -1e30f, t_hi = 1e30f;
  if (!cull_slab(F.e0, r.dox, F.blo0, F.bhi0, t_lo, t_hi)) return false;
  if (!cull_slab(F.e1, r.doy, F.blo1, F.bhi1, t_lo, t_hi)) return false;
  if (!cull_slab(F.e2, r.doz, F.blo2, F.bhi2, t_lo, t_hi)) return false;
  return t_lo <= t_hi;
}

/* Ray / oriented box (cu:156-194).  The box axes are the columns of R, so axis . d is the
 * object-frame direction component the march needs anyway. */
SDFR_HD bool ray_box(const Frame& F, const Ray& r, float& t_min, float& t_max) {
  t_min = -1e-10f;
  t_max = 1e10f;
  if (!slab(F.e0, r.dox, F.scale, t_min, t_max)) return false;
  if (!slab(F.e1, r.doy, F.scale, t_min, t_max)) return false;
  if (!slab(F.e2, r.doz, F.scale, t_min, t_max)) return false;
  t_min = fmaxf(t_min, 0.0f);
  return true;
}

/* Culling-box test and ray / oriented box in one go: what the render kernels call per pixel.
 *
 * Device build: the six slab evaluations (three of the culling box, three of the reference's box, cu:156-194)
 * divide by the same three direction components, so ONE reciprocal per axis (MUFU.RCP, exactly what
 * __fdividef issues per quotient -- the quotients are bit-identical to SDFR_SLAB_DIV's) serves all twelve
 * quotients, and the per-slab branches become selects.  __fdividef also carries a denormal-divisor rescue
 * (compare, select, two scalings) per quotient that is dead code here: the divisor is > 1e-20 in magnitude.
 * ~150 -> ~60 SASS instructions per ray; per-pixel set-up was 31 % of the fused kernel's instructions
 * (profiles/r02ag_ncu_fused_segments.txt).  The early exits of cu:171-189 can be taken at the end instead:
 * t_min only grows and t_max only shrinks over the slabs, so `t_min > t_max || t_max < 0` after any slab
 * implies the same after the last.  Host build: the two separate tests above. */
SDFR_HD bool ray_cull_and_box(const Frame& F, const Ray& r, float& t_min, float& t_max) {
#if defined(__CUDA_ARCH__)
  const bool a0 = fabsf(r.dox) > 1e-20f, a1 = fabsf(r.doy) > 1e-20f, a2 = fabsf(r.doz) > 1e-20f;
  float i0, i1, i2;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i0) : "f"(a0 ? r.dox : 1.0f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i1) : "f"(a1 ? r.doy : 1.0f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i2) : "f"(a2 ? r.doz : 1.0f));
  /* culling box: the ray's object coordinate is -e + t f; inside [lo, hi] for t between the two quotients */
  float c_lo = -1e30f, c_hi = 1e30f;
  bool ok = true;
  {
    const float ta = (F.e0 + F.blo0) * i0, tb = (F.e0 + F.bhi0) * i0;
    c_lo = a0 ? fmaxf(c_lo, fminf(ta, tb)) : c_lo;
    c_hi = a0 ? fminf(c_hi, fmaxf(ta, tb)) : c_hi;
    ok = ok && (a0 || !(-F.e0 < F.blo0 || -F.e0 > F.bhi0));
  }
  {
    const float ta = (F.e1 + F.blo1) * i1, tb = (F.e1 + F.bhi1) * i1;
    c_lo = a1 ? fmaxf(c_lo, fminf(ta, tb)) : c_lo;
    c_hi = a1 ? fminf(c_hi, fmaxf(ta, tb)) : c_hi;
    ok = ok && (a1 || !(-F.e1 < F.blo1 || -F.e1 > F.bhi1));
  }
  {
    const float ta = (F.e2 + F.blo2) * i2, tb = (F.e2 + F.bhi2) * i2;
    c_lo = a2 ? fmaxf(c_lo, fminf(ta, tb)) : c_lo;
    c_hi = a2 ? fminf(c_hi, fmaxf(ta, tb)) : c_hi;
    ok = ok && (a2 || !(-F.e2 < F.blo2 || -F.e2 > F.bhi2));
  }
  if (!ok || !(c_lo <= c_hi)) return false;
  /* the reference's box [-scale, scale]^3 (cu:156-194): min / max of the two quotients = its swap */
  float lo = -1e-10f, hi = 1e10f;
  const float s = F.scale;
  {
    const float t1 = (F.e0 + s) * i0, t2 = (F.e0 - s) * i0;
    lo = a0 ? fmaxf(lo, fminf(t1, t2)) : lo;
    hi = a0 ? fminf(hi, fmaxf(t1, t2)) : hi;
    ok = ok && (a0 || !(-F.e0 > s || -F.e0 < -s));
  }
  {
    const float t1 = (F.e1 + s) * i1, t2 = (F.e1 - s) * i1;
    lo = a1 ? fmaxf(lo, fminf(t1, t2)) : lo;
    hi = a1 ? fminf(hi, fmaxf(t1, t2)) : hi;
    ok = ok && (a1 || !(-F.e1 > s || -F.e1 < -s));
  }
  {
    const float t1 = (F.e2 + s) * i2, t2 = (F.e2 - s) * i2;
    lo = a2 ? fmaxf(lo, fminf(t1, t2)) : lo;
    hi = a2 ? fminf(hi, fmaxf(t1, t2)) : hi;
    ok = ok && (a2 || !(-F.e2 > s || -F.e2 < -s));
  }
  if (!ok || lo > hi || hi < 0) return false;
  t_min = fmaxf(lo, 0.0f);
  t_max = hi;
  return true;
#else
  return ray_enters_cull_box(F, r) && ray_box(F, r, t_min, t_max);
#endif
}

/* Cell lookup for a normalised object coordinate (cu:196-215): base index and cell origin. */
SDFR_HD int cell_index(const Grid& G, float u) {
  int i = SDFR_FLOOR_TO_INT((u + 1.0f) * G.Rm1f * 0.5f);
  i = i < G.Rm2 ? i : G.Rm2;
  return i > 0 ? i : 0;
}

struct Corners {
  float c000, c001, c010, c011, c100, c101, c110, c111; /* c{x}{y}{z} */
};

/* RT > 0 fixes resolution AND layout LT at compile time: the 8 gathers then share one 64-bit
 * address computation and use immediate offsets (RT = 0: run-time pitches G.py / G.px). */
template <int RT, int LT = kLayoutDense>
SDFR_HD Corners gather(const float* __restrict__ g, const Grid& G, int ix, int iy, int iz) {
  const int PY = RT > 0 ? (LT == kLayoutSkewed ? skew_pitch_y(RT) : RT) : G.py;
  const int PX = RT > 0 ? (LT == kLayoutSkewed ? skew_pitch_x(RT) : RT * RT) : G.px;
  const float* c = g + (ix * PX + iy * PY + iz);
  Corners k;
  k.c000 = SDFR_LDG(c);
  k.c001 = SDFR_LDG(c + 1);
  k.c010 = SDFR_LDG(c + PY);
  k.c011 = SDFR_LDG(c + PY + 1);
  k.c100 = SDFR_LDG(c + PX);
  k.c101 = SDFR_LDG(c + PX + 1);
  k.c110 = SDFR_LDG(c + PX + PY);
  k.c111 = SDFR_LDG(c + PX + PY + 1);
  return k;
}

/* Trilinear sample at object-frame point (x,y,z) (cu:217-239); offsets are not clamped. */
template <int RT, int LT = kLayoutDense>
SDFR_HD float trilinear(const float* __restrict__ g, const Grid& G, float x, float y, float z,
                        float inv_scale) {
  const float ux = x * inv_scale, uy = y * inv_scale, uz = z * inv_scale;
  const int ix = cell_index(G, ux), iy = cell_index(G, uy), iz = cell_index(G, uz);
  const float offx = G.hinv_fwd * (ux - ((float)ix * G.h - 1.0f));
  const float offy = G.hinv_fwd * (uy - ((float)iy * G.h - 1.0f));
  const float offz = G.hinv_fwd * (uz - ((float)iz * G.h - 1.0f));
  const Corners k = gather<RT, LT>(g, G, ix, iy, iz);
  const float c00 = k.c000 * (1 - offx) + k.c100 * offx;
  const float c01 = k.c001 * (1 - offx) + k.c101 * offx;
  const float c10 = k.c010 * (1 - offx) + k.c110 * offx;
  const float c11 = k.c011 * (1 - offx) + k.c111 * offx;
  const float c0 = c00 * (1 - offy) + c10 * offy;
  const float c1 = c01 * (1 - offy) + c11 * offy;
  return c0 * (1 - offz) + c1 * offz;
}

/*
 * Sphere trace (cu:283-293).  Returns the depth (-t*d_z) at the first sample with
 * dist < threshold*t, or 0.  `steps` counts trilinear samples; `capped` is set when the
 * step cap stopped the loop.
 */
template <int RT, int LT = kLayoutDense>
SDFR_HD float march(const float* __restrict__ g, const Grid& G, const Frame& F, const Ray& r,
                    float t_min, float t_max, float threshold, int& steps, bool& capped) {
  float t = t_min;
  int n = 0;
  capped = false;
  /* loop invariants in registers (F may live in shared memory) */
  const float ox = F.ox, oy = F.oy, oz = F.oz, inv_scale = F.inv_scale, scale = F.scale;
  const float dox = r.dox, doy = r.doy, doz = r.doz;
#ifndef SDFR_REFERENCE_ROUNDING
  /* Cell coordinate along the ray as ONE fma per axis: v(t) = ((o + t d) inv_scale + 1)(R-1)/2
   * = t a + b with per-ray a, b; cell = clamp(floor v), offset = v - cell; lerps as fma(f, hi - lo, lo).
   * 47 instead of 61 instructions per sample; the sample differs from the reference's expression
   * (cu:217-239, kept in trilinear<> for the backward and the other callers) by a few ulp of the
   * cell coordinate, ~1e-7 of the depth -- the parity tolerance is 1e-5. */
  const float hs = G.hinv_fwd * inv_scale;
  const float ax = dox * hs, ay = doy * hs, az = doz * hs;
  const float bx = fmaf(ox, hs, G.hinv_fwd), by = fmaf(oy, hs, G.hinv_fwd), bz = fmaf(oz, hs, G.hinv_fwd);
#endif
  while (t < t_max) {
#ifndef SDFR_REFERENCE_ROUNDING
    const float vx = fmaf(t, ax, bx), vy = fmaf(t, ay, by), vz = fmaf(t, az, bz);
    int ix = SDFR_FLOOR_TO_INT(vx), iy = SDFR_FLOOR_TO_INT(vy), iz = SDFR_FLOOR_TO_INT(vz);
    ix = ix < G.Rm2 ? ix : G.Rm2; ix = ix > 0 ? ix : 0;
    iy = iy < G.Rm2 ? iy : G.Rm2; iy = iy > 0 ? iy : 0;
    iz = iz < G.Rm2 ? iz : G.Rm2; iz = iz > 0 ? iz : 0;
    const float fx = vx - (float)ix, fy = vy - (float)iy, fz = vz - (float)iz;
    const Corners k = gather<RT, LT>(g, G, ix, iy, iz);
    const float c00 = fmaf(fx, k.c100 - k.c000, k.c000), c01 = fmaf(fx, k.c101 - k.c001, k.c001);
    const float c10 = fmaf(fx, k.c110 - k.c010, k.c010), c11 = fmaf(fx, k.c111 - k.c011, k.c011);
    const float c0 = fmaf(fy, c10 - c00, c00), c1 = fmaf(fy, c11 - c01, c01);
    const float dist = fmaf(fz, c1 - c0, c0) * scale;
#else
    const float dist =
        trilinear<RT, LT>(g, G, ox + t * dox, oy + t * doy, oz + t * doz, inv_scale) * scale;
#endif
    ++n;
    if (dist < threshold * t) {
      steps = n;
      return -t * r.dz;
    }
    t += dist;
    if (n >= kMaxSteps) {
      capped = true;
      break;
    }
  }
  steps = n;
  return 0.0f;
}

/* Result of the per-pixel backward: where to scatter and what. */
struct PixelGrad {
  int base;      /* linear index of corner 000 in the DENSE gradient grid */
  float w[8];    /* d depth / d corner, order 000,001,010,011,100,101,110,111 (x,y,z) */
  float pose[8]; /* d depth / d (x, y, z, qx, qy, qz, qw, inv_scale) */
};

/*
 * Analytic derivatives of one hit pixel (cu:334-457, simple_renderer.py:317-458).  The hit
 * point is re-derived from the stored depth (t = -z/d_z, cu:336-338).  exact_weights selects
 * the true trilinear corner weights (simple_renderer.py:399-408) instead of the list the
 * reference CUDA kernel uses (cu:373-388).  Values are NOT yet multiplied by the upstream
 * gradient, except w[] which follows the reference's multiplication order
 * ((((g*a)*b)*c)*f) when g is passed.
 */
template <int RT, bool WANT_SDF, bool WANT_POSE, int LT = kLayoutDense>
SDFR_HD void pixel_backward(const float* __restrict__ g, const Grid& G, const Frame& F,
                            const Ray& r, float z, float upstream, bool exact_weights,
                            PixelGrad& out) {
  const float t = -z / r.dz;
  const float xw = t * r.dx, yw = t * r.dy, zw = t * r.dz;                           /* cu:344 */
  const float o0 = F.ox + t * r.dox, o1 = F.oy + t * r.doy, o2 = F.oz + t * r.doz;   /* cu:345 */
  const float n0 = o0 * F.inv_scale, n1 = o1 * F.inv_scale, n2 = o2 * F.inv_scale;   /* cu:346 */
  const int ix = cell_index(G, n0), iy = cell_index(G, n1), iz = cell_index(G, n2);
  const float cx = G.hinv_bwd * (n0 - ((float)ix * G.h - 1.0f));                     /* cu:351-354 */
  const float cy = G.hinv_bwd * (n1 - ((float)iy * G.h - 1.0f));
  const float cz = G.hinv_bwd * (n2 - ((float)iz * G.h - 1.0f));
  const int Rr = RT > 0 ? RT : G.R;
  out.base = (ix * Rr + iy) * Rr + iz;
  const float absdz = fabsf(r.dz);
  const float f = F.scale * absdz;                                                   /* cu:372 */

  if (WANT_SDF) {
    const float gx1 = upstream * cx, gx0 = upstream * (1 - cx);
    if (exact_weights) {
      out.w[0] = gx0 * (1 - cy) * (1 - cz) * f;
      out.w[1] = gx0 * (1 - cy) * cz * f;
      out.w[2] = gx0 * cy * (1 - cz) * f;
      out.w[3] = gx0 * cy * cz * f;
      out.w[4] = gx1 * (1 - cy) * (1 - cz) * f;
      out.w[5] = gx1 * (1 - cy) * cz * f;
      out.w[6] = gx1 * cy * (1 - cz) * f;
      out.w[7] = gx1 * cy * cz * f;
    } else { /* cu:373-388 verbatim weight list */
      out.w[0] = gx0 * (1 - cy) * cz * f;
      out.w[1] = gx0 * cy * (1 - cz) * f;
      out.w[2] = gx0 * cy * cz * f;
      out.w[3] = gx1 * (1 - cy) * (1 - cz) * f;
      out.w[4] = gx1 * (1 - cy) * cz * f;
      out.w[5] = gx1 * (1 - cy) * cz * f;
      out.w[6] = gx1 * cy * (1 - cz) * f;
      out.w[7] = gx1 * cy * cz * f;
    }
  }

  if (WANT_POSE) {
    const Corners k = gather<RT, LT>(g, G, ix, iy, iz);
    const float c00 = k.c000 * (1 - cx) + k.c100 * cx;
    const float c01 = k.c001 * (1 - cx) + k.c101 * cx;
    const float c10 = k.c010 * (1 - cx) + k.c110 * cx;
    const float c11 = k.c011 * (1 - cx) + k.c111 * cx;
    const float c0 = c00 * (1 - cy) + c10 * cy;
    const float c1 = c01 * (1 - cy) + c11 * cy;
    const float t_diff = c0 * (1 - cz) + c1 * cz;

    const float qx = F.qx, qy = F.qy, qz = F.qz, qw = F.qw;
    const float s = F.inv_scale * G.hinv_bwd;                                        /* cu:391 */
    const float rx = xw - F.px, ry = yw - F.py, rz = zw - F.pz;                      /* cu:392 */
    float dc[8][3];
    /* position (cu:393-401) */
    dc[0][0] = (2 * (qy * qy + qz * qz) - 1) * s;
    dc[0][1] = 2 * (qw * qz - qx * qy) * s;
    dc[0][2] = -2 * (qx * qz + qw * qy) * s;
    dc[1][0] = -2 * (qx * qy + qw * qz) * s;
    dc[1][1] = (2 * (qx * qx + qz * qz) - 1) * s;
    dc[1][2] = 2 * (qw * qx - qy * qz) * s;
    dc[2][0] = 2 * (qw * qy - qx * qz) * s;
    dc[2][1] = -2 * (qy * qz + qw * qx) * s;
    dc[2][2] = (2 * (qx * qx + qy * qy) - 1) * s;
    /* quaternion x, y, z, w (cu:402-437) */
    dc[3][0] = (2 * qx * rx + 2 * qy * ry + 2 * qz * rz - 2 * qx * o0) * s;
    dc[3][1] = (2 * qy * rx - 2 * qx * ry + 2 * qw * rz - 2 * qx * o1) * s;
    dc[3][2] = (2 * qz * rx - 2 * qw * ry - 2 * qx * rz - 2 * qx * o2) * s;
    dc[4][0] = (-2 * qy * rx + 2 * qx * ry - 2 * qw * rz - 2 * qy * o0) * s;
    dc[4][1] = (2 * qx * rx + 2 * qy * ry + 2 * qz * rz - 2 * qy * o1) * s;
    dc[4][2] = (2 * qw * rx + 2 * qz * ry - 2 * qy * rz - 2 * qy * o2) * s;
    dc[5][0] = (-2 * qz * rx + 2 * qw * ry + 2 * qx * rz - 2 * qz * o0) * s;
    dc[5][1] = (-2 * qw * rx - 2 * qz * ry + 2 * qy * rz - 2 * qz * o1) * s;
    dc[5][2] = (2 * qx * rx + 2 * qy * ry + 2 * qz * rz - 2 * qz * o2) * s;
    dc[6][0] = (2 * qw * rx + 2 * qz * ry - 2 * qy * rz - 2 * qw * o0) * s;
    dc[6][1] = (-2 * qz * rx + 2 * qw * ry + 2 * qx * rz - 2 * qw * o1) * s;
    dc[6][2] = (2 * qy * rx - 2 * qx * ry + 2 * qw * rz - 2 * qw * o2) * s;
    /* inverse scale (cu:438) */
    dc[7][0] = o0 * G.hinv_bwd;
    dc[7][1] = o1 * G.hinv_bwd;
    dc[7][2] = o2 * G.hinv_bwd;
#pragma unroll
    for (int i = 0; i < 8; ++i) { /* cu:444-456 */
      const float dc00 = -k.c000 * dc[i][0] + k.c100 * dc[i][0];
      const float dc01 = -k.c001 * dc[i][0] + k.c101 * dc[i][0];
      const float dc10 = -k.c010 * dc[i][0] + k.c110 * dc[i][0];
      const float dc11 = -k.c011 * dc[i][0] + k.c111 * dc[i][0];
      const float dc0 = dc00 * (1 - cy) - c00 * dc[i][1] + dc10 * cy + c10 * dc[i][1];
      const float dc1 = dc01 * (1 - cy) - c01 * dc[i][1] + dc11 * cy + c11 * dc[i][1];
      const float dtdiff = dc0 * (1 - cz) - c0 * dc[i][2] + dc1 * cz + c1 * dc[i][2];
      out.pose[i] = F.scale * dtdiff * absdz;
    }
    out.pose[7] -= (t_diff * F.scale * F.scale) * absdz; /* cu:457 */
  }
}

/*
 * Pose gradients through MOMENTS (what the kernels use; pixel_backward above is the per-pixel
 * statement in the reference's operation order, kept for the host emulation and as documentation).
 *
 * Every pose derivative of cu:391-457 has the form  scale |d_z| (T . dc_i)  with T = grad of the
 * trilinear interpolant w.r.t. the local cell coordinate (cu:444-456 is that chain rule written out
 * eight times) and dc_i = d(local coordinate)/d(parameter i), and every dc_i is LINEAR in the
 * object-frame hit point o with coefficients that depend on the hypothesis only:
 *   position     dc_j   = -s R[j][:]                       (o = R^T (x - p))
 *   quaternion   dc_3+k = s (C_k (R o) - 2 q_k o)          (cu:402-437; R o = x - p)
 *   inv_scale    dc_7   = o hinv                           (cu:438), minus t_diff scale^2 |d_z| (cu:457)
 * with s = inv_scale * hinv.  So the sum over the pixels of a CTA needs only 13 accumulators,
 *   A_a  = sum w T_a,   Mo_ac = sum w T_a o_c,   D = sum w t_diff,     w = upstream * scale * |d_z|,
 * and the 13 -> 8 map is applied ONCE per CTA (moments_to_pose) instead of ~250 flops and a 24-entry
 * register table per pixel.  Same mathematics, different rounding (a sum of products instead of a
 * product of sums) -- well inside the 1e-3 gradient tolerance, which already has to absorb the
 * reordering of the fp32 atomics.
 */
constexpr int kMoments = 13;

template <int RT, bool WANT_SDF, bool WANT_POSE, int LT = kLayoutDense>
SDFR_HD void pixel_backward_moments(const float* __restrict__ g, const Grid& G, const Frame& F,
                                    const Ray& r, float z, float upstream, bool exact_weights,
                                    int& base, float (&w)[8], float (&acc)[kMoments]) {
  const float t = -z / r.dz;                                                         /* cu:336-338 */
  const float o0 = F.ox + t * r.dox, o1 = F.oy + t * r.doy, o2 = F.oz + t * r.doz;   /* cu:345 */
  const float n0 = o0 * F.inv_scale, n1 = o1 * F.inv_scale, n2 = o2 * F.inv_scale;   /* cu:346 */
  const int ix = cell_index(G, n0), iy = cell_index(G, n1), iz = cell_index(G, n2);
  const float cx = G.hinv_bwd * (n0 - ((float)ix * G.h - 1.0f));                     /* cu:351-354 */
  const float cy = G.hinv_bwd * (n1 - ((float)iy * G.h - 1.0f));
  const float cz = G.hinv_bwd * (n2 - ((float)iz * G.h - 1.0f));
  const int Rr = RT > 0 ? RT : G.R;
  base = (ix * Rr + iy) * Rr + iz;
  const float f = F.scale * fabsf(r.dz);                                             /* cu:372 */
  if (WANT_SDF) {
    const float gx1 = upstream * cx, gx0 = upstream * (1 - cx);
    if (exact_weights) { /* simple_renderer.py:399-408 */
      w[0] = gx0 * (1 - cy) * (1 - cz) * f; w[1] = gx0 * (1 - cy) * cz * f;
      w[2] = gx0 * cy * (1 - cz) * f;       w[3] = gx0 * cy * cz * f;
      w[4] = gx1 * (1 - cy) * (1 - cz) * f; w[5] = gx1 * (1 - cy) * cz * f;
      w[6] = gx1 * cy * (1 - cz) * f;       w[7] = gx1 * cy * cz * f;
    } else { /* cu:373-388 verbatim weight list */
      w[0] = gx0 * (1 - cy) * cz * f;       w[1] = gx0 * cy * (1 - cz) * f;
      w[2] = gx0 * cy * cz * f;             w[3] = gx1 * (1 - cy) * (1 - cz) * f;
      w[4] = gx1 * (1 - cy) * cz * f;       w[5] = gx1 * (1 - cy) * cz * f;
      w[6] = gx1 * cy * (1 - cz) * f;       w[7] = gx1 * cy * cz * f;
    }
  }
  if (WANT_POSE) {
    const Corners k = gather<RT, LT>(g, G, ix, iy, iz);
    /* differences along x of the four x-edges, then the interpolant and its gradient */
    const float e00 = k.c100 - k.c000, e01 = k.c101 - k.c001, e10 = k.c110 - k.c010, e11 = k.c111 - k.c011;
    const float c00 = k.c000 + cx * e00, c01 = k.c001 + cx * e01;
    const float c10 = k.c010 + cx * e10, c11 = k.c011 + cx * e11;
    const float ex0 = e00 + cy * (e10 - e00), ex1 = e01 + cy * (e11 - e01);
    const float c0 = c00 + cy * (c10 - c00), c1 = c01 + cy * (c11 - c01);
    const float Tx = ex0 + cz * (ex1 - ex0);
    const float Ty = (c10 - c00) + cz * ((c11 - c01) - (c10 - c00));
    const float Tz = c1 - c0;
    const float t_diff = c0 + cz * Tz;
    const float wt = upstream * f;
    const float a0 = wt * Tx, a1 = wt * Ty, a2 = wt * Tz;
    acc[0] += a0; acc[1] += a1; acc[2] += a2;
    acc[3] += a0 * o0; acc[4] += a0 * o1; acc[5] += a0 * o2;
    acc[6] += a1 * o0; acc[7] += a1 * o1; acc[8] += a1 * o2;
    acc[9] += a2 * o0; acc[10] += a2 * o1; acc[11] += a2 * o2;
    acc[12] += wt * t_diff;
  }
}

/* The 13 -> 8 map: gradients w.r.t. (x, y, z, qx, qy, qz, qw, inv_scale) from the moment sums, evaluated
 * in MT (float in the kernels, double in the host checks).  The quaternion rows are written as ONE
 * matrix K_k = C_k R - q_k I contracted with Mo, so that their two halves (C_k (x - p) and -2 q_k o of
 * cu:402-437) cancel in the nine entries of K_k -- once per CTA, on numbers of size 1 -- instead of
 * between sums over all pixels. */
template <typename MT>
SDFR_HD void moments_to_pose(const Frame& F, const Grid& G, const MT* m, float* out) {
  const MT s = (MT)F.inv_scale * (MT)G.hinv_bwd;                                     /* cu:391 */
  const MT qx = F.qx, qy = F.qy, qz = F.qz, qw = F.qw;
  const MT R[3][3] = {{(MT)F.r00, (MT)F.r01, (MT)F.r02}, {(MT)F.r10, (MT)F.r11, (MT)F.r12},
                      {(MT)F.r20, (MT)F.r21, (MT)F.r22}};
#pragma unroll
  for (int j = 0; j < 3; ++j)                                                        /* cu:393-401 */
    out[j] = (float)(-s * (R[j][0] * (MT)m[0] + R[j][1] * (MT)m[1] + R[j][2] * (MT)m[2]));
  /* C_k[a][b]: coefficient of (x - p)_b in component a of d c / d q_k (cu:402-437) */
  const MT C[4][3][3] = {
      {{qx, qy, qz}, {qy, -qx, qw}, {qz, -qw, -qx}},
      {{-qy, qx, -qw}, {qx, qy, qz}, {qw, qz, -qy}},
      {{-qz, qw, qx}, {-qw, -qz, qy}, {qx, qy, qz}},
      {{qw, qz, -qy}, {-qz, qw, qx}, {qy, -qx, qw}}};
  const MT qk[4] = {qx, qy, qz, qw};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    MT acc = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        /* K_k[a][c] = sum_b C_k[a][b] R[b][c] - q_k delta_ac  (x - p = R o) */
        MT kac = C[k][a][0] * R[0][c] + C[k][a][1] * R[1][c] + C[k][a][2] * R[2][c];
        if (a == c) kac -= qk[k];
        acc += kac * (MT)m[3 + 3 * a + c];
      }
    }
    out[3 + k] = (float)((MT)2 * s * acc);
  }
  const MT N = (MT)m[3] + (MT)m[7] + (MT)m[11]; /* sum w (T . o) */
  out[7] = (float)((MT)G.hinv_bwd * N - (MT)F.scale * (MT)m[12]);                    /* cu:438, 457 */
}

}  // namespace sdfr
#endif /* SDFR_CORE_CUH_ */
