/*
 * sdfr_decoder.cuh -- the tail of the SDF decoder as sm_100a kernels (SURVEY.md section 8f, rank 2).
 * Included by sdfrender.cu inside its anonymous namespace.
 *
 * The reference decoder (sdfest/vae/sdf_vae.py:217-259, layer sizes
 * estimation/configs/models/mug.yaml:2-12) ends with
 *     interpolate(x[N,C,S,S,S] -> (R,R,R), mode="trilinear", align_corners=False)   sdf_vae.py:235-244
 *     Conv3d(C -> 1, kernel_size=1), no ReLU                                          sdf_vae.py:245-247
 * (C = 4, S = 30, R = 64 for every shipped model).  Run through torch this materialises a
 * C x R^3 intermediate per hypothesis (4 MiB at 64^3; 256 MiB for 64 hypotheses) that is written,
 * read back by the convolution, and -- in the backward -- produced and consumed once more.  Both
 * operators are linear and act on different axes (channels vs. space), so they commute:
 *     sdf[o] = bias + sum_s W(o, s) * (sum_c weight[c] * x[c, s])
 * and the tail becomes ONE pass that reads the 4 x 30^3 input and writes the R^3 grid directly in
 * whichever layout the renderer wants (dense, or the bank-conflict-free skewed layout of
 * sdfr_core.cuh -- which also removes the separate sdfr_skew_grids pass from the loop).
 *
 * Interpolation weights follow ATen's upsample_trilinear3d exactly (align_corners = False,
 * no scale_factor):  src = max(0, (S/R) * (o + 0.5) - 0.5),  i0 = (int)src,
 * i1 = i0 + (i0 < S-1),  l1 = src - i0,  l0 = 1 - l1.  Floating point: the summation order differs
 * from torch's (channel contraction first), so parity is to fp32 rounding, not bit-exact.
 *
 * Backward = the adjoint: grad_x[c, s] = weight[c] * sum_o W(o, s) * g[o], evaluated separably
 * (x, then z, then y) in shared memory by one CTA per source x-plane, with the deferred
 * per-hypothesis normalisation of the fused render-and-compare gradient (upstream/n_overlap,
 * sdfr_compare_fused) and an optional second gradient grid (the point-cloud loss) folded into the
 * load:  g = coef[b] * grad_sdf + grad_sdf_extra.  The decoder weights are frozen in the
 * estimation loop (simple_setup.py:65), so no weight/bias gradients are produced.
 */
#ifndef SDFR_DECODER_CUH_
#define SDFR_DECODER_CUH_

constexpr int kTailMaxChannels = 16;
constexpr int kTailMaxSize = 128; /* S, R <= 128: the separable backward keeps an R x R plane in shared memory */

struct TailParams {
  const float* __restrict__ x;       /* [B, C, S, S, S] */
  const float* __restrict__ weight;  /* [C] */
  const float* __restrict__ bias;    /* [1] or NULL */
  const float* __restrict__ base;    /* [R,R,R] dense, added to every hypothesis' grid, or NULL */
  int C, S, R;
  /* forward */
  float* __restrict__ out;
  long long out_stride;
  int py, px; /* output pitches (elements) between consecutive y / x */
  /* backward */
  const float* __restrict__ g_main;
  long long g_main_stride;
  const float* __restrict__ n_overlap; /* [B] or NULL */
  const float* __restrict__ upstream;  /* [B] or NULL */
  const float* __restrict__ g_extra;   /* or NULL */
  long long g_extra_stride;
  float* __restrict__ g_x; /* [B, C, S, S, S] */
  int z_offset;
  CellBounds* __restrict__ bounds; /* forward, optional: per-hypothesis empty-space bounds (tau pre-set by
                                    * sdfr_bounds_init_kernel), updated from the values as they are written */
  int xb; /* forward: output x-planes per CTA */
  int fast4; /* forward: 4-row groups (tail_forward_plan); backward: float4 loads of the gradient planes */
};

/* ATen area_pixel_compute_source_index, align_corners = false, linear */
__device__ __forceinline__ void tail_source(int o, float ratio, int S, int& i0, int& i1, float& l1) {
  float src = ratio * ((float)o + 0.5f) - 0.5f;
  src = src < 0.0f ? 0.0f : src;
  i0 = (int)src;
  i0 = i0 < S - 1 ? i0 : S - 1;
  i1 = i0 + (i0 < S - 1 ? 1 : 0);
  l1 = src - (float)i0;
}

/* Host copy of tail_source (same fp32 arithmetic) for sizing the staging buffer. */
inline void tail_source_host(int o, int S, int R, int& i0, int& i1) {
  const float ratio = (float)S / (float)R;
  float src = ratio * ((float)o + 0.5f) - 0.5f;
  src = src < 0.0f ? 0.0f : src;
  i0 = (int)src;
  i0 = i0 < S - 1 ? i0 : S - 1;
  i1 = i0 + (i0 < S - 1 ? 1 : 0);
}

/*
 * One CTA per (slab of P.xb consecutive output x-planes, hypothesis): the source x-planes the slab
 * reads are channel-contracted once into shared memory, then every output is a trilinear blend of
 * 8 shared-memory values.  (First version: one CTA per output x-plane -- 4096..16384 CTAs of three
 * barrier-separated phases each, 60 M warp instructions for the 64^3 tail and bound by CTA turnover,
 * not bandwidth: profiles/r01j_ncu_decoder.txt.)
 */
template <int ST, int RT> /* compile-time sizes for the shipped decoders' resizes, 0 = run time */
__global__ void __launch_bounds__(256)
sdfr_decoder_tail_forward_kernel(const __grid_constant__ TailParams P) {
  extern __shared__ __align__(16) float tail_smem[];
  const int S = ST ? ST : P.S, R = RT ? RT : P.R, C = P.C;
  int* ti0 = (int*)tail_smem;         /* [R] */
  int* ti1 = ti0 + R;                 /* [R] */
  float* tl1 = (float*)(ti1 + R);     /* [R] */
  float* wy = tl1 + R;                /* [R][4] (fast4): weight of source row ti0[4*(oy/4)] + k on output row oy */
  float* src = wy + (P.fast4 ? 4 * R : 0); /* [np][S*S] channel-contracted source planes */
  const int b = blockIdx.y + P.z_offset;
  const int ox0 = blockIdx.x * P.xb;
  const int nxo = R - ox0 < P.xb ? R - ox0 : P.xb;
  const float ratio = (float)S / (float)R;
  for (int o = threadIdx.x; o < R; o += blockDim.x) {
    int i0, i1;
    float l1;
    tail_source(o, ratio, S, i0, i1, l1);
    ti0[o] = i0; ti1[o] = i1; tl1[o] = l1;
  }
  __syncthreads();
  if (P.fast4) {
    for (int e = threadIdx.x; e < 4 * R; e += blockDim.x) {
      const int oy = e >> 2, row = ti0[oy & ~3] + (e & 3);
      const float l1 = tl1[oy];
      wy[e] = (ti0[oy] == row ? 1.0f - l1 : 0.0f) + (ti1[oy] == row ? l1 : 0.0f);
    }
  }
  const int xs_lo = ti0[ox0], np = ti1[ox0 + nxo - 1] - xs_lo + 1;
  float w[kTailMaxChannels];
#pragma unroll
  for (int c = 0; c < kTailMaxChannels; ++c)
    w[c] = c < C ? (P.weight ? __ldg(P.weight + c) : 1.0f) : 0.0f; /* NULL weight: plain upsampling */
  const int S2 = S * S;
  const size_t S3 = (size_t)S2 * S;
  const float* __restrict__ xb = P.x + (size_t)b * C * S3 + (size_t)xs_lo * S2;
  for (int e = threadIdx.x; e < np * S2; e += blockDim.x) {
    float v = 0.0f;
#pragma unroll
    for (int c = 0; c < kTailMaxChannels; ++c)
      if (c < C) v += w[c] * __ldg(xb + c * S3 + e);
    src[e] = v;
  }
  __syncthreads();
  const float bias = P.bias ? __ldg(P.bias) : 0.0f;
  float* __restrict__ out = P.out + (size_t)b * P.out_stride;
  /* empty-space bounds while the grid is being written (sdfr_bounds_scan_kernel's rule: bounding box of the
   * voxels below tau, low side moved down one cell): saves the separate read of the grids */
  const float tau = P.bounds ? P.bounds[b].tau : -3.0e38f;
  int vxl = 0x7fffffff, vxh = -1, vyl = 0x7fffffff, vyh = -1, vzl = 0x7fffffff, vzh = -1;
  if (P.fast4) {
    /* A thread keeps ONE output column oz (z-interpolation constants in registers) and produces FOUR
     * consecutive output rows per step: the <= 4 source rows they read are blended in x and z once
     * (16 shared-memory loads) and combined with a 4x4 weight block from wy.  The first version
     * produced one output per step from 8 loads and ~70 instructions, most of them integer address
     * arithmetic (profiles/r01s_ncu_decoder.txt); this one needs ~19 per output. */
    const int oz = threadIdx.x % R, rl = threadIdx.x / R, rows = 256 / R, G = R >> 2;
    const int z0 = ti0[oz], z1 = ti1[oz];
    const float lz1 = tl1[oz], lz0 = 1.0f - lz1;
    const size_t R2 = (size_t)R * R;
    for (int dx = 0; dx < nxo; ++dx) {
      const int ox = ox0 + dx;
      const float* __restrict__ pa = src + (ti0[ox] - xs_lo) * S2;
      const float* __restrict__ pb = src + (ti1[ox] - xs_lo) * S2;
      const float lx1 = tl1[ox], lx0 = 1.0f - lx1;
      float* __restrict__ o = out + (size_t)ox * P.px + oz;
      const float* __restrict__ base = P.base ? P.base + (size_t)ox * R2 + oz : nullptr;
      for (int g = rl; g < G; g += rows) {
        const int yb = ti0[4 * g];
        float r[4];
        if (yb + 3 < S) {
          /* the four source rows are consecutive: with compile-time S the 16 loads share four base
           * addresses and differ by immediates (the clamped form below computes 16 addresses) */
          const float* __restrict__ a0 = pa + yb * S + z0;
          const float* __restrict__ a1 = pa + yb * S + z1;
          const float* __restrict__ c0 = pb + yb * S + z0;
          const float* __restrict__ c1 = pb + yb * S + z1;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float a = lz0 * a0[k * S] + lz1 * a1[k * S];
            const float c = lz0 * c0[k * S] + lz1 * c1[k * S];
            r[k] = lx0 * a + lx1 * c;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int row = (yb + k < S ? yb + k : S - 1) * S;
            const float a = lz0 * pa[row + z0] + lz1 * pa[row + z1];
            const float c = lz0 * pb[row + z0] + lz1 * pb[row + z1];
            r[k] = lx0 * a + lx1 * c;
          }
        }
        const float4* __restrict__ W = reinterpret_cast<const float4*>(wy + 16 * g);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 w4 = W[i];
          float v = (w4.x * r[0] + w4.y * r[1] + w4.z * r[2] + w4.w * r[3]) + bias;
          const int oy = 4 * g + i;
          if (base) v += __ldg(base + oy * R);
          o[(size_t)oy * P.py] = v;
          if (v < tau) {
            vxl = min(vxl, ox); vxh = max(vxh, ox);
            vyl = min(vyl, oy); vyh = max(vyh, oy);
            vzl = oz; vzh = oz;
          }
        }
      }
    }
  } else {
  for (int j = threadIdx.x; j < nxo * R * R; j += blockDim.x) {
    const int dx = j / (R * R), r = j - dx * R * R;
    const int oy = r / R, oz = r - oy * R, ox = ox0 + dx;
    const float* __restrict__ pa = src + (ti0[ox] - xs_lo) * S2;
    const float* __restrict__ pb = src + (ti1[ox] - xs_lo) * S2;
    const int r0 = ti0[oy] * S, r1 = ti1[oy] * S, z0 = ti0[oz], z1 = ti1[oz];
    const float lx1 = tl1[ox], ly1 = tl1[oy], lz1 = tl1[oz];
    const float lx0 = 1.0f - lx1, ly0 = 1.0f - ly1, lz0 = 1.0f - lz1;
    const float a0 = lz0 * pa[r0 + z0] + lz1 * pa[r0 + z1];
    const float a1 = lz0 * pa[r1 + z0] + lz1 * pa[r1 + z1];
    const float b0 = lz0 * pb[r0 + z0] + lz1 * pb[r0 + z1];
    const float b1 = lz0 * pb[r1 + z0] + lz1 * pb[r1 + z1];
    float v = (lx0 * (ly0 * a0 + ly1 * a1) + lx1 * (ly0 * b0 + ly1 * b1)) + bias;
    if (P.base) v += __ldg(P.base + (size_t)ox * R * R + r);
    out[(size_t)ox * P.px + oy * P.py + oz] = v;
    if (v < tau) {
      vxl = min(vxl, ox); vxh = max(vxh, ox);
      vyl = min(vyl, oy); vyh = max(vyh, oy);
      vzl = min(vzl, oz); vzh = max(vzh, oz);
    }
  }
  }
  if (P.bounds) { /* uniform over the grid */
    vxl = __reduce_min_sync(0xffffffffu, vxl); vxh = __reduce_max_sync(0xffffffffu, vxh);
    vyl = __reduce_min_sync(0xffffffffu, vyl); vyh = __reduce_max_sync(0xffffffffu, vyh);
    vzl = __reduce_min_sync(0xffffffffu, vzl); vzh = __reduce_max_sync(0xffffffffu, vzh);
    if ((threadIdx.x & 31) == 0 && vxh >= 0) {
      bounds_commit(P.bounds + b, 0, vxl, vxh, R);
      bounds_commit(P.bounds + b, 1, vyl, vyh, R);
      bounds_commit(P.bounds + b, 2, vzl, vzh, R);
    }
  }
}

/* weight of output index o on source index s along one axis */
__device__ __forceinline__ float tail_weight(const int* ti0, const int* ti1, const float* tl1, int o,
                                             int s) {
  const float l1 = tl1[o];
  return (ti0[o] == s ? 1.0f - l1 : 0.0f) + (ti1[o] == s ? l1 : 0.0f);
}

/* upper bound on the number of output indices that read one source index along an axis */
__host__ __device__ constexpr int tail_taps(int S, int R) { return 2 * ((R + S - 1) / S) + 2; }

/* One CTA per (source x-plane, hypothesis). */
template <int ST, int RT>
__global__ void __launch_bounds__(256)
sdfr_decoder_tail_backward_kernel(const __grid_constant__ TailParams P) {
  extern __shared__ __align__(16) float tail_smem[];
  const int S = ST ? ST : P.S, R = RT ? RT : P.R, C = P.C;
  const int KW = tail_taps(S, R);
  float* Pl = tail_smem;              /* [R][R]  x-collapsed gradient plane */
  float* Q = Pl + R * R;              /* [R][S]  ... z-collapsed */
  float* Wt = Q + R * S;              /* [S][KW] weight of output lo[s]+k on source s (0 past hi[s]) */
  int* ti0 = (int*)(Wt + S * KW);     /* [R] */
  int* ti1 = ti0 + R;
  float* tl1 = (float*)(ti1 + R);
  int* lo = (int*)(tl1 + R);          /* [S] first / last output index touching source s */
  int* hi = lo + S;
  const int b = blockIdx.y + P.z_offset, sx = blockIdx.x;
  const float ratio = (float)S / (float)R;
  for (int o = threadIdx.x; o < R; o += blockDim.x) {
    int i0, i1;
    float l1;
    tail_source(o, ratio, S, i0, i1, l1);
    ti0[o] = i0; ti1[o] = i1; tl1[o] = l1;
  }
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    lo[s] = R;
    hi[s] = -1;
  }
  __syncthreads();
  /* first / last output index reading each source index: one shared-memory atomic pair per output
   * (the first version scanned all R outputs serially per source index -- 30 threads busy for
   * 64 iterations while the other 226 waited at the barrier, in each of 1920 CTAs) */
  for (int o = threadIdx.x; o < R; o += blockDim.x) {
    atomicMin(&lo[ti0[o]], o);
    atomicMax(&hi[ti0[o]], o);
    atomicMin(&lo[ti1[o]], o);
    atomicMax(&hi[ti1[o]], o);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < S * KW; e += blockDim.x) {
    const int s = e / KW, o = lo[s] + (e - s * KW);
    Wt[e] = o <= hi[s] ? tail_weight(ti0, ti1, tl1, o, s) : 0.0f;
  }
  __syncthreads();

  float coef = 1.0f;
  if (P.n_overlap) {
    const float n = __ldg(P.n_overlap + b);
    coef = n > 0.0f ? (P.upstream ? __ldg(P.upstream + b) : 1.0f) / n : 0.0f;
  } else if (P.upstream) {
    coef = __ldg(P.upstream + b);
  }
  const size_t R2 = (size_t)R * R;
  const float* __restrict__ ga = P.g_main + (size_t)b * P.g_main_stride;
  const float* __restrict__ ge = P.g_extra ? P.g_extra + (size_t)b * P.g_extra_stride : nullptr;
  const int xlo = lo[sx], nx = hi[sx] - xlo + 1;
  const float* __restrict__ wx = Wt + sx * KW;
  /* 1. collapse x:  Pl[oy][oz] = sum_ox W(ox, sx) g[ox][oy][oz]  (float4 when the planes allow it:
   * the scalar loop below costs 37 instructions per element, half of the kernel) */
  if (P.fast4) {
    const int n4 = (int)(R2 >> 2);
    const float4* __restrict__ ga4 = reinterpret_cast<const float4*>(ga + (size_t)xlo * R2);
    const float4* __restrict__ ge4 = ge ? reinterpret_cast<const float4*>(ge + (size_t)xlo * R2) : nullptr;
    const bool use_main = coef != 0.0f;
    constexpr int KU = ST ? tail_taps(ST ? ST : 1, RT ? RT : 1) : 1; /* all taps' loads in flight at once */
    for (int j = threadIdx.x; j < n4; j += blockDim.x) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll KU
      for (int k = 0; k < nx; ++k) {
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (use_main) {
          g = __ldg(ga4 + (size_t)k * n4 + j);
          g.x *= coef; g.y *= coef; g.z *= coef; g.w *= coef;
        }
        if (ge4) {
          const float4 e = __ldg(ge4 + (size_t)k * n4 + j);
          g.x += e.x; g.y += e.y; g.z += e.z; g.w += e.w;
        }
        const float w = wx[k];
        acc.x += w * g.x; acc.y += w * g.y; acc.z += w * g.z; acc.w += w * g.w;
      }
      reinterpret_cast<float4*>(Pl)[j] = acc;
    }
  } else
  for (int j = threadIdx.x; j < (int)R2; j += blockDim.x) {
    float acc = 0.0f;
    for (int k = 0; k < nx; ++k) {
      const size_t idx = (size_t)(xlo + k) * R2 + j;
      float g = coef != 0.0f ? coef * __ldg(ga + idx) : 0.0f;
      if (ge) g += __ldg(ge + idx);
      acc += wx[k] * g;
    }
    Pl[j] = acc;
  }
  __syncthreads();
  /* 2. collapse z:  Q[oy][sz] = sum_oz W(oz, sz) Pl[oy][oz] */
  for (int j = threadIdx.x; j < R * S; j += blockDim.x) {
    const int oy = j / S, sz = j - oy * S;
    const float* __restrict__ w = Wt + sz * KW;
    const float* __restrict__ p = Pl + oy * R + lo[sz];
    const int n = hi[sz] - lo[sz] + 1;
    float acc = 0.0f;
    for (int k = 0; k < n; ++k) acc += w[k] * p[k];
    Q[j] = acc;
  }
  __syncthreads();
  /* 3. collapse y and fan out over the channels */
  const size_t S2 = (size_t)S * S, S3 = S2 * S;
  float* __restrict__ gx = P.g_x + (size_t)b * C * S3 + (size_t)sx * S2;
  for (int j = threadIdx.x; j < (int)S2; j += blockDim.x) {
    const int sy = j / S, sz = j - sy * S;
    const float* __restrict__ w = Wt + sy * KW;
    const float* __restrict__ q = Q + lo[sy] * S + sz;
    const int n = hi[sy] - lo[sy] + 1;
    float acc = 0.0f;
    for (int k = 0; k < n; ++k) acc += w[k] * q[k * S];
    for (int c = 0; c < C; ++c) gx[c * S3 + j] = (P.weight ? __ldg(P.weight + c) : 1.0f) * acc;
  }
}

/* Slab thickness (output x-planes per CTA) and the shared memory it needs: aim at ~32 K outputs
 * per CTA, shrink while the staged source planes do not fit. */
size_t tail_forward_plan(int S, int R, int batch, int& xb, int& fast4) {
  fast4 = (R % 4 == 0 && R <= 256 && 256 % R == 0) ? 1 : 0;
  for (int g = 0; fast4 && g < R / 4; ++g) { /* every 4-row group must read at most 4 source rows */
    int a0, a1, b0, b1;
    tail_source_host(4 * g, S, R, a0, a1);
    tail_source_host(4 * g + 3, S, R, b0, b1);
    if (b1 - a0 > 3) fast4 = 0;
  }
  xb = 32768 / (R * R);
  xb = xb < 1 ? 1 : (xb > R ? R : xb);
  /* thinner slabs only when the grid would not even fill the SMs twice (measured: 4 instead of 8
   * planes per CTA at 64 hypotheses re-stages more than the extra CTAs hide, 75 -> 81 us) */
  while (xb > 2 && (long)((R + xb - 1) / xb) * batch < 296) xb /= 2;
  for (;;) {
    int np = 1;
    for (int ox0 = 0; ox0 < R; ox0 += xb) {
      const int last = ox0 + xb - 1 < R - 1 ? ox0 + xb - 1 : R - 1;
      int a0, a1, b0, b1;
      tail_source_host(ox0, S, R, a0, a1);
      tail_source_host(last, S, R, b0, b1);
      np = b1 - a0 + 1 > np ? b1 - a0 + 1 : np;
    }
    const size_t bytes = sizeof(float) * ((size_t)np * S * S + (fast4 ? 7 : 3) * (size_t)R);
    if (bytes <= 160 * 1024 || xb == 1) return bytes;
    xb = xb / 2;
  }
}
size_t tail_backward_smem(int S, int R) {
  return sizeof(float) * ((size_t)R * R + (size_t)R * S + (size_t)S * tail_taps(S, R) + 3 * (size_t)R +
                          2 * (size_t)S);
}

int tail_check(int C, int S, int R, int batch) {
  if (C < 1 || C > kTailMaxChannels) return fail(SDFR_E_SHAPE, "decoder tail: channels must be in [1, 16]");
  if (S < 1 || S > kTailMaxSize || R < 2 || R > kTailMaxSize)
    return fail(SDFR_E_SHAPE, "decoder tail: in_size must be in [1, 128] and resolution in [2, 128]");
  if (batch < 0) return fail(SDFR_E_SHAPE, "negative batch");
  return 0;
}

template <int ST, int RT>
int launch_tail_forward_t(TailParams P, int batch, size_t smem, cudaStream_t s) {
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(sdfr_decoder_tail_forward_kernel<ST, RT>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "decoder tail forward: shared memory opt-in failed");
  }
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid((P.R + P.xb - 1) / P.xb, batch - z0 < 65535 ? batch - z0 : 65535);
    sdfr_decoder_tail_forward_kernel<ST, RT><<<grid, 256, smem, s>>>(P);
  }
  return check_launch("sdfr_decoder_tail_forward_kernel");
}

/* the resizes of every decoder the reference ships (mug.yaml and siblings: 8 -> 6 -> 16, 14 -> 32,
 * 30 -> 64) get compile-time sizes: most of the generic kernels' instructions are index arithmetic */
int launch_tail_forward(TailParams P, int batch, cudaStream_t s) {
  const size_t smem = tail_forward_plan(P.S, P.R, batch, P.xb, P.fast4);
  if (P.S == 30 && P.R == 64) return launch_tail_forward_t<30, 64>(P, batch, smem, s);
  if (P.S == 14 && P.R == 32) return launch_tail_forward_t<14, 32>(P, batch, smem, s);
  if (P.S == 6 && P.R == 16) return launch_tail_forward_t<6, 16>(P, batch, smem, s);
  return launch_tail_forward_t<0, 0>(P, batch, smem, s);
}

template <int ST, int RT>
int launch_tail_backward_t(TailParams P, int batch, size_t smem, cudaStream_t s) {
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(sdfr_decoder_tail_backward_kernel<ST, RT>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "decoder tail backward: shared memory opt-in failed");
  }
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid(P.S, batch - z0 < 65535 ? batch - z0 : 65535);
    sdfr_decoder_tail_backward_kernel<ST, RT><<<grid, 256, smem, s>>>(P);
  }
  return check_launch("sdfr_decoder_tail_backward_kernel");
}

int launch_tail_backward(TailParams P, int batch, cudaStream_t s) {
  const size_t smem = tail_backward_smem(P.S, P.R);
  const uintptr_t al = reinterpret_cast<uintptr_t>(P.g_main) | reinterpret_cast<uintptr_t>(P.g_extra);
  P.fast4 = ((P.R * P.R) % 4 == 0 && P.R >= 32 && (al & 15) == 0 && P.g_main_stride % 4 == 0 &&
             (!P.g_extra || P.g_extra_stride % 4 == 0)) ? 1 : 0;
  if (P.S == 30 && P.R == 64) return launch_tail_backward_t<30, 64>(P, batch, smem, s);
  if (P.S == 14 && P.R == 32) return launch_tail_backward_t<14, 32>(P, batch, smem, s);
  if (P.S == 6 && P.R == 16) return launch_tail_backward_t<6, 16>(P, batch, smem, s);
  return launch_tail_backward_t<0, 0>(P, batch, smem, s);
}


/* ------------------------------------------------------------------------------------------
 * Decoder trunk stages (sdfest/vae/sdf_vae.py:225-247): per stage
 *     interpolate(x -> in_size^3, trilinear, align_corners=False)      -> the tail kernels above with
 *                                                                         weight = NULL (C = 1)
 *     Conv3d(Ci -> Co, kernel_size=3), + bias, optional ReLU           -> sdfr_conv3_kernel
 * and the data gradient of the convolution (the decoder is frozen: no weight gradients).
 * Every shipped decoder (vae/configs/*.yaml, initialization/configs/vae_models/*.yaml) uses 3x3x3
 * "valid" convolutions with 4..32 channels on 8^3..32^3 volumes: ~37 MFLOP-pairs per hypothesis, for
 * which cuDNN picks kernels that take 1.5 ms per layer and direction at 64 hypotheses
 * (profiles/r01g_decoder_ops.txt).  Direct fp32 convolution: a CTA owns a 4 x 8 x (8*ZR) tile of
 * output positions for ALL output channels, input tile + weights staged in shared memory 4 input
 * channels at a time, each thread accumulating CO x ZR outputs (a run of ZR consecutive z) in
 * registers: per (ci, dx, dy) it reads ZR+2 inputs and 3*CO broadcast weights for 3*ZR*CO FFMAs.
 * DGRAD = true computes the transposed convolution with the same code: input = grad_out (times the
 * ReLU mask y > 0) shifted by K-1 with zero padding, weights flipped and channel-transposed while
 * they are staged.
 * ---------------------------------------------------------------------------------------- */
struct ConvParams {
  const float* __restrict__ in;   /* fwd: x [B,CI,n_in^3];  dgrad: grad_y [B,CI,n_in^3] */
  const float* __restrict__ mask; /* dgrad: y [B,CI,n_in^3] (ReLU mask y > 0) or NULL */
  const float* __restrict__ w;    /* [Co_orig, Ci_orig, 27] as torch stores it */
  const float* __restrict__ bias; /* fwd: [CO] or NULL */
  float* __restrict__ out;        /* fwd: y [B,CO,n_out^3];  dgrad: grad_x [B,CO,n_out^3] */
  int CI, n_in, n_out, relu;
  int tiles_y, tiles_z;
  int z_offset;
  int cc; /* channels staged per pass = min(CI, ConvTile::CC) */
  int co_total; /* output channels of the launch; a CTA computes CO of them starting at blockIdx.z * CO */
};

/* Shared-memory geometry of one CTA: CC input channels of the (TX+2) x (TY+2) x (TZ+2) input tile,
 * z-pitch PZ a multiple of 4 floats so that staging and the inner loop use 128 / 64-bit accesses. */
template <int CO, int ZR>
struct ConvTile {
  static constexpr int K = 3, TX = 4, TY = 8, TZ = 8 * ZR;
  /* channels staged per pass: the tile must leave room for >= 3 CTAs per SM */
  static constexpr int CC = 8;
  static constexpr int IX = TX + K - 1, IY = TY + K - 1, IZ = TZ + K - 1;
  static constexpr int PZ = ((IZ + 3) / 4) * 4;
  static constexpr int CH = IX * IY * PZ; /* floats per staged channel */
  static size_t bytes(int cc) { return sizeof(float) * (size_t)cc * (CH + 27 * CO); }
};

/* VEC = floats per staging access: 4 (forward, n_in % 4 == 0), 2 (n_in even: every dgrad of a
 * decoder whose stage sizes are even), 1 (anything).  A staging "slot" is VEC consecutive z of one
 * (channel, x, y) row of the tile; every slot of the tile is written (zero outside the volume),
 * so there is no separate clearing pass.  First version: per-element staging with 2 slots per
 * thread and plane -- ~29 instructions per element, 43 % of all instructions executed
 * (profiles/r01j_ncu_decoder.txt: 127 M warp instructions for 56 M warp-FFMAs). */
/* KS > 1: a thread-block cluster of KS CTAs (cluster dims (1,1,KS)) splits the INPUT channels of one
 * tile; the partial sums meet in the leader's shared memory over DSMEM.  For the smallest stage
 * (8^3 -> 6^3: 2 tiles per volume, 128 CTAs of 9 k instructions per thread at 64 hypotheses --
 * one CTA per SM, latency-bound at 8 warps) this quadruples the resident warps without shrinking
 * the per-thread accumulator block (splitting the OUTPUT channels instead was measured slower). */
/* A thread computing two adjacent output rows, sharing their input rows and weights, was measured slower
 * (8 -> 4 channel stage: 118.8 against 100.4 us, profiles/r02ad_conv_ffma2_ab.json). */
template <int CO, int ZR, bool DGRAD, int VEC, int KS = 1>
__global__ void __launch_bounds__(256, (CO * ZR <= 16 ? 4 : (CO * ZR <= 32 ? 3 : (CO * ZR <= 64 ? 2 : 1))))
sdfr_conv3_kernel(const __grid_constant__ ConvParams P) {
  using T = ConvTile<CO, ZR>;
  constexpr int K = 3, TX = T::TX, TY = T::TY, TZ = T::TZ, CC = T::CC;
  constexpr int IX = T::IX, IY = T::IY, PZ = T::PZ;
  extern __shared__ __align__(16) float conv_smem[];
  float* __restrict__ tile = conv_smem;          /* [CC][IX][IY][PZ] */
  float* __restrict__ ws = conv_smem + P.cc * T::CH;  /* [CC][27][CO] */

  const int b = blockIdx.y + P.z_offset;
  const int kr = KS > 1 ? (int)(blockIdx.z % KS) : 0; /* rank in the cluster = input-channel slice */
  const int co0 = (int)(blockIdx.z / KS) * CO, COT = P.co_total;
  int t = blockIdx.x;
  const int tz = t % P.tiles_z; t /= P.tiles_z;
  const int tyy = t % P.tiles_y;
  const int txx = t / P.tiles_y;
  const int X0 = txx * TX, Y0 = tyy * TY, Z0 = tz * TZ;
  const int zr = threadIdx.x & 7, ly = (threadIdx.x >> 3) & 7, lx = threadIdx.x >> 6;
  const int z0 = zr * ZR;
  const int n_in = P.n_in, n_out = P.n_out, CI = P.CI;
  const size_t in_vol = (size_t)n_in * n_in * n_in;
  constexpr int shift = DGRAD ? K - 1 : 0; /* input coordinate = output coordinate + tap - shift */

  /* Accumulators as float2 pairs over adjacent output channels: the weight vector of a tap arrives as
   * float4 = two aligned channel pairs, the input value is duplicated into a pair once per row, and every
   * multiply-add is one FFMA2 (fma.rn.f32x2, sm_100) -- two IEEE fp32 fmas per issue slot and per fma-pipe
   * cycle, bit-identical to scalar FFMAs. */
  float2 acc2[CO / 2][ZR];
#pragma unroll
  for (int c2 = 0; c2 < CO / 2; ++c2)
#pragma unroll
    for (int i = 0; i < ZR; ++i) acc2[c2][i] = make_float2(0.0f, 0.0f);

  const int ci_begin = kr * (CI / KS), ci_end = ci_begin + CI / KS; /* CI % KS == 0 (launcher) */
  for (int ci0 = ci_begin; ci0 < ci_end; ci0 += CC) {
    const int nc = ci_end - ci0 < CC ? ci_end - ci0 : CC;
    /* stage the input tile */
    constexpr int SL = PZ / VEC; /* slots per row */
    const int n_slots = nc * IX * IY * SL;
    const float* __restrict__ src = P.in + ((size_t)b * CI + ci0) * in_vol;
    const float* __restrict__ msk = (DGRAD && P.mask) ? P.mask + ((size_t)b * CI + ci0) * in_vol : nullptr;
    for (int e = threadIdx.x; e < n_slots; e += 256) {
      const int row = e / SL, j = (e - row * SL) * VEC;
      const int c = row / (IX * IY), r2 = row - c * (IX * IY);
      const int x = r2 / IY, y = r2 - x * IY;
      const int gx = X0 + x - shift, gy = Y0 + y - shift, gz = Z0 + j - shift;
      const bool ok = gx >= 0 && gx < n_in && gy >= 0 && gy < n_in && gz >= 0 && gz < n_in;
      const size_t g = (size_t)c * in_vol + ((size_t)gx * n_in + gy) * n_in + gz;
      float* __restrict__ d = tile + ((c * IX + x) * IY + y) * PZ + j;
      if constexpr (VEC == 4) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) {
          v = __ldg(reinterpret_cast<const float4*>(src + g));
          if (msk) {
            const float4 m = __ldg(reinterpret_cast<const float4*>(msk + g));
            v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f;
            v.z = m.z > 0.f ? v.z : 0.f; v.w = m.w > 0.f ? v.w : 0.f;
          }
        }
        *reinterpret_cast<float4*>(d) = v;
      } else if constexpr (VEC == 2) {
        float2 v = make_float2(0.f, 0.f);
        if (ok) {
          v = __ldg(reinterpret_cast<const float2*>(src + g));
          if (msk) {
            const float2 m = __ldg(reinterpret_cast<const float2*>(msk + g));
            v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f;
          }
        }
        *reinterpret_cast<float2*>(d) = v;
      } else {
        float v = 0.f;
        if (ok) {
          v = __ldg(src + g);
          if (msk) v = __ldg(msk + g) > 0.f ? v : 0.f;
        }
        *d = v;
      }
    }
    /* stage the weights of these input channels as [c][tap][co] */
    for (int e = threadIdx.x; e < nc * 27 * CO; e += 256) {
      const int co = e % CO;
      const int tap = (e / CO) % 27;
      const int c = e / (CO * 27);
      float v;
      if (!DGRAD) v = __ldg(P.w + ((size_t)(co0 + co) * CI + ci0 + c) * 27 + tap);
      else v = __ldg(P.w + ((size_t)(ci0 + c) * COT + co0 + co) * 27 + (26 - tap)); /* w[co_orig = in ch][ci_orig = out ch], flipped */
      ws[e] = v;
    }
    __syncthreads();
    /* one row per (dx, dy) at a time: loading the three rows of a dx up front costs the 8 -> 4 channel
     * stage 12 us -- more live registers, later first FFMA */
    for (int c = 0; c < nc; ++c) {
#pragma unroll
      for (int dx = 0; dx < K; ++dx) {
#pragma unroll
        for (int dy = 0; dy < K; ++dy) {
          float v[ZR + K - 1];
          const float* __restrict__ row = tile + ((c * IX + lx + dx) * IY + ly + dy) * PZ + z0;
          if constexpr (ZR == 4) {
            const float4 a = *reinterpret_cast<const float4*>(row);
            const float2 e2 = *reinterpret_cast<const float2*>(row + 4);
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = e2.x; v[5] = e2.y;
          } else if constexpr (ZR == 2) {
            const float2 a = *reinterpret_cast<const float2*>(row);
            const float2 e2 = *reinterpret_cast<const float2*>(row + 2);
            v[0] = a.x; v[1] = a.y; v[2] = e2.x; v[3] = e2.y;
          } else {
#pragma unroll
            for (int i = 0; i < ZR + K - 1; ++i) v[i] = row[i];
          }
          float2 vv[ZR + K - 1];
#pragma unroll
          for (int i = 0; i < ZR + K - 1; ++i) vv[i] = make_float2(v[i], v[i]);
#pragma unroll
          for (int dz = 0; dz < K; ++dz) {
            const float4* __restrict__ wp =
                reinterpret_cast<const float4*>(ws + (c * 27 + (dx * K + dy) * K + dz) * CO);
#pragma unroll
            for (int c4 = 0; c4 < CO / 4; ++c4) {
              const float4 w4 = wp[c4];
              const float2 wa = make_float2(w4.x, w4.y), wb = make_float2(w4.z, w4.w);
#pragma unroll
              for (int i = 0; i < ZR; ++i) {
                acc2[2 * c4 + 0][i] = __ffma2_rn(wa, vv[i + dz], acc2[2 * c4 + 0][i]);
                acc2[2 * c4 + 1][i] = __ffma2_rn(wb, vv[i + dz], acc2[2 * c4 + 1][i]);
              }
            }
          }
        }
      }
    }
    if (ci0 + CC < ci_end) __syncthreads();
  }

  if constexpr (KS > 1) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __syncthreads(); /* everyone is done with the tile: its memory becomes the exchange buffer */
    float* red = conv_smem; /* [CO * ZR][256] */
    if (kr != 0) {
#pragma unroll
      for (int co = 0; co < CO; ++co)
#pragma unroll
        for (int i = 0; i < ZR; ++i)
          red[(co * ZR + i) * 256 + threadIdx.x] = (co & 1) ? acc2[co >> 1][i].y : acc2[co >> 1][i].x;
    }
    cluster.sync();
    if (kr == 0) {
      for (int r = 1; r < KS; ++r) {
        const float* __restrict__ peer = cluster.map_shared_rank(red, r);
#pragma unroll
        for (int c2 = 0; c2 < CO / 2; ++c2)
#pragma unroll
          for (int i = 0; i < ZR; ++i) {
            acc2[c2][i].x += peer[(2 * c2 * ZR + i) * 256 + threadIdx.x];
            acc2[c2][i].y += peer[((2 * c2 + 1) * ZR + i) * 256 + threadIdx.x];
          }
      }
    }
    cluster.sync(); /* peers keep their shared memory alive until the leader has read it */
    if (kr != 0) return;
  }

  const int ox = X0 + lx;
  if (ox >= n_out) return;
  const size_t out_vol = (size_t)n_out * n_out * n_out;
  const int oy = Y0 + ly;
  if (oy >= n_out) return;
#pragma unroll
  for (int co = 0; co < CO; ++co) {
    const float bias = (!DGRAD && P.bias) ? __ldg(P.bias + co0 + co) : 0.0f;
    float* __restrict__ o = P.out + ((size_t)b * COT + co0 + co) * out_vol + ((size_t)ox * n_out + oy) * n_out;
#pragma unroll
    for (int i = 0; i < ZR; ++i) {
      const int oz = Z0 + z0 + i;
      if (oz < n_out) {
        float v = ((co & 1) ? acc2[co >> 1][i].y : acc2[co >> 1][i].x) + bias;
        if (!DGRAD && P.relu) v = v > 0.0f ? v : 0.0f;
        o[oz] = v;
      }
    }
  }
}

template <int CO, int ZR, bool DGRAD, int VEC, int KS = 1>
int launch_conv3_v(ConvParams P, int batch, cudaStream_t s) {
  using T = ConvTile<CO, ZR>;
  const int tiles_x = (P.n_out + T::TX - 1) / T::TX;
  P.tiles_y = (P.n_out + T::TY - 1) / T::TY;
  P.tiles_z = (P.n_out + T::TZ - 1) / T::TZ;
  const int per_cta = P.CI / KS;
  P.cc = per_cta < T::CC ? per_cta : T::CC;
  size_t smem = T::bytes(P.cc);
  if (KS > 1 && smem < sizeof(float) * CO * ZR * 256) smem = sizeof(float) * CO * ZR * 256;
  auto kernel = sdfr_conv3_kernel<CO, ZR, DGRAD, VEC, KS>;
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "conv3d: shared memory opt-in failed");
  }
  for (int z0 = 0; z0 < batch; z0 += 65535) {
    P.z_offset = z0;
    const dim3 grid(tiles_x * P.tiles_y * P.tiles_z, batch - z0 < 65535 ? batch - z0 : 65535,
                    (P.co_total / CO) * KS);
    if (KS == 1) {
      kernel<<<grid, 256, smem, s>>>(P);
    } else {
      cudaLaunchConfig_t cfg;
      memset(&cfg, 0, sizeof(cfg));
      cfg.gridDim = grid;
      cfg.blockDim = dim3(256);
      cfg.dynamicSmemBytes = smem;
      cfg.stream = s;
      cudaLaunchAttribute attr;
      attr.id = cudaLaunchAttributeClusterDimension;
      attr.val.clusterDim.x = 1;
      attr.val.clusterDim.y = 1;
      attr.val.clusterDim.z = KS;
      cfg.attrs = &attr;
      cfg.numAttrs = 1;
      const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, P);
      if (e != cudaSuccess) return fail((int)e, "conv3d: cluster launch failed");
    }
  }
  return 0;
}

/* widest staging access the operands allow: rows start at multiples of n_in elements and tiles at
 * multiples of 8 (minus 2 for dgrad), so alignment follows from n_in and the base pointers */
template <int CO, int ZR, bool DGRAD>
int launch_conv3_t(const ConvParams& P, int batch, cudaStream_t s) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(P.in) | reinterpret_cast<uintptr_t>(P.mask);
  if constexpr (ZR == 1 && CO <= 16) {
    /* smallest stage, too few tiles to fill the SMs: 4-CTA clusters over the input channels */
    const long ctas = (long)((P.n_out + 3) / 4) * ((P.n_out + 7) / 8) * ((P.n_out + 7) / 8) * batch *
                      (P.co_total / CO);
    if (P.CI % 16 == 0 && ctas < 296) {
      if (!DGRAD && P.n_in % 4 == 0 && (a & 15) == 0) return launch_conv3_v<CO, ZR, DGRAD, DGRAD ? 2 : 4, 4>(P, batch, s);
      if (P.n_in % 2 == 0 && (a & 7) == 0) return launch_conv3_v<CO, ZR, DGRAD, 2, 4>(P, batch, s);
    }
  }
  if constexpr (!DGRAD)
    if (P.n_in % 4 == 0 && (a & 15) == 0) return launch_conv3_v<CO, ZR, DGRAD, 4>(P, batch, s);
  if (P.n_in % 2 == 0 && (a & 7) == 0) return launch_conv3_v<CO, ZR, DGRAD, 2>(P, batch, s);
  return launch_conv3_v<CO, ZR, DGRAD, 1>(P, batch, s);
}

/* z-extent of the CTA tile (8 * ZR) follows the volume: 32 for n_out > 16, 16 for > 8, else 8 --
 * a 14^3 output in 32-deep tiles would leave 56 % of the lanes idle */
template <int CO, bool DGRAD>
int launch_conv3_zr(const ConvParams& P, int batch, cudaStream_t s) {
  if (P.n_out > 16 && CO <= 16) return launch_conv3_t<CO, (CO <= 16 ? 4 : 2), DGRAD>(P, batch, s);
  if (P.n_out > 8) return launch_conv3_t<CO, 2, DGRAD>(P, batch, s);
  return launch_conv3_t<CO, 1, DGRAD>(P, batch, s);
}

/* CO = output channels of THIS launch (forward: Co; dgrad: Ci of the layer) */
template <bool DGRAD>
int launch_conv3(ConvParams P, int CO, int batch, cudaStream_t s) {
  int rc = 0;
  P.co_total = CO;
  if (P.n_out <= 8) {
    /* the smallest stage (8^3 -> 6^3 in every shipped decoder) has 2 tiles per volume; with few
     * hypotheses the output channels are split over blockIdx.z to fill the SMs.  (At 64 hypotheses
     * = 128 CTAs splitting was measured SLOWER, 33 -> 41 us: 4 accumulators per thread starve the FMA
     * pipe; the stage is latency-bound at 8 warps per SM, not CTA-count-bound.) */
    const long tiles = (long)((P.n_out + 3) / 4) * batch;
    while (CO > 8 && tiles * (P.co_total / CO) < 74) CO /= 2;
  }
  switch (CO) {
    case 4: rc = launch_conv3_zr<4, DGRAD>(P, batch, s); break;
    case 8: rc = launch_conv3_zr<8, DGRAD>(P, batch, s); break;
    case 16: rc = launch_conv3_zr<16, DGRAD>(P, batch, s); break;
    case 32: rc = launch_conv3_zr<32, DGRAD>(P, batch, s); break;
    default:
      return fail(SDFR_E_SHAPE, "conv3d: this launch's output channels must be 4, 8, 16 or 32");
  }
  return rc ? rc : check_launch("sdfr_conv3_kernel");
}

#endif /* SDFR_DECODER_CUH_ */
