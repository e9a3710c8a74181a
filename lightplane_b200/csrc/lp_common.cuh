// Device-side building blocks shared by all kernels of the hot path: grid-list addressing
// (tri/bi-linear taps), the depth schedule, coordinate contraction, activations, the hash RNG and the gradient w.r.t.
// a sample's position.
// Every function cites the reference lines whose semantics it implements
// (paths relative to facebookresearch/lightplane).
#pragma once

#include "../../include/lightplane_b200.h"
#include "lp_platform.cuh"

// ---------------------------------------------------------------------------------------------
// Kernel-parameter structs (built on the host in lp_cabi.cu, passed by value)
// ---------------------------------------------------------------------------------------------
enum LpGridKind { LP_VOXEL = 0, LP_PLANE_XY = 1, LP_PLANE_XZ = 2, LP_PLANE_YZ = 3 };

struct LpGrid {
  int B, D, H, W;
  int kind;
  int pad_;
  long long base;  // element offset of this grid inside the flat tensor
};

struct LpGridSet {
  float* data;  // flat [rows, C]
  int n;
  int C;
  int tri;      // 1: g[0..2] are the XY, XZ, YZ planes of one W x H x D volume, in this order (the kernels' triplane fast path)
  int pad_;
  LpGrid g[LP_MAX_GRIDS];
};

struct LpRays {
  const float* dir;
  const float* org;
  const int* gidx;
  const float* near;
  const float* far;
  const float* enc;
  int n;
  int enc_dim;
};

struct LpMarch {
  int S, S_inf;
  float gain, disparity_at_inf;
  int mask_oob, contract;
  int noise;
  float sigma;
  int seed, noise_num_rays;
  int img_w;  // > 0: rays form a row-major image of this width, walked in 16x8-pixel tiles (validated on the host)
};

// One dense layer inside the flat parameter vector.
struct LpLayer {
  int w_off, b_off;  // offsets (floats) into mlp_params
  int K, N;          // rows / row stride of W (y = x@W + b)
  int n_used;        // columns actually evaluated (== N except for the padded colour head)
  int relu;          // ReLU after this layer
};

struct LpMlp {
  int n_layers;
  LpLayer l[LP_MAX_LAYERS];
};

// ---------------------------------------------------------------------------------------------
// activations (reference: triton_src/shared/func_util.py:13-29)
// ---------------------------------------------------------------------------------------------
LP_DEVICE float lp_softplus(float x) {  // log(1+exp(x)), stable form of func_util.py:19-22
  return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x)));
}
LP_DEVICE float lp_sigmoid(float x) {  // also d/dx softplus (func_util.py:25-28)
  if (x >= 0.f) return 1.f / (1.f + expf(-x));
  float e = expf(x);
  return e / (1.f + e);
}

// ---------------------------------------------------------------------------------------------
// depth schedule (reference: triton_src/shared/ray_util.py:47-58; renderer_fw.py:209-226)
// ---------------------------------------------------------------------------------------------
// Depth of sample `step` in [-1, S+S_inf).  step == -1 extrapolates below `near` so that
// delta_0 = (far-near)/(S-1) (1 when S == 1, naive_renderer.py:252-256); step in [S, S+S_inf)
// are the background samples far / ((d_inf-1)(k+1)/S_inf + 1), k = step - S, with k == -1 giving
// `far`.  1/n_disp is evaluated as 1 / ((1-f) + d_inf*f) to avoid the fp32 cancellation of
// (d_inf-1)*f + 1 near f = 1 (the naive reference evaluates it in double, naive_renderer.py:810-813).
LP_DEVICE float lp_depth(int step, float near, float far, int S, int S_inf, float d_inf) {
  if (step < S) {
    if (S <= 1) return step < 0 ? near - 1.f : near;
    float frac = (float)step / (float)(S - 1);
    return (far - near) * frac + near;
  }
  int k = step - S;  // 0..S_inf-1
  float f = (float)(k + 1) / (float)S_inf;
  float one_minus_f = (float)(S_inf - (k + 1)) / (float)S_inf;
  float n_disp = one_minus_f + d_inf * f;
  return far * (1.f / n_disp);
}
// Step length of sample `step`: depth(step) - depth(step-1) as the reference's NAIVE path forms it (depths.diff(),
// naive_renderer.py:252-257): with S == 1 the depth before the first background sample is depth_0 = near.  (The
// reference's Triton kernels use `far` there, depth_inv_sphere(..., -1); for S > 1 both agree since depth_{S-1} = far.
// Like for the background schedule itself -- DESIGN.md section 2 -- this implementation follows the naive semantics.)
LP_DEVICE float lp_delta(int step, float depth, float near, float far, int S, int S_inf, float d_inf) {
  return depth - lp_depth(step - 1, near, far, S, S_inf, d_inf);
}

// MERF contraction then x0.5 (ray_util.py:12-45).
LP_DEVICE float lp_contract_one(float v, float n) {
  float out = v;
  if (n > 1.f) {
    float a = fabsf(v);
    if (fabsf(a - n) <= 1e-8f) out = (2.f - 1.f / a) * (v / a);
    else out = v / n;
  }
  return out * 0.5f;
}
LP_DEVICE void lp_contract(float& x, float& y, float& z) {
  float n = fmaxf(fmaxf(fabsf(x), fabsf(y)), fabsf(z));
  x = lp_contract_one(x, n);
  y = lp_contract_one(y, n);
  z = lp_contract_one(z, n);
}
LP_DEVICE float lp_in_bounds(float x, float y, float z) {  // grid_sample_util.py:22-37
  return (fabsf(x) <= 1.f && fabsf(y) <= 1.f && fabsf(z) <= 1.f) ? 1.f : 0.f;
}

// ---------------------------------------------------------------------------------------------
// hash RNG (reference: triton_src/shared/rand_util.py:38-79), int32 wrap-around arithmetic
// ---------------------------------------------------------------------------------------------
LP_DEVICE int lp_hash32(int x) {
  x = (int)((unsigned)((x >> 16) ^ x) * 0x45D9F3Bu);
  x = (int)((unsigned)((x >> 16) ^ x) * 0x45D9F3Bu);
  return (x >> 16) ^ x;
}
LP_DEVICE int lp_pair_hash32(int x, int h) {
  unsigned u = (unsigned)(h ^ x);
  return (int)((u << 24) + u * 0x193u);
}
LP_DEVICE float lp_int_to_01(int x) {
  return (((float)x + 2147483647.0f) + 3.0f) / 4294967298.0f;
}
LP_DEVICE float lp_int_to_randn(int x1, int x2, int seed) {
  int h1 = lp_pair_hash32(lp_pair_hash32(105097564, seed), lp_hash32(x1));
  int h2 = lp_pair_hash32(lp_pair_hash32(105097564, (int)((unsigned)seed + 1u)), lp_hash32(x2));
  float u1 = lp_int_to_01(h1), u2 = lp_int_to_01(h2);
  return sqrtf(-2.f * logf(u1)) * cosf(6.28318530718f * u2);
}
// noise of sample `step` of ray `ray` (fwbw_util.py:66-70; renderer_fw.py:289-296)
// (not inlined: logf + large-argument cosf are long code sequences and the callers are unrolled)
static __device__ __noinline__ float lp_sample_noise(const LpMarch& m, int ray, int step) {
  int tot = m.S + m.S_inf;
  int i1 = (int)((unsigned)ray * (unsigned)tot + (unsigned)step + 1u);
  int i2 = (int)((unsigned)i1 + (unsigned)m.noise_num_rays * (unsigned)tot);
  return lp_int_to_randn(i1, i2, m.seed);
}

// ---------------------------------------------------------------------------------------------
// taps of one grid (reference: grid_sample_util.py:209-333 sample info + corner order,
// :638-714 clamp + validity mask = zero padding, :1111-1173 grid classification)
// ---------------------------------------------------------------------------------------------
// Continuous index along one axis (align_corners=False); singleton axes are pinned to 0.
LP_DEVICE void lp_axis(float p, int size, float& i0, float& frac) {
  float i = ((p + 1.f) * 0.5f) * (float)size - 0.5f;
  if (size <= 1) i = 0.f;
  i0 = floorf(i);
  frac = i - i0;
}
LP_DEVICE void lp_corner(float i0, float frac, int hi, int size, float& w, int& idx) {
  float ia = i0 + (float)hi;
  float ww = hi ? frac : 1.f - frac;
  bool ok = (ia >= 0.f) && (ia < (float)size);
  w = ok ? ww : 0.f;
  idx = (int)fminf(fmaxf(ia, 0.f), (float)(size - 1));
}

// Computes the taps of grid `g` for point (x,y,z) of batch element b.  `off` = element offsets of
// the C-channel rows inside the flat tensor, `w` = interpolation weights (0 for taps outside the
// grid).  Returns the number of taps (8 voxel / 4 plane).
LP_DEVICE int lp_taps(const LpGrid& g, int C, int b, float x, float y, float z, long long* off,
                      float* w) {
  if (g.kind == LP_VOXEL) {
    float x0, fx, y0, fy, z0, fz;
    lp_axis(x, g.W, x0, fx);
    lp_axis(y, g.H, y0, fy);
    lp_axis(z, g.D, z0, fz);
    long long bbase = g.base + (long long)b * g.D * g.H * g.W * C;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float wx, wy, wz;
      int ix, iy, iz;
      lp_corner(x0, fx, c & 1, g.W, wx, ix);
      lp_corner(y0, fy, (c >> 1) & 1, g.H, wy, iy);
      lp_corner(z0, fz, (c >> 2) & 1, g.D, wz, iz);
      w[c] = wx * wy * wz;
      off[c] = bbase + ((long long)(iz * g.H + iy) * g.W + ix) * C;
    }
    return 8;
  }
  // planes: (u -> fastest axis U, v -> slower axis V)
  float u, v;
  int U, V;
  if (g.kind == LP_PLANE_XY) { u = x; v = y; U = g.W; V = g.H; }
  else if (g.kind == LP_PLANE_XZ) { u = x; v = z; U = g.W; V = g.D; }
  else { u = y; v = z; U = g.H; V = g.D; }
  float u0, fu, v0, fv;
  lp_axis(u, U, u0, fu);
  lp_axis(v, V, v0, fv);
  long long bbase = g.base + (long long)b * U * V * C;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float wu, wv;
    int iu, iv;
    lp_corner(u0, fu, c & 1, U, wu, iu);
    lp_corner(v0, fv, (c >> 1) & 1, V, wv, iv);
    w[c] = wu * wv;
    off[c] = bbase + ((long long)iv * U + iu) * C;
  }
  return 4;
}

// ---------------------------------------------------------------------------------------------
// gradient w.r.t. the sample position (ray-geometry gradients of lp_render_backward_rays)
// ---------------------------------------------------------------------------------------------
// One axis of lp_axis / lp_corner with the derivative of both corner weights w.r.t. the coordinate: d frac / d p =
// size / 2, 0 on pinned singleton axes; a corner outside the grid has weight and derivative 0 (zero padding).
LP_DEVICE void lp_axis_d(float p, int size, float (&w)[2], float (&dw)[2], int (&idx)[2]) {
  float i0, frac;
  lp_axis(p, size, i0, frac);
  const float s = size > 1 ? 0.5f * (float)size : 0.f;
#pragma unroll
  for (int hi = 0; hi < 2; ++hi) {
    const float ia = i0 + (float)hi;
    const bool ok = (ia >= 0.f) && (ia < (float)size);
    w[hi] = ok ? (hi ? frac : 1.f - frac) : 0.f;
    dw[hi] = ok ? (hi ? s : -s) : 0.f;
    idx[hi] = (int)fminf(fmaxf(ia, 0.f), (float)(size - 1));
  }
}

// Gradient w.r.t. the grid-space point (x,y,z) of sum over the grids of G and their taps t of w_t(x,y,z) <v_t, a>, i.e.
// sum_t <v_t, a> grad w_t, for the sampled-feature gradient a of one sample.  `dot(row)` returns <row, a> for the C
// floats of a texel row; it is called only for taps whose weight gradient is non-zero.  Adds into (gx, gy, gz).
template <class Dot>
LP_DEVICE void lp_pos_grad(const LpGridSet& G, int b, float x, float y, float z, const Dot& dot, float& gx, float& gy,
                           float& gz) {
  const int C = G.C;
  for (int gi = 0; gi < G.n; ++gi) {
    const LpGrid& g = G.g[gi];
    if (g.kind == LP_VOXEL) {
      float wx[2], dwx[2], wy[2], dwy[2], wz[2], dwz[2];
      int ix[2], iy[2], iz[2];
      lp_axis_d(x, g.W, wx, dwx, ix);
      lp_axis_d(y, g.H, wy, dwy, iy);
      lp_axis_d(z, g.D, wz, dwz, iz);
      const long long bbase = g.base + (long long)b * g.D * g.H * g.W * C;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int i = c & 1, j = (c >> 1) & 1, k = c >> 2;
        const float ex = dwx[i] * wy[j] * wz[k], ey = wx[i] * dwy[j] * wz[k], ez = wx[i] * wy[j] * dwz[k];
        if (ex != 0.f || ey != 0.f || ez != 0.f) {
          const float d = dot(G.data + bbase + ((long long)(iz[k] * g.H + iy[j]) * g.W + ix[i]) * C);
          gx = fmaf(d, ex, gx); gy = fmaf(d, ey, gy); gz = fmaf(d, ez, gz);
        }
      }
      continue;
    }
    // planes: (u -> fastest axis U, v -> slower axis V), as lp_taps
    float u, v;
    int U, V;
    if (g.kind == LP_PLANE_XY) { u = x; v = y; U = g.W; V = g.H; }
    else if (g.kind == LP_PLANE_XZ) { u = x; v = z; U = g.W; V = g.D; }
    else { u = y; v = z; U = g.H; V = g.D; }
    float wu[2], dwu[2], wv[2], dwv[2];
    int iu[2], iv[2];
    lp_axis_d(u, U, wu, dwu, iu);
    lp_axis_d(v, V, wv, dwv, iv);
    const long long bbase = g.base + (long long)b * U * V * C;
    float gu = 0.f, gv = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int i = c & 1, j = c >> 1;
      const float eu = dwu[i] * wv[j], ev = wu[i] * dwv[j];
      if (eu != 0.f || ev != 0.f) {
        const float d = dot(G.data + bbase + ((long long)iv[j] * U + iu[i]) * C);
        gu = fmaf(d, eu, gu); gv = fmaf(d, ev, gv);
      }
    }
    if (g.kind == LP_PLANE_XY) { gx += gu; gy += gv; }
    else if (g.kind == LP_PLANE_XZ) { gx += gu; gz += gv; }
    else { gy += gu; gz += gv; }
  }
}

// Vector-Jacobian product of lp_contract at the pre-contraction point p: (gx, gy, gz), the gradient w.r.t. the
// contracted point, becomes J_c(p)^T g.  Differentiated as autograd differentiates the MERF formula: a coordinate on the
// max-norm n maps through (2 - 1/a) sign(v) -> 0.5 / a^2; the others through v / n -> 0.5 / n, plus -0.5 v / n^2 via n,
// which reaches the coordinate(s) at the maximum (shared evenly between ties, like the gradient of a max).
LP_DEVICE void lp_contract_vjp(float px, float py, float pz, float& gx, float& gy, float& gz) {
  const float ax = fabsf(px), ay = fabsf(py), az = fabsf(pz);
  const float n = fmaxf(fmaxf(ax, ay), az);
  if (!(n > 1.f)) { gx *= 0.5f; gy *= 0.5f; gz *= 0.5f; return; }
  float gn = 0.f;
  auto one = [&](float v, float a, float& g) {
    if (fabsf(a - n) <= 1e-8f) {
      g = 0.5f * g / (a * a);
    } else {
      gn -= 0.5f * g * v / (n * n);
      g = 0.5f * g / n;
    }
  };
  one(px, ax, gx); one(py, ay, gy); one(pz, az, gz);
  const float kx = ax == n ? 1.f : 0.f, ky = ay == n ? 1.f : 0.f, kz = az == n ? 1.f : 0.f;
  const float share = gn / (kx + ky + kz);
  gx += kx * (px < 0.f ? -share : share); gy += ky * (py < 0.f ? -share : share); gz += kz * (pz < 0.f ? -share : share);
}

// Nearest-neighbour lookup of a 1-channel voxel grid with zero padding and an additional
// in-bounds mask (scaffold).  Rounding: to nearest, ties to even, as `F.grid_sample(mode="nearest")` of the reference's
// naive path (naive_renderer.py:568-589); its Triton kernels round ties up (floor(x + 0.5), grid_sample_util.py:717-777) --
// the two differ only for coordinates exactly half-way between two cells.
LP_DEVICE float lp_nearest(const LpGridSet& s, int b, float x, float y, float z) {
  const LpGrid& g = s.g[0];
  float ix = ((x + 1.f) * 0.5f) * (float)g.W - 0.5f;
  float iy = ((y + 1.f) * 0.5f) * (float)g.H - 0.5f;
  float iz = ((z + 1.f) * 0.5f) * (float)g.D - 0.5f;
  if (g.W <= 1) ix = 0.f;
  if (g.H <= 1) iy = 0.f;
  if (g.D <= 1) iz = 0.f;
  ix = rintf(ix); iy = rintf(iy); iz = rintf(iz);
  bool ok = ix >= 0.f && ix < (float)g.W && iy >= 0.f && iy < (float)g.H && iz >= 0.f && iz < (float)g.D;
  if (!ok) return 0.f;
  long long o = g.base + (((long long)b * g.D + (int)iz) * g.H + (int)iy) * g.W + (int)ix;
  return __ldg(s.data + o) * lp_in_bounds(x, y, z);
}
