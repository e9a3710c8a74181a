// Generic Renderer kernels: any layer counts / widths, colour-grid mode, scaffold, noise,
// background samples, contraction.  One lane = one ray; per-sample activations live in shared
// memory as [feature][lane] (lane stride 33 -> conflict-free both for lane-local column access and
// for the warp-cooperative dW reduction); MLP weights are read as warp-uniform broadcasts from a
// shared-memory copy of `mlp_params`.  This is the coverage kernel; the specialised tensor-core
// kernel for the default decoder shape lives in lp_render_fast.cuh.
//
// Semantics restated from the reference: renderer_fw.py:85-375 (forward march + compositing),
// renderer_bw.py:89-627 (analytic compositing gradient; marched in forward order here, see
// include/lightplane_b200.h lp_render_backward),
// renderer_mlp_util.py:100-178 (MLP forward / backward), grid_sample_util.py (taps).
#pragma once

#include "lp_common.cuh"

#define LP_LS 33  // lane stride of [feature][lane] shared-memory tiles

struct LpDecoder {
  LpMlp trunk, opacity, color;
  int n_params;
  int C;               // grid channels
  int in_c;            // colour-head input width == ray-encoding width
  int n_feat;          // colour channels rendered
  int use_color_grid;  // relu-field mode (no trunk)
  int max_dim;         // max width of any activation vector
};

// Slots (in units of LP_LS floats) of the per-warp activation arena used by the backward pass.
struct LpActMap {
  int x0;                   // sampled grid feature (relu'd in colour-grid mode)      [C]
  int xcs;                  // colour-grid mode: relu(sampled colour feature)         [C]
  int xc;                   // colour-head input = trunk (or xcs) + ray encoding      [in_c]
  int yt[LP_MAX_LAYERS];    // trunk layer outputs (post-ReLU)
  int yo[LP_MAX_LAYERS];    // opacity hidden outputs (last = 1-wide raw opacity)
  int yc[LP_MAX_LAYERS];    // colour hidden outputs (last = n_feat-wide pre-sigmoid colour)
  int total;                // arena size in feature rows
};

// Pointers of the backward pass (forward outputs, upstream gradients, gradient outputs).
struct LpBwdIo {
  const float* len; const float* feat; int feat_stride;
  const float* g_len; const float* g_nlt; const float* g_feat; int g_feat_stride;
  float* g_grid; float* g_cgrid; float* g_params; float* g_enc;
  float* g_org; float* g_dir;  // [N,3] ray-geometry gradients (kernel instantiations with RAYG only; either may be NULL)
};

// Everything a renderer launch needs, built by lp_render_common() in lp_cabi.cu.
struct LpRenderArgs {
  LpRays R; LpMarch M; LpDecoder D; LpActMap A; LpGridSet G, CG, SC; int use_scaffold;
};

// -------------------------------------------------------------------------------------------
// lane-local dense layer:  out[j] = act(b[j] + sum_k in[k] * W[k][j]),  j < n_used
// -------------------------------------------------------------------------------------------
LP_DEVICE void lp_lane_linear(const float* __restrict__ P, const LpLayer& L, const float* in,
                              float* out, int lane) {
  const float* W = P + L.w_off;
  const float* Bv = P + L.b_off;
  const int n = L.n_used, N = L.N, K = L.K;
  for (int j0 = 0; j0 < n; j0 += 4) {
    const int j1 = min(j0 + 1, n - 1), j2 = min(j0 + 2, n - 1), j3 = min(j0 + 3, n - 1);
    float a0 = Bv[j0], a1 = Bv[j1], a2 = Bv[j2], a3 = Bv[j3];
    for (int k = 0; k < K; ++k) {
      const float x = in[k * LP_LS + lane];
      const float* wr = W + (long long)k * N;
      a0 = fmaf(x, wr[j0], a0);
      a1 = fmaf(x, wr[j1], a1);
      a2 = fmaf(x, wr[j2], a2);
      a3 = fmaf(x, wr[j3], a3);
    }
    if (L.relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); a2 = fmaxf(a2, 0.f); a3 = fmaxf(a3, 0.f); }
    out[j0 * LP_LS + lane] = a0;
    if (j0 + 1 < n) out[(j0 + 1) * LP_LS + lane] = a1;
    if (j0 + 2 < n) out[(j0 + 2) * LP_LS + lane] = a2;
    if (j0 + 3 < n) out[(j0 + 3) * LP_LS + lane] = a3;
  }
}

// lane-local input gradient: dx[k] = sum_{j<n_used} W[k][j] * dy[j]
LP_DEVICE void lp_lane_linear_dx(const float* __restrict__ P, const LpLayer& L, const float* dy,
                                 float* dx, int lane) {
  const float* W = P + L.w_off;
  const int n = L.n_used, N = L.N, K = L.K;
  for (int k0 = 0; k0 < K; k0 += 4) {
    const int k1 = min(k0 + 1, K - 1), k2 = min(k0 + 2, K - 1), k3 = min(k0 + 3, K - 1);
    const float *w0 = W + (long long)k0 * N, *w1 = W + (long long)k1 * N,
                *w2 = W + (long long)k2 * N, *w3 = W + (long long)k3 * N;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int j = 0; j < n; ++j) {
      const float d = dy[j * LP_LS + lane];
      a0 = fmaf(d, w0[j], a0);
      a1 = fmaf(d, w1[j], a1);
      a2 = fmaf(d, w2[j], a2);
      a3 = fmaf(d, w3[j], a3);
    }
    dx[k0 * LP_LS + lane] = a0;
    if (k0 + 1 < K) dx[(k0 + 1) * LP_LS + lane] = a1;
    if (k0 + 2 < K) dx[(k0 + 2) * LP_LS + lane] = a2;
    if (k0 + 3 < K) dx[(k0 + 3) * LP_LS + lane] = a3;
  }
}

// warp-cooperative parameter gradient over the warp's 32 samples:
//   dW[i][j] += sum_s x[i][s] * dy[j][s],  db[j] += sum_s dy[j][s]      (accumulated in smem)
// Callers must __syncwarp() before (tiles complete) and after (tiles reusable).
LP_DEVICE void lp_warp_dw(float* dP, const LpLayer& L, const float* x, const float* dy, int lane) {
  const int n = L.n_used, total = L.K * n;
  for (int e = lane; e < total; e += LP_WARP) {
    const int i = e / n, j = e - i * n;
    const float* xr = x + i * LP_LS;
    const float* dr = dy + j * LP_LS;
    float acc = 0.f;
#pragma unroll 8
    for (int s = 0; s < LP_WARP; ++s) acc = fmaf(xr[s], dr[s], acc);
    if (acc != 0.f) atomicAdd(dP + L.w_off + i * L.N + j, acc);
  }
  for (int j = lane; j < n; j += LP_WARP) {
    const float* dr = dy + j * LP_LS;
    float acc = 0.f;
#pragma unroll 8
    for (int s = 0; s < LP_WARP; ++s) acc += dr[s];
    if (acc != 0.f) atomicAdd(dP + L.b_off + j, acc);
  }
}

// Sample a grid-list at one point into a [C][lane] tile (sum over grids; optional OOB mask,
// optional ReLU).  (grid_sample_util.py:1088-1216)
LP_DEVICE void lp_lane_sample(const LpGridSet& G, int b, float x, float y, float z, float oob,
                              bool relu, float* tile, int lane) {
  const int C = G.C;
  for (int gi = 0; gi < G.n; ++gi) {
    long long off[8];
    float w[8];
    const int nt = lp_taps(G.g[gi], C, b, x, y, z, off, w);
    for (int c = 0; c < C; c += 4) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gi > 0) {
        acc.x = tile[(c + 0) * LP_LS + lane]; acc.y = tile[(c + 1) * LP_LS + lane];
        acc.z = tile[(c + 2) * LP_LS + lane]; acc.w = tile[(c + 3) * LP_LS + lane];
      }
      for (int t = 0; t < nt; ++t) {
        if (w[t] != 0.f) {
          const float4 v = lp_ldg4(G.data + off[t] + c);
          acc.x = fmaf(w[t], v.x, acc.x); acc.y = fmaf(w[t], v.y, acc.y);
          acc.z = fmaf(w[t], v.z, acc.z); acc.w = fmaf(w[t], v.w, acc.w);
        }
      }
      if (gi == G.n - 1) {
        acc.x *= oob; acc.y *= oob; acc.z *= oob; acc.w *= oob;
        if (relu) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
      }
      tile[(c + 0) * LP_LS + lane] = acc.x; tile[(c + 1) * LP_LS + lane] = acc.y;
      tile[(c + 2) * LP_LS + lane] = acc.z; tile[(c + 3) * LP_LS + lane] = acc.w;
    }
  }
}

// Adjoint: scatter a [C][lane] gradient tile into the grid-list gradient with vector atomics
// (grid_sample_util.py:40-206,1219-1246).
LP_DEVICE void lp_lane_splat(const LpGridSet& G, float* grad, int b, float x, float y, float z,
                             float scale, const float* tile, int lane) {
  const int C = G.C;
  if (scale == 0.f) return;
  for (int gi = 0; gi < G.n; ++gi) {
    long long off[8];
    float w[8];
    const int nt = lp_taps(G.g[gi], C, b, x, y, z, off, w);
    for (int c = 0; c < C; c += 4) {
      const float d0 = tile[(c + 0) * LP_LS + lane] * scale, d1 = tile[(c + 1) * LP_LS + lane] * scale,
                  d2 = tile[(c + 2) * LP_LS + lane] * scale, d3 = tile[(c + 3) * LP_LS + lane] * scale;
      for (int t = 0; t < nt; ++t)
        if (w[t] != 0.f) lp_red_add4(grad + off[t] + c, w[t] * d0, w[t] * d1, w[t] * d2, w[t] * d3);
    }
  }
}

struct LpRayState {
  float ox, oy, oz, dx, dy, dz, near, far;
  int b, ray;
  bool active;
};

LP_DEVICE LpRayState lp_load_ray(const LpRays& R, int ray, int batch) {
  LpRayState s;
  s.active = ray < R.n;
  s.ray = ray;
  const int r = s.active ? ray : R.n - 1;  // inactive lanes shadow the last ray (finite data)
  s.ox = R.org[3 * r]; s.oy = R.org[3 * r + 1]; s.oz = R.org[3 * r + 2];
  s.dx = R.dir[3 * r]; s.dy = R.dir[3 * r + 1]; s.dz = R.dir[3 * r + 2];
  s.near = R.near[r]; s.far = R.far[r];
  s.b = min(max(R.gidx[r], 0), batch - 1);
  return s;
}

// Evaluate the decoder for the lane's current sample.  Fills the arena slots of `A` (all of them
// -- the forward kernel passes a map whose hidden slots alias ping-pong buffers) and returns the
// raw opacity; pre-sigmoid colours end in slot yc[last].
LP_DEVICE float lp_eval_decoder(const LpDecoder& D, const LpActMap& A, const float* P, float* arena,
                                const float* enc, const LpGridSet& G, const LpGridSet& CG, int b,
                                float x, float y, float z, float oob, int lane) {
  float* x0 = arena + A.x0 * LP_LS;
  lp_lane_sample(G, b, x, y, z, oob, D.use_color_grid != 0, x0, lane);
  const float* trunk = x0;
  for (int l = 0; l < D.trunk.n_layers; ++l) {
    float* out = arena + A.yt[l] * LP_LS;
    lp_lane_linear(P, D.trunk.l[l], trunk, out, lane);
    trunk = out;
  }
  // opacity head
  const float* h = trunk;
  for (int l = 0; l < D.opacity.n_layers; ++l) {
    float* out = arena + A.yo[l] * LP_LS;
    lp_lane_linear(P, D.opacity.l[l], h, out, lane);
    h = out;
  }
  const float raw = h[lane];
  // colour head input
  float* xc = arena + A.xc * LP_LS;
  if (D.use_color_grid) {
    float* xcs = arena + A.xcs * LP_LS;
    lp_lane_sample(CG, b, x, y, z, oob, true, xcs, lane);
    for (int k = 0; k < D.in_c; ++k) xc[k * LP_LS + lane] = xcs[k * LP_LS + lane] + enc[k * LP_LS + lane];
  } else {
    for (int k = 0; k < D.in_c; ++k) xc[k * LP_LS + lane] = trunk[k * LP_LS + lane] + enc[k * LP_LS + lane];
  }
  h = xc;
  for (int l = 0; l < D.color.n_layers; ++l) {
    float* out = arena + A.yc[l] * LP_LS;
    lp_lane_linear(P, D.color.l[l], h, out, lane);
    h = out;
  }
  return raw;
}

// ===========================================================================================
// forward
// ===========================================================================================
__global__ void lp_render_fwd_generic_kernel(LpRays R, LpMarch M, LpDecoder D, LpActMap A,
                                             LpGridSet G, LpGridSet CG, LpGridSet SC,
                                             int use_scaffold, const float* __restrict__ params,
                                             int params_in_smem, float* __restrict__ out_len,
                                             float* __restrict__ out_nlt,
                                             float* __restrict__ out_feat, int feat_stride) {
  LP_DYN_SMEM(float, smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int pfloats = params_in_smem ? ((D.n_params + 3) & ~3) : 0;
  const float* P = params;
  if (params_in_smem) {
    for (int i = threadIdx.x; i < D.n_params; i += blockDim.x) smem[i] = params[i];
    P = smem;
  }
  __syncthreads();
  const int per_warp = (A.total + D.in_c + D.n_feat) * LP_LS;
  float* arena = smem + pfloats + warp * per_warp;
  float* enc = arena + A.total * LP_LS;
  float* facc = enc + D.in_c * LP_LS;

  const int ray = (blockIdx.x * nwarps + warp) * LP_WARP + lane;
  const LpRayState s = lp_load_ray(R, ray, G.g[0].B);
  for (int k = 0; k < D.in_c; ++k) enc[k * LP_LS + lane] = R.enc[(long long)(s.active ? ray : R.n - 1) * D.in_c + k];
  for (int c = 0; c < D.n_feat; ++c) facc[c * LP_LS + lane] = 0.f;

  float nlt = 0.f, T = 1.f, len = 0.f;
  const int tot = M.S + M.S_inf;
  const float* logc = arena + A.yc[D.color.n_layers - 1] * LP_LS;
  for (int step = 0; step < tot; ++step) {
    const float depth = lp_depth(step, s.near, s.far, M.S, M.S_inf, M.disparity_at_inf);
    const float delta = lp_delta(step, depth, s.near, s.far, M.S, M.S_inf, M.disparity_at_inf);
    float x = s.ox + depth * s.dx, y = s.oy + depth * s.dy, z = s.oz + depth * s.dz;
    if (M.contract) lp_contract(x, y, z);
    float occ = 1.f;
    if (use_scaffold) occ = lp_nearest(SC, s.b, x, y, z);
    if (!__any_sync(LP_FULL_MASK, occ != 0.f)) continue;  // empty space: nothing changes
    const float oob = M.mask_oob ? lp_in_bounds(x, y, z) : 1.f;
    float raw = lp_eval_decoder(D, A, P, arena, enc, G, CG, s.b, x, y, z, oob, lane);
    if (M.noise) raw += M.sigma * lp_sample_noise(M, ray, step);
    const float dop = delta * M.gain * lp_softplus(raw) * occ;
    nlt += dop;
    const float Tn = expf(-nlt);
    const float w = T - Tn;
    len = fmaf(w, depth, len);
    for (int c = 0; c < D.n_feat; ++c)
      facc[c * LP_LS + lane] = fmaf(w * occ, lp_sigmoid(logc[c * LP_LS + lane]), facc[c * LP_LS + lane]);
    T = Tn;
  }
  if (s.active) {
    out_len[ray] = len;
    out_nlt[ray] = nlt;
    for (int c = 0; c < D.n_feat; ++c) out_feat[(long long)ray * feat_stride + c] = facc[c * LP_LS + lane];
  }
}

// ===========================================================================================
// backward
// ===========================================================================================
// Back-propagate one MLP for the lane's sample.  dy_last: [n_used_last][lane] tile holding the
// gradient w.r.t. the last layer's (pre-activation) output.  Ping-pongs between g0/g1; returns the
// tile holding the gradient w.r.t. the MLP input.  `in0` = input tile of layer 0, `ys` = slots of
// the layer outputs.  Accumulates dW/db into the shared accumulator dP.
LP_DEVICE float* lp_mlp_backward(const LpMlp& Mlp, const float* P, float* dP, const float* arena,
                                 const float* in0, const int* ys, float* dy, float* other, int lane) {
  for (int l = Mlp.n_layers - 1; l >= 0; --l) {
    const LpLayer& L = Mlp.l[l];
    const float* xin = (l == 0) ? in0 : arena + ys[l - 1] * LP_LS;
    if (L.relu) {  // dy was w.r.t. the post-ReLU output: gate it
      const float* yout = arena + ys[l] * LP_LS;
      for (int j = 0; j < L.n_used; ++j)
        if (!(yout[j * LP_LS + lane] > 0.f)) dy[j * LP_LS + lane] = 0.f;
    }
    __syncwarp();
    lp_warp_dw(dP, L, xin, dy, lane);
    lp_lane_linear_dx(P, L, dy, other, lane);
    __syncwarp();
    float* t = dy; dy = other; other = t;
  }
  return dy;
}

// Gradient w.r.t. the sample position of the lane's [C][lane] sampled-feature gradient tile (lp_lane_splat's adjoint
// partner: the same taps, weighted by their weight gradients instead of their weights)
LP_DEVICE void lp_lane_pos_grad(const LpGridSet& G, int b, float x, float y, float z, const float* tile, int lane,
                                float& gx, float& gy, float& gz) {
  const int C = G.C;
  lp_pos_grad(G, b, x, y, z, [&](const float* row) {
    float acc = 0.f;
    for (int c = 0; c < C; c += 4) {
      const float4 v = lp_ldg4(row + c);
      acc = fmaf(v.x, tile[(c + 0) * LP_LS + lane], acc); acc = fmaf(v.y, tile[(c + 1) * LP_LS + lane], acc);
      acc = fmaf(v.z, tile[(c + 2) * LP_LS + lane], acc); acc = fmaf(v.w, tile[(c + 3) * LP_LS + lane], acc);
    }
    return acc;
  }, gx, gy, gz);
}

// RAYG: also the gradients w.r.t. the rays' origins and directions (io.g_org / io.g_dir, lp_render_backward_rays):
// per sample j at p_j = o + t_j d, g_j = d L / d p_j from the taps' weight gradients (lp_pos_grad) and the contraction's
// Jacobian; dL/do = sum_j g_j, dL/dd = sum_j t_j g_j.
template <bool RAYG>
__global__ void lp_render_bwd_generic_kernel(LpRays R, LpMarch M, LpDecoder D, LpActMap A, LpGridSet G,
                                             LpGridSet CG, LpGridSet SC, int use_scaffold,
                                             const float* __restrict__ params, int params_in_smem,
                                             LpBwdIo io) {
  LP_DYN_SMEM(float, smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int pfloats = (D.n_params + 3) & ~3;
  const float* P = params;
  float* dP = smem;  // [pfloats] parameter-gradient accumulator of this block
  for (int i = threadIdx.x; i < pfloats; i += blockDim.x) dP[i] = 0.f;
  float* base = smem + pfloats;
  if (params_in_smem) {
    for (int i = threadIdx.x; i < D.n_params; i += blockDim.x) base[i] = params[i];
    P = base;
    base += pfloats;
  }
  __syncthreads();
  // per-warp: arena | 3 gradient tiles | enc | enc-grad | g_feat
  const int per_warp = (A.total + 3 * D.max_dim + 2 * D.in_c + D.n_feat) * LP_LS;
  float* arena = base + warp * per_warp;
  float* gA = arena + A.total * LP_LS;
  float* gB = gA + D.max_dim * LP_LS;
  float* gT = gB + D.max_dim * LP_LS;
  float* enc = gT + D.max_dim * LP_LS;
  float* genc = enc + D.in_c * LP_LS;
  float* gF = genc + D.in_c * LP_LS;

  const int ray = (blockIdx.x * nwarps + warp) * LP_WARP + lane;
  const LpRayState s = lp_load_ray(R, ray, G.g[0].B);
  const int rr = s.active ? ray : R.n - 1;
  const float act = s.active ? 1.f : 0.f;
  for (int k = 0; k < D.in_c; ++k) {
    enc[k * LP_LS + lane] = R.enc[(long long)rr * D.in_c + k];
    genc[k * LP_LS + lane] = 0.f;
  }
  const float g_len = act * io.g_len[rr], g_nlt = act * io.g_nlt[rr];
  // total = sum_k w_k p_k, recovered from the forward outputs
  float total = g_len * io.len[rr];
  for (int c = 0; c < D.n_feat; ++c) {
    const float g = act * io.g_feat[(long long)rr * io.g_feat_stride + c];
    gF[c * LP_LS + lane] = g;
    total = fmaf(g, io.feat[(long long)rr * io.feat_stride + c], total);
  }
  float nlt = 0.f, T = 1.f, prefix = 0.f;
  float gox = 0.f, goy = 0.f, goz = 0.f, gdx = 0.f, gdy = 0.f, gdz = 0.f;  // RAYG: dL/d origin, dL/d direction

  const int tot = M.S + M.S_inf;
  const int nc = D.color.n_layers, nt = D.trunk.n_layers;
  const float* logc = arena + A.yc[nc - 1] * LP_LS;
  for (int step = 0; step < tot; ++step) {
    const float depth = lp_depth(step, s.near, s.far, M.S, M.S_inf, M.disparity_at_inf);
    const float delta = lp_delta(step, depth, s.near, s.far, M.S, M.S_inf, M.disparity_at_inf);
    float x = s.ox + depth * s.dx, y = s.oy + depth * s.dy, z = s.oz + depth * s.dz;
    const float px = x, py = y, pz = z;
    float gx = 0.f, gy = 0.f, gz = 0.f;  // RAYG: dL/d (grid-space sample point)
    if (M.contract) lp_contract(x, y, z);
    float occ = 1.f;
    if (use_scaffold) occ = lp_nearest(SC, s.b, x, y, z);
    if (!__any_sync(LP_FULL_MASK, occ != 0.f)) continue;  // w = 0 for every lane: no gradient
    const float oob = M.mask_oob ? lp_in_bounds(x, y, z) : 1.f;
    float raw = lp_eval_decoder(D, A, P, arena, enc, G, CG, s.b, x, y, z, oob, lane);
    if (M.noise) raw += M.sigma * lp_sample_noise(M, ray, step);
    // ---- compositing gradient ----
    nlt += delta * M.gain * lp_softplus(raw) * occ;
    const float Tn = expf(-nlt);
    const float w = T - Tn;  // render weight of this sample
    T = Tn;
    float p = depth * g_len;
    for (int c = 0; c < D.n_feat; ++c) p = fmaf(lp_sigmoid(logc[c * LP_LS + lane]), gF[c * LP_LS + lane], p);
    p *= occ;
    prefix = fmaf(w, p, prefix);
    // suffix = sum_{k>j} w_k p_k; exactly 0 behind the last sample (its huge background step
    // length would otherwise amplify the rounding residue of total - prefix)
    const float suffix = (step == tot - 1) ? 0.f : total - prefix;
    const float g_dop = Tn * p - suffix + g_nlt;
    const float g_raw = g_dop * delta * M.gain * occ * lp_sigmoid(raw);

    // ---- colour head ----
    for (int c = 0; c < D.n_feat; ++c) {
      const float sg = lp_sigmoid(logc[c * LP_LS + lane]);
      gA[c * LP_LS + lane] = w * occ * gF[c * LP_LS + lane] * sg * (1.f - sg);
    }
    float* d_xc = lp_mlp_backward(D.color, P, dP, arena, arena + A.xc * LP_LS, A.yc, gA, gB, lane);
    for (int k = 0; k < D.in_c; ++k) genc[k * LP_LS + lane] += d_xc[k * LP_LS + lane];
    // gT <- gradient w.r.t. the trunk output (or stays the colour-branch sample gradient)
    float* free_tile = (d_xc == gA) ? gB : gA;
    if (D.use_color_grid) {
      const float* xcs = arena + A.xcs * LP_LS;
      for (int k = 0; k < D.C; ++k)
        if (!(xcs[k * LP_LS + lane] > 0.f)) d_xc[k * LP_LS + lane] = 0.f;
      lp_lane_splat(CG, io.g_cgrid, s.b, x, y, z, oob, d_xc, lane);
      if (RAYG && oob != 0.f) lp_lane_pos_grad(CG, s.b, x, y, z, d_xc, lane, gx, gy, gz);
      for (int k = 0; k < D.C; ++k) gT[k * LP_LS + lane] = 0.f;
    } else {
      for (int k = 0; k < D.in_c; ++k) gT[k * LP_LS + lane] = d_xc[k * LP_LS + lane];
    }
    // ---- opacity head ----
    float* go = d_xc;  // reuse: gradient of the 1-wide raw opacity
    go[lane] = g_raw;
    const float* op_in = (nt > 0) ? arena + A.yt[nt - 1] * LP_LS : arena + A.x0 * LP_LS;
    float* d_oin = lp_mlp_backward(D.opacity, P, dP, arena, op_in, A.yo, go, free_tile, lane);
    const int trunk_dim = (nt > 0) ? D.trunk.l[nt - 1].n_used : D.C;
    for (int k = 0; k < trunk_dim; ++k) gT[k * LP_LS + lane] += d_oin[k * LP_LS + lane];
    // ---- trunk / sampled feature ----
    if (nt > 0) {
      // lp_mlp_backward gates by the trunk's own (post-ReLU) outputs, incl. the last layer;
      // gA/gB/gT stay three distinct tiles, only their contents are consumed here
      float* d_x0 = lp_mlp_backward(D.trunk, P, dP, arena, arena + A.x0 * LP_LS, A.yt, gT, gA, lane);
      lp_lane_splat(G, io.g_grid, s.b, x, y, z, oob, d_x0, lane);
      if (RAYG && oob != 0.f) lp_lane_pos_grad(G, s.b, x, y, z, d_x0, lane, gx, gy, gz);
    } else {
      const float* x0 = arena + A.x0 * LP_LS;  // relu-field: gate by relu(sampled) > 0
      for (int k = 0; k < D.C; ++k)
        if (!(x0[k * LP_LS + lane] > 0.f)) gT[k * LP_LS + lane] = 0.f;
      lp_lane_splat(G, io.g_grid, s.b, x, y, z, oob, gT, lane);
      if (RAYG && oob != 0.f) lp_lane_pos_grad(G, s.b, x, y, z, gT, lane, gx, gy, gz);
    }
    if (RAYG) {
      if (M.contract) lp_contract_vjp(px, py, pz, gx, gy, gz);
      gox += gx; goy += gy; goz += gz;
      gdx = fmaf(depth, gx, gdx); gdy = fmaf(depth, gy, gdy); gdz = fmaf(depth, gz, gdz);
    }
  }
  if (s.active)
    for (int k = 0; k < D.in_c; ++k) io.g_enc[(long long)ray * D.in_c + k] = genc[k * LP_LS + lane];
  if (RAYG && s.active) {
    if (io.g_org) { io.g_org[3 * ray] = gox; io.g_org[3 * ray + 1] = goy; io.g_org[3 * ray + 2] = goz; }
    if (io.g_dir) { io.g_dir[3 * ray] = gdx; io.g_dir[3 * ray + 1] = gdy; io.g_dir[3 * ray + 2] = gdz; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < D.n_params; i += blockDim.x) {
    const float v = dP[i];
    if (v != 0.f) lp_red_add1(io.g_params + i, v);
  }
}
