// C-ABI entry points of include/lightplane_b200.h: argument validation, kernel-parameter
// construction (grid tables, MLP layer tables, shared-memory budgeting) and launches.
// Stateless; everything runs on the caller's stream.
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <cstdlib>
#include "lp_common.cuh"
#include "lp_render_generic.cuh"
#include "lp_splat.cuh"
#include "lp_ray_embed.cuh"
#include "lp_render_tc.cuh"
#include "lp_render_tc_bwd.cuh"
#include "lp_render_tc_cg.cuh"
#include "lp_splat_tc.cuh"
#include "lp_render_tc_wide.cuh"
#include "lp_render_tc_deep.cuh"

static thread_local char g_err[512] = "";

#define LP_FAIL(code, ...)                         \
  do {                                             \
    snprintf(g_err, sizeof(g_err), __VA_ARGS__);   \
    return (code);                                 \
  } while (0)

#ifdef LP_HOSTSIM
static const int kMaxSmem = 227 * 1024;
static int lp_set_smem(const void*, size_t) { return 0; }
#define LP_SET_SMEM(kernel, bytes) lp_set_smem(nullptr, (bytes))
static int lp_check_launch(const char*) { return LP_OK; }
#else
static const int kMaxSmem = 227 * 1024;
#define LP_SET_SMEM(kernel, bytes) \
  (cudaFuncSetAttribute((kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)) == cudaSuccess ? 0 : 1)
static int lp_check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) LP_FAIL(LP_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return LP_OK;
}
#endif

// ---------------------------------------------------------------------------------------------
// struct conversion
// ---------------------------------------------------------------------------------------------
static int lp_make_gridset(const lp_grid_list* in, LpGridSet* out, const char* name) {
  memset(out, 0, sizeof(*out));
  if (!in) return LP_OK;
  if (in->num_grids < 1 || in->num_grids > LP_MAX_GRIDS)
    LP_FAIL(LP_ERR_INVALID_ARG, "%s: num_grids=%d not in [1,%d]", name, in->num_grids, LP_MAX_GRIDS);
  if (!in->data) LP_FAIL(LP_ERR_INVALID_ARG, "%s: data is NULL", name);
  if (((uintptr_t)in->data & 15) != 0)  // the kernels read / reduce rows as 16-byte vectors
    LP_FAIL(LP_ERR_INVALID_ARG, "%s: data is not 16-byte aligned", name);
  out->data = in->data;
  out->n = in->num_grids;
  out->C = in->channels;
  long long base = 0;
  for (int i = 0; i < in->num_grids; ++i) {
    const int32_t* s = in->sizes[i];
    if (s[0] < 1 || s[1] < 1 || s[2] < 1 || s[3] < 1)
      LP_FAIL(LP_ERR_INVALID_ARG, "%s: grid %d has a non-positive size", name, i);
    if (s[0] != in->sizes[0][0]) LP_FAIL(LP_ERR_INVALID_ARG, "%s: grids differ in batch size", name);
    if (s[4] != in->channels)
      LP_FAIL(LP_ERR_INVALID_ARG, "%s: grid %d has %d channels, the list says %d", name, i, s[4], in->channels);
    LpGrid& g = out->g[i];
    g.B = s[0]; g.D = s[1]; g.H = s[2]; g.W = s[3];
    // classification of grid_sample_util.py:1111-1173
    if ((long long)(g.D - 1) * (g.H - 1) * (g.W - 1) > 0) g.kind = LP_VOXEL;
    else if (g.D == 1) g.kind = LP_PLANE_XY;
    else if (g.H == 1) g.kind = LP_PLANE_XZ;
    else g.kind = LP_PLANE_YZ;
    g.base = base;
    base += (long long)g.B * g.D * g.H * g.W * in->channels;
  }
  // Triplane: exactly one XY, one XZ and one YZ plane with consistent axis sizes.  The entries are put in that order
  // (each keeps its own base offset, so the order of the table is free) and the kernels take their fast path.
  if (out->n == 3) {
    int at[3] = {-1, -1, -1};
    for (int i = 0; i < 3; ++i) {
      const int k = out->g[i].kind;
      if (k == LP_PLANE_XY) at[0] = i; else if (k == LP_PLANE_XZ) at[1] = i; else if (k == LP_PLANE_YZ) at[2] = i;
    }
    if (at[0] >= 0 && at[1] >= 0 && at[2] >= 0) {
      const LpGrid xy = out->g[at[0]], xz = out->g[at[1]], yz = out->g[at[2]];
      if (xy.W == xz.W && xy.H == yz.H && xz.D == yz.D && xy.W > 1 && xy.H > 1 && xz.D > 1) {
        out->g[0] = xy; out->g[1] = xz; out->g[2] = yz;
        out->tri = 1;
      }
    }
  }
  return LP_OK;
}

static int lp_make_rays(const lp_rays* in, LpRays* out, int need_enc_dim) {
  if (!in) LP_FAIL(LP_ERR_INVALID_ARG, "rays is NULL");
  if (in->num_rays < 0) LP_FAIL(LP_ERR_INVALID_ARG, "num_rays < 0");
  if (in->num_rays > 0 && (!in->directions || !in->origins || !in->grid_idx || !in->near || !in->far))
    LP_FAIL(LP_ERR_INVALID_ARG, "a ray field is NULL");
  if (need_enc_dim >= 0) {
    if (in->num_rays > 0 && !in->encoding) LP_FAIL(LP_ERR_INVALID_ARG, "rays.encoding is NULL");
    if (in->encoding_dim != need_enc_dim)
      LP_FAIL(LP_ERR_INVALID_ARG, "rays.encoding_dim=%d, expected %d", in->encoding_dim, need_enc_dim);
    if (((uintptr_t)in->encoding & 15) != 0) LP_FAIL(LP_ERR_INVALID_ARG, "rays.encoding is not 16-byte aligned");
  }
  out->dir = in->directions; out->org = in->origins; out->gidx = in->grid_idx;
  out->near = in->near; out->far = in->far; out->enc = in->encoding;
  out->n = in->num_rays; out->enc_dim = in->encoding_dim;
  return LP_OK;
}

static int lp_make_march(const lp_march_cfg* c, LpMarch* m) {
  if (!c) LP_FAIL(LP_ERR_INVALID_ARG, "cfg is NULL");
  if (c->num_samples < 1) LP_FAIL(LP_ERR_INVALID_ARG, "num_samples must be >= 1");
  if (c->num_samples_inf < 0) LP_FAIL(LP_ERR_INVALID_ARG, "num_samples_inf must be >= 0");
  m->S = c->num_samples; m->S_inf = c->num_samples_inf;
  m->gain = c->gain; m->disparity_at_inf = c->disparity_at_inf;
  m->mask_oob = c->mask_out_of_bounds != 0; m->contract = c->contract_coords != 0;
  m->noise = c->inject_noise != 0 && c->noise_sigma > 0.f;
  m->sigma = c->noise_sigma; m->seed = c->noise_seed; m->noise_num_rays = c->noise_num_rays;
  m->img_w = c->ray_image_width > 0 ? c->ray_image_width : 0;  // validated against the ray count by the renderer entry points
  return LP_OK;
}

// Fill the layer table of one MLP laid out as all weights then all biases starting at `*pos`.
static int lp_fill_mlp(LpMlp* m, int n_layers, int d_in, int d_hid, int d_out, int n_used_last,
                       int relu_last, int* pos) {
  memset(m, 0, sizeof(*m));
  if (n_layers < 0 || n_layers > LP_MAX_LAYERS)
    LP_FAIL(LP_ERR_UNSUPPORTED, "n_layers=%d exceeds LP_MAX_LAYERS=%d", n_layers, LP_MAX_LAYERS);
  m->n_layers = n_layers;
  int p = *pos;
  for (int l = 0; l < n_layers; ++l) {
    LpLayer& L = m->l[l];
    L.K = (l == 0) ? d_in : d_hid;
    L.N = (l == n_layers - 1) ? d_out : d_hid;
    L.n_used = (l == n_layers - 1) ? n_used_last : L.N;
    L.relu = (l < n_layers - 1) || relu_last;
    if (L.K < 1 || L.N < 1 || L.n_used < 1 || L.n_used > L.N)
      LP_FAIL(LP_ERR_INVALID_ARG, "bad layer dims K=%d N=%d used=%d", L.K, L.N, L.n_used);
    L.w_off = p;
    p += L.K * L.N;
  }
  for (int l = 0; l < n_layers; ++l) {
    m->l[l].b_off = p;
    p += m->l[l].N;
  }
  *pos = p;
  return LP_OK;
}

static int imax(int a, int b) { return a > b ? a : b; }

static int lp_make_decoder(const lp_decoder_spec* s, int C, LpDecoder* D, LpActMap* A) {
  if (!s) LP_FAIL(LP_ERR_INVALID_ARG, "decoder spec is NULL");
  memset(D, 0, sizeof(*D));
  memset(A, 0, sizeof(*A));
  if (s->n_layers_opacity < 1 || s->n_layers_color < 1)
    LP_FAIL(LP_ERR_INVALID_ARG, "opacity and colour MLPs need at least one layer");
  if (C % 4 != 0) LP_FAIL(LP_ERR_UNSUPPORTED, "grid channels (%d) must be a multiple of 4", C);
  D->use_color_grid = s->n_layers_trunk == 0;
  D->C = C;
  int pos = 0, rc;
  if ((rc = lp_fill_mlp(&D->trunk, s->n_layers_trunk, s->dim_in_trunk, s->dim_hidden_trunk,
                        s->dim_out_trunk, s->dim_out_trunk, 1, &pos)))
    return rc;
  if (s->n_layers_trunk > 0 && s->dim_in_trunk != C)
    LP_FAIL(LP_ERR_INVALID_ARG, "dim_in_trunk=%d != grid channels %d", s->dim_in_trunk, C);
  const int head_in = D->use_color_grid ? C : s->dim_out_trunk;
  if (s->dim_in_opacity != head_in || s->dim_in_color != head_in)
    LP_FAIL(LP_ERR_INVALID_ARG, "head input dims (%d,%d) != %d", s->dim_in_opacity, s->dim_in_color, head_in);
  if ((rc = lp_fill_mlp(&D->opacity, s->n_layers_opacity, s->dim_in_opacity, s->dim_hidden_opacity, 1, 1, 0, &pos)))
    return rc;
  if (s->num_color_used < 1 || s->num_color_used > s->dim_out_color)
    LP_FAIL(LP_ERR_INVALID_ARG, "num_color_used=%d not in [1,%d]", s->num_color_used, s->dim_out_color);
  if ((rc = lp_fill_mlp(&D->color, s->n_layers_color, s->dim_in_color, s->dim_hidden_color,
                        s->dim_out_color, s->num_color_used, 0, &pos)))
    return rc;
  D->n_params = pos;
  D->in_c = s->dim_in_color;
  D->n_feat = s->num_color_used;
  // activation arena
  int row = 0, md = imax(C, imax(D->in_c, D->n_feat));
  A->x0 = row; row += C;
  if (D->use_color_grid) { A->xcs = row; row += C; }
  A->xc = row; row += D->in_c;
  for (int l = 0; l < D->trunk.n_layers; ++l) { A->yt[l] = row; row += D->trunk.l[l].n_used; md = imax(md, D->trunk.l[l].N); }
  for (int l = 0; l < D->opacity.n_layers; ++l) { A->yo[l] = row; row += D->opacity.l[l].n_used; md = imax(md, D->opacity.l[l].N); }
  for (int l = 0; l < D->color.n_layers; ++l) { A->yc[l] = row; row += D->color.l[l].n_used; md = imax(md, D->color.l[l].n_used); }
  A->total = row;
  D->max_dim = md;
  return LP_OK;
}

// Choose warps per block so that the dynamic shared memory fits; params go to shared memory when
// they fit next to at least one warp, else they are read from global (L1-cached broadcasts).
static int lp_plan_smem(int fixed_floats, int params_floats, int per_warp_floats, int* warps,
                        int* params_in_smem, size_t* bytes) {
  for (int pin = 1; pin >= 0; --pin) {
    for (int w = 4; w >= 1; --w) {
      size_t b = 4ull * ((size_t)fixed_floats + (pin ? params_floats : 0) + (size_t)w * per_warp_floats);
      if (b <= (size_t)kMaxSmem) {
        *warps = w; *params_in_smem = pin; *bytes = b;
        return LP_OK;
      }
    }
  }
  LP_FAIL(LP_ERR_RESOURCE, "MLP too large for the shared-memory tiles of the generic kernel "
          "(%d floats per warp)", per_warp_floats);
}

// ---------------------------------------------------------------------------------------------
extern "C" {

int lp_abi_version(void) { return LP_ABI_VERSION; }
const char* lp_last_error(void) { return g_err; }
int lp_is_device_build(void) { return LP_IS_DEVICE_BUILD; }

// LP_ONLY_GENERIC=1 in the environment routes every renderer launch to the generic fp32 kernels (lp_render_generic.cuh):
// a measurement aid -- it gives the error of a plain fp32 implementation of the same decoder against the fp64 oracle, the
// floor the tensor-core paths' tolerances are judged against (tests/test_gpu_parity.py).
static bool lp_only_generic() {
  const char* e = getenv("LP_ONLY_GENERIC");
  return e != nullptr && e[0] == '1';
}

static int lp_render_common(const lp_march_cfg* cfg, const lp_decoder_spec* spec, const lp_rays* rays,
                            const lp_grid_list* grid, const lp_grid_list* color_grid,
                            const lp_grid_list* scaffold, const float* mlp_params, LpRenderArgs* a) {
  int rc;
  if (!grid) LP_FAIL(LP_ERR_INVALID_ARG, "grid is NULL");
  if (!mlp_params) LP_FAIL(LP_ERR_INVALID_ARG, "mlp_params is NULL");
  if ((rc = lp_make_march(cfg, &a->M))) return rc;
  if ((rc = lp_make_gridset(grid, &a->G, "grid"))) return rc;
  if ((rc = lp_make_gridset(color_grid, &a->CG, "color_grid"))) return rc;
  if ((rc = lp_make_gridset(scaffold, &a->SC, "scaffold"))) return rc;
  if ((rc = lp_make_decoder(spec, a->G.C, &a->D, &a->A))) return rc;
  if ((rc = lp_make_rays(rays, &a->R, a->D.in_c))) return rc;
  // the tile walk is a hint: it applies only when the rays really are whole 16x8-pixel tiles of an image that wide
  if (a->M.img_w % 16 != 0 || a->R.n % (a->M.img_w > 0 ? a->M.img_w * 8 : 1) != 0) a->M.img_w = 0;
  if (a->D.use_color_grid) {
    if (!color_grid) LP_FAIL(LP_ERR_INVALID_ARG, "n_layers_trunk == 0 requires a color_grid");
    if (a->CG.C != a->G.C) LP_FAIL(LP_ERR_INVALID_ARG, "color_grid channels != grid channels");
    if (a->CG.g[0].B != a->G.g[0].B) LP_FAIL(LP_ERR_INVALID_ARG, "color_grid batch != grid batch");
  } else if (color_grid) {
    LP_FAIL(LP_ERR_INVALID_ARG, "a color_grid requires n_layers_trunk == 0");
  }
  a->use_scaffold = scaffold != nullptr;
  if (scaffold) {
    if (a->SC.n != 1 || a->SC.C != 1) LP_FAIL(LP_ERR_INVALID_ARG, "scaffold must be one [B,D,H,W,1] grid");
    if (a->SC.g[0].B != a->G.g[0].B) LP_FAIL(LP_ERR_INVALID_ARG, "scaffold batch != grid batch");
    a->SC.g[0].kind = LP_VOXEL;
  }
  return LP_OK;
}

int lp_render_forward(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                      const lp_rays* rays, const lp_grid_list* grid, const lp_grid_list* color_grid,
                      const lp_grid_list* scaffold, const float* mlp_params, float* out_ray_length,
                      float* out_neg_log_transmittance, float* out_features, int32_t features_stride) {
  LpRenderArgs a;
  int rc;
  if ((rc = lp_render_common(cfg, spec, rays, grid, color_grid, scaffold, mlp_params, &a))) return rc;
  if (a.R.n == 0) return LP_OK;
  if (!out_ray_length || !out_neg_log_transmittance || !out_features)
    LP_FAIL(LP_ERR_INVALID_ARG, "an output pointer is NULL");
  if (features_stride < a.D.n_feat) LP_FAIL(LP_ERR_INVALID_ARG, "features_stride < num_color_used");
  cudaStream_t st = (cudaStream_t)stream;
  const bool fast = !lp_only_generic();
  if (fast && lptc::lp_tc_render_supported(a)) {
    if ((rc = lptc::lp_tc_render_forward(st, a, mlp_params, out_ray_length, out_neg_log_transmittance, out_features,
                                         features_stride)))
      LP_FAIL(rc, "fast forward launch setup failed");
    return lp_check_launch("lp_render_forward(fast)");
  }
  if (fast && lptc::lp_cg_render_supported(a)) {
    if ((rc = lptc::lp_cg_render_forward(st, a, mlp_params, out_ray_length, out_neg_log_transmittance, out_features,
                                         features_stride)))
      LP_FAIL(rc, "colour-grid forward launch setup failed");
    return lp_check_launch("lp_render_forward(colour grid)");
  }
  if (fast && lptc::lp_tcw_forward_supported(a)) {
    if ((rc = lptc::lp_tcw_render_forward(st, a, mlp_params, out_ray_length, out_neg_log_transmittance, out_features,
                                          features_stride)))
      LP_FAIL(rc, "hidden-64 forward launch setup failed");
    return lp_check_launch("lp_render_forward(hidden 64)");
  }
  lptc::DeepPlan dpl;
  if (fast && lptc::lp_deep_plan(a, &dpl)) {
    if ((rc = lptc::lp_deep_render_forward(st, a, dpl, mlp_params, out_ray_length, out_neg_log_transmittance, out_features,
                                           features_stride)))
      LP_FAIL(rc, "layer-count-general forward launch setup failed");
    return lp_check_launch("lp_render_forward(deep)");
  }
  const int pf = (a.D.n_params + 3) & ~3;
  const int per_warp = (a.A.total + a.D.in_c + a.D.n_feat) * LP_LS;
  int warps, pin; size_t bytes;
  if ((rc = lp_plan_smem(0, pf, per_warp, &warps, &pin, &bytes))) return rc;
  if (LP_SET_SMEM(lp_render_fwd_generic_kernel, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
  const int rays_per_block = warps * LP_WARP;
  dim3 gridDimv((a.R.n + rays_per_block - 1) / rays_per_block), block(rays_per_block);
  LP_LAUNCH(lp_render_fwd_generic_kernel, gridDimv, block, bytes, st, a.R, a.M, a.D, a.A, a.G, a.CG, a.SC,
            a.use_scaffold, mlp_params, pin, out_ray_length, out_neg_log_transmittance, out_features,
            (int)features_stride);
  return lp_check_launch("lp_render_forward");
}

// lp_render_backward and lp_render_backward_rays: grad_origins / grad_directions NULL = that gradient is not wanted;
// with both NULL the kernels without the ray-geometry terms run.
static int lp_render_backward_impl(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                                   const lp_rays* rays, const lp_grid_list* grid, const lp_grid_list* color_grid,
                                   const lp_grid_list* scaffold, const float* mlp_params, const float* ray_length,
                                   const float* features, int32_t features_stride, const float* grad_ray_length,
                                   const float* grad_neg_log_transmittance, const float* grad_features,
                                   int32_t grad_features_stride, float* grad_grid, float* grad_color_grid,
                                   float* grad_mlp_params, float* grad_encoding, float* grad_origins,
                                   float* grad_directions) {
  LpRenderArgs a;
  int rc;
  if ((rc = lp_render_common(cfg, spec, rays, grid, color_grid, scaffold, mlp_params, &a))) return rc;
  if (a.R.n == 0) return LP_OK;
  if (!ray_length || !features || !grad_ray_length || !grad_neg_log_transmittance || !grad_features)
    LP_FAIL(LP_ERR_INVALID_ARG, "a forward-output / upstream-gradient pointer is NULL");
  if (!grad_grid || !grad_mlp_params || !grad_encoding) LP_FAIL(LP_ERR_INVALID_ARG, "a gradient output is NULL");
  if (a.D.use_color_grid && !grad_color_grid) LP_FAIL(LP_ERR_INVALID_ARG, "grad_color_grid is NULL");
  if (grad_features_stride < a.D.n_feat || features_stride < a.D.n_feat)
    LP_FAIL(LP_ERR_INVALID_ARG, "a features stride is smaller than num_color_used");
  cudaStream_t st = (cudaStream_t)stream;
  LpBwdIo io;
  io.len = ray_length; io.feat = features; io.feat_stride = features_stride;
  io.g_len = grad_ray_length; io.g_nlt = grad_neg_log_transmittance; io.g_feat = grad_features;
  io.g_feat_stride = grad_features_stride;
  io.g_grid = grad_grid; io.g_cgrid = grad_color_grid; io.g_params = grad_mlp_params; io.g_enc = grad_encoding;
  io.g_org = grad_origins; io.g_dir = grad_directions;
  const bool rayg = grad_origins || grad_directions;
  const bool fast = !lp_only_generic();
  if (fast && lptc::lp_tc_render_supported(a)) {
    if ((rc = lptc::lp_tc_render_backward(st, a, mlp_params, io, rayg))) LP_FAIL(rc, "fast backward launch setup failed");
    return lp_check_launch("lp_render_backward(fast)");
  }
  // the other tensor-core variants have no ray-geometry terms: such requests take the generic kernel
  if (fast && !rayg && lptc::lp_cg_render_supported(a)) {
    if ((rc = lptc::lp_cg_render_backward(st, a, mlp_params, io))) LP_FAIL(rc, "colour-grid backward launch setup failed");
    return lp_check_launch("lp_render_backward(colour grid)");
  }
  if (fast && !rayg && lptc::lp_tcw_forward_supported(a)) {
    if ((rc = lptc::lp_tcw_render_backward(st, a, mlp_params, io))) LP_FAIL(rc, "hidden-64 backward launch setup failed");
    return lp_check_launch("lp_render_backward(hidden 64)");
  }
  lptc::DeepPlan dpl;
  if (fast && !rayg && lptc::lp_deep_plan(a, &dpl)) {
    if ((rc = lptc::lp_deep_render_backward(st, a, dpl, mlp_params, io))) LP_FAIL(rc, "layer-count-general backward launch setup failed");
    return lp_check_launch("lp_render_backward(deep)");
  }
  const int pf = (a.D.n_params + 3) & ~3;
  const int per_warp = (a.A.total + 3 * a.D.max_dim + 2 * a.D.in_c + a.D.n_feat) * LP_LS;
  int warps, pin; size_t bytes;
  if ((rc = lp_plan_smem(pf, pf, per_warp, &warps, &pin, &bytes))) return rc;
  const int rays_per_block = warps * LP_WARP;
  dim3 gridDimv((a.R.n + rays_per_block - 1) / rays_per_block), block(rays_per_block);
  if (rayg) {
    if (LP_SET_SMEM(lp_render_bwd_generic_kernel<true>, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
    LP_LAUNCH(lp_render_bwd_generic_kernel<true>, gridDimv, block, bytes, st, a.R, a.M, a.D, a.A, a.G, a.CG, a.SC,
              a.use_scaffold, mlp_params, pin, io);
  } else {
    if (LP_SET_SMEM(lp_render_bwd_generic_kernel<false>, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
    LP_LAUNCH(lp_render_bwd_generic_kernel<false>, gridDimv, block, bytes, st, a.R, a.M, a.D, a.A, a.G, a.CG, a.SC,
              a.use_scaffold, mlp_params, pin, io);
  }
  return lp_check_launch("lp_render_backward");
}

int lp_render_backward(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                       const lp_rays* rays, const lp_grid_list* grid, const lp_grid_list* color_grid,
                       const lp_grid_list* scaffold, const float* mlp_params, const float* ray_length,
                       const float* features, int32_t features_stride, const float* grad_ray_length,
                       const float* grad_neg_log_transmittance, const float* grad_features,
                       int32_t grad_features_stride, float* grad_grid, float* grad_color_grid,
                       float* grad_mlp_params, float* grad_encoding) {
  return lp_render_backward_impl(stream, cfg, spec, rays, grid, color_grid, scaffold, mlp_params, ray_length, features,
                                 features_stride, grad_ray_length, grad_neg_log_transmittance, grad_features,
                                 grad_features_stride, grad_grid, grad_color_grid, grad_mlp_params, grad_encoding,
                                 nullptr, nullptr);
}

int lp_render_backward_rays(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                            const lp_rays* rays, const lp_grid_list* grid, const lp_grid_list* color_grid,
                            const lp_grid_list* scaffold, const float* mlp_params, const float* ray_length,
                            const float* features, int32_t features_stride, const float* grad_ray_length,
                            const float* grad_neg_log_transmittance, const float* grad_features,
                            int32_t grad_features_stride, float* grad_grid, float* grad_color_grid,
                            float* grad_mlp_params, float* grad_encoding, float* grad_origins,
                            float* grad_directions) {
  return lp_render_backward_impl(stream, cfg, spec, rays, grid, color_grid, scaffold, mlp_params, ray_length, features,
                                 features_stride, grad_ray_length, grad_neg_log_transmittance, grad_features,
                                 grad_features_stride, grad_grid, grad_color_grid, grad_mlp_params, grad_encoding,
                                 grad_origins, grad_directions);
}

// ---- plain splatter ---------------------------------------------------------------------------
static int lp_splat_geometry(int C, int* lpr, int* vpl) {
  if (C % 4 != 0 || C < 4) LP_FAIL(LP_ERR_UNSUPPORTED, "splat channels (%d) must be a multiple of 4", C);
  const int chunks = C / 4;
  int l = 1;
  while (l * 2 <= 32 && chunks % (l * 2) == 0) l *= 2;  // largest power of two dividing chunks, <= 32
  const int v = chunks / l;
  if (v != 1 && v != 2 && v != 4 && v != 8)
    LP_FAIL(LP_ERR_UNSUPPORTED, "splat channels (%d) need %d float4 per lane; supported: 1,2,4,8", C, v);
  *lpr = l; *vpl = v;
  return LP_OK;
}

// the plain splat kernels address grid rows with 32-bit indices
static int lp_splat_rows_fit(const LpGridSet& G, const char* name) {
  const LpGrid& g = G.g[G.n - 1];
  const long long rows = g.base / G.C + (long long)g.B * g.D * g.H * g.W;
  if (rows > 0x7fffffffLL) LP_FAIL(LP_ERR_UNSUPPORTED, "%s: %lld grid rows; the splatter supports < 2^31", name, rows);
  return LP_OK;
}

int lp_splat_forward(void* stream, const lp_march_cfg* cfg, const lp_rays* rays, const float* valid_mask,
                     const lp_grid_list* out, float* weight_grid) {
  LpRays R; LpMarch M; LpGridSet O;
  int rc, lpr, vpl;
  if (!out) LP_FAIL(LP_ERR_INVALID_ARG, "out is NULL");
  if ((rc = lp_make_march(cfg, &M))) return rc;
  if ((rc = lp_make_gridset(out, &O, "out"))) return rc;
  if ((rc = lp_make_rays(rays, &R, O.C))) return rc;
  if (R.n == 0) return LP_OK;
  if ((rc = lp_splat_geometry(O.C, &lpr, &vpl))) return rc;
  if ((rc = lp_splat_rows_fit(O, "out"))) return rc;
  const int threads = 128, rays_per_block = threads / lpr;
  dim3 g((R.n + rays_per_block - 1) / rays_per_block), b(threads);
  cudaStream_t st = (cudaStream_t)stream;
  switch (vpl) {
    case 1: LP_LAUNCH(lp_splat_fwd_kernel<1>, g, b, 0, st, R, M, O, weight_grid, valid_mask, lpr); break;
    case 2: LP_LAUNCH(lp_splat_fwd_kernel<2>, g, b, 0, st, R, M, O, weight_grid, valid_mask, lpr); break;
    case 4: LP_LAUNCH(lp_splat_fwd_kernel<4>, g, b, 0, st, R, M, O, weight_grid, valid_mask, lpr); break;
    default: LP_LAUNCH(lp_splat_fwd_kernel<8>, g, b, 0, st, R, M, O, weight_grid, valid_mask, lpr); break;
  }
  return lp_check_launch("lp_splat_forward");
}

int lp_splat_backward(void* stream, const lp_march_cfg* cfg, const lp_rays* rays, const float* valid_mask,
                      const lp_grid_list* grad_grid, float* grad_feature) {
  LpRays R; LpMarch M; LpGridSet GG;
  int rc, lpr, vpl;
  if (!grad_grid || !grad_feature) LP_FAIL(LP_ERR_INVALID_ARG, "grad_grid / grad_feature is NULL");
  if ((rc = lp_make_march(cfg, &M))) return rc;
  if ((rc = lp_make_gridset(grad_grid, &GG, "grad_grid"))) return rc;
  if ((rc = lp_make_rays(rays, &R, GG.C))) return rc;
  if (R.n == 0) return LP_OK;
  if ((rc = lp_splat_geometry(GG.C, &lpr, &vpl))) return rc;
  if ((rc = lp_splat_rows_fit(GG, "grad_grid"))) return rc;
  const int threads = 128, rays_per_block = threads / lpr;
  dim3 g((R.n + rays_per_block - 1) / rays_per_block), b(threads);
  cudaStream_t st = (cudaStream_t)stream;
  switch (vpl) {
    case 1: LP_LAUNCH(lp_splat_bwd_kernel<1>, g, b, 0, st, R, M, GG, valid_mask, grad_feature, lpr); break;
    case 2: LP_LAUNCH(lp_splat_bwd_kernel<2>, g, b, 0, st, R, M, GG, valid_mask, grad_feature, lpr); break;
    case 4: LP_LAUNCH(lp_splat_bwd_kernel<4>, g, b, 0, st, R, M, GG, valid_mask, grad_feature, lpr); break;
    default: LP_LAUNCH(lp_splat_bwd_kernel<8>, g, b, 0, st, R, M, GG, valid_mask, grad_feature, lpr); break;
  }
  return lp_check_launch("lp_splat_backward");
}

int lp_splat_normalize(void* stream, float* feature_grid, float* weight_grid, int64_t num_rows, int32_t channels) {
  if (!feature_grid || !weight_grid) LP_FAIL(LP_ERR_INVALID_ARG, "feature_grid / weight_grid is NULL");
  if (channels % 4 != 0) LP_FAIL(LP_ERR_UNSUPPORTED, "channels must be a multiple of 4");
  if (num_rows <= 0) return LP_OK;
  const long long total = (long long)num_rows * (channels / 4);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  LP_LAUNCH(lp_splat_normalize_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream,
            feature_grid, weight_grid, (long long)num_rows, (int)channels);
  return lp_check_launch("lp_splat_normalize");
}

int lp_int_to_randn(void* stream, const int32_t* x1, const int32_t* x2, int32_t seed, float* out, int64_t n) {
  if (!x1 || !x2 || !out) LP_FAIL(LP_ERR_INVALID_ARG, "NULL pointer");
  if (n <= 0) return LP_OK;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  LP_LAUNCH(lp_int_to_randn_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, x1, x2,
            (int)seed, out, (long long)n);
  return lp_check_launch("lp_int_to_randn");
}

// ---- module glue: ray encoding and background epilogue (lp_ray_embed.cuh) ------------------------
static int lp_embed_check(int64_t n, const float* directions, int32_t n_harmonics, int32_t out_dim, int* items) {
  if (n < 0) LP_FAIL(LP_ERR_INVALID_ARG, "num_rays < 0");
  if (n > 0 && !directions) LP_FAIL(LP_ERR_INVALID_ARG, "directions is NULL");
  if (n_harmonics < 0 || n_harmonics > LP_EMB_MAX_HARM)
    LP_FAIL(LP_ERR_UNSUPPORTED, "n_harmonics=%d not in [0,%d]", n_harmonics, LP_EMB_MAX_HARM);
  if (out_dim < 4 || out_dim % 4 != 0) LP_FAIL(LP_ERR_UNSUPPORTED, "encoding_dim (%d) must be a positive multiple of 4", out_dim);
  *items = (3 + 6 * n_harmonics + 1) * (out_dim / 4);
  if (*items > LP_EMB_MAX_ITEMS * LP_EMB_TILE)
    LP_FAIL(LP_ERR_UNSUPPORTED, "(3 + 6 * n_harmonics + 1) * encoding_dim / 4 = %d exceeds %d", *items, LP_EMB_MAX_ITEMS * LP_EMB_TILE);
  return LP_OK;
}

int lp_ray_embed_forward(void* stream, int64_t num_rays, const float* directions, int32_t n_harmonics,
                         const float* weight, const float* bias, int32_t encoding_dim, float* encoding) {
  int rc, items;
  if ((rc = lp_embed_check(num_rays, directions, n_harmonics, encoding_dim, &items))) return rc;
  if (num_rays == 0) return LP_OK;
  if (!weight || !encoding) LP_FAIL(LP_ERR_INVALID_ARG, "weight / encoding is NULL");
  if (((uintptr_t)encoding & 15) != 0) LP_FAIL(LP_ERR_INVALID_ARG, "encoding is not 16-byte aligned");
  const int in_dim = 3 + 6 * n_harmonics;
  const size_t bytes = sizeof(float) * ((size_t)encoding_dim * in_dim + encoding_dim + (size_t)LP_EMB_TILE * (in_dim + 1));
  if (LP_SET_SMEM(lp_ray_embed_fwd_kernel, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
  long long blocks = (num_rays + LP_EMB_TILE - 1) / LP_EMB_TILE;
  if (blocks > 148 * 4) blocks = 148 * 4;
  LP_LAUNCH(lp_ray_embed_fwd_kernel, dim3((unsigned)blocks), dim3(LP_EMB_TILE), bytes, (cudaStream_t)stream, directions,
            (long long)num_rays, (int)n_harmonics, weight, bias, (int)encoding_dim, encoding);
  return lp_check_launch("lp_ray_embed_forward");
}

int lp_ray_embed_backward(void* stream, int64_t num_rays, const float* directions, int32_t n_harmonics,
                          const float* grad_encoding, int32_t encoding_dim, float* grad_weight, float* grad_bias) {
  int rc, items;
  if ((rc = lp_embed_check(num_rays, directions, n_harmonics, encoding_dim, &items))) return rc;
  if (num_rays == 0) return LP_OK;
  if (!grad_encoding || !grad_weight) LP_FAIL(LP_ERR_INVALID_ARG, "grad_encoding / grad_weight is NULL");
  if (((uintptr_t)grad_encoding & 15) != 0) LP_FAIL(LP_ERR_INVALID_ARG, "grad_encoding is not 16-byte aligned");
  const int in_dim = 3 + 6 * n_harmonics;
  const size_t bytes = sizeof(float) * (size_t)LP_EMB_TILE * ((in_dim + 2) + (encoding_dim + 4));
  if (LP_SET_SMEM(lp_ray_embed_bwd_kernel, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
  long long blocks = (num_rays + LP_EMB_TILE - 1) / LP_EMB_TILE;
  if (blocks > 148 * 2) blocks = 148 * 2;
  LP_LAUNCH(lp_ray_embed_bwd_kernel, dim3((unsigned)blocks), dim3(LP_EMB_TILE), bytes, (cudaStream_t)stream, directions,
            (long long)num_rays, (int)n_harmonics, grad_encoding, (int)encoding_dim, grad_weight, grad_bias);
  return lp_check_launch("lp_ray_embed_backward");
}

int lp_bg_composite_forward(void* stream, int64_t num_rays, int32_t channels, const float* nlt, const float* features,
                            const float* bg_color, int32_t return_log_transmittance, float* alpha, float* out) {
  if (num_rays < 0 || channels < 1) LP_FAIL(LP_ERR_INVALID_ARG, "num_rays < 0 or channels < 1");
  if (num_rays == 0) return LP_OK;
  if (!nlt || !features || !bg_color || !alpha || !out) LP_FAIL(LP_ERR_INVALID_ARG, "NULL pointer");
  long long blocks = (num_rays + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  LP_LAUNCH(lp_bg_fwd_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, (long long)num_rays,
            (int)channels, nlt, features, bg_color, (int)return_log_transmittance, alpha, out);
  return lp_check_launch("lp_bg_composite_forward");
}

int lp_bg_composite_backward(void* stream, int64_t num_rays, int32_t channels, const float* nlt, const float* bg_color,
                             int32_t return_log_transmittance, const float* grad_alpha, const float* grad_out,
                             float* grad_nlt) {
  if (num_rays < 0 || channels < 1) LP_FAIL(LP_ERR_INVALID_ARG, "num_rays < 0 or channels < 1");
  if (num_rays == 0) return LP_OK;
  if (!nlt || !bg_color || !grad_nlt) LP_FAIL(LP_ERR_INVALID_ARG, "NULL pointer");
  long long blocks = (num_rays + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  LP_LAUNCH(lp_bg_bwd_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, (long long)num_rays,
            (int)channels, nlt, bg_color, (int)return_log_transmittance, grad_alpha, grad_out, grad_nlt);
  return lp_check_launch("lp_bg_composite_backward");
}

// ---- MLP splatter -----------------------------------------------------------------------------
static int lp_make_splat_mlp(const lp_mlp_spec* s, int c_in, int c_out, LpSplatMlp* S) {
  if (!s) LP_FAIL(LP_ERR_INVALID_ARG, "mlp spec is NULL");
  memset(S, 0, sizeof(*S));
  if (s->n_layers < 1) LP_FAIL(LP_ERR_INVALID_ARG, "the splatter MLP needs at least one layer");
  if (s->dim_in != c_in || s->dim_out != c_out)
    LP_FAIL(LP_ERR_INVALID_ARG, "mlp dims (%d->%d) do not match feature/grid channels (%d->%d)",
            s->dim_in, s->dim_out, c_in, c_out);
  if (c_in % 4 != 0 || c_out % 4 != 0) LP_FAIL(LP_ERR_UNSUPPORTED, "channels must be multiples of 4");
  int pos = 0, rc;
  if ((rc = lp_fill_mlp(&S->mlp, s->n_layers, s->dim_in, s->dim_hidden, s->dim_out, s->dim_out, 0, &pos)))
    return rc;
  S->n_params = pos; S->c_in = c_in; S->c_out = c_out;
  int row = 0, md = imax(c_in, c_out);
  S->x0 = row; row += c_in;
  S->xin = row; row += c_in;
  for (int l = 0; l < S->mlp.n_layers; ++l) { S->y[l] = row; row += S->mlp.l[l].N; md = imax(md, S->mlp.l[l].N); }
  S->total = row; S->max_dim = md;
  return LP_OK;
}

int lp_mlp_splat_forward(void* stream, const lp_march_cfg* cfg, const lp_mlp_spec* spec, const lp_rays* rays,
                         const float* valid_mask, const lp_grid_list* input_grid, const float* mlp_params,
                         const lp_grid_list* out, float* weight_grid) {
  LpRays R; LpMarch M; LpGridSet IN, O; LpSplatMlp S;
  int rc;
  if (!input_grid || !out || !mlp_params) LP_FAIL(LP_ERR_INVALID_ARG, "NULL argument");
  if ((rc = lp_make_march(cfg, &M))) return rc;
  if ((rc = lp_make_gridset(input_grid, &IN, "input_grid"))) return rc;
  if ((rc = lp_make_gridset(out, &O, "out"))) return rc;
  if ((rc = lp_make_splat_mlp(spec, IN.C, O.C, &S))) return rc;
  if ((rc = lp_make_rays(rays, &R, IN.C))) return rc;
  if (IN.g[0].B != O.g[0].B) LP_FAIL(LP_ERR_INVALID_ARG, "input / output grid batch sizes differ");
  if (R.n == 0) return LP_OK;
  if (lptc::lp_tc_mlp_splat_supported(S, IN, O)) {
    if ((rc = lptc::lp_tc_mlp_splat_forward((cudaStream_t)stream, R, M, S, IN, O, weight_grid, valid_mask, mlp_params)))
      LP_FAIL(rc, "tensor-core MLP splatter launch setup failed");
    return lp_check_launch("lp_mlp_splat_forward(tc)");
  }
  const int pf = (S.n_params + 3) & ~3;
  const int per_warp = (S.total + S.c_in + S.c_out) * LP_LS;
  int warps, pin; size_t bytes;
  if ((rc = lp_plan_smem(0, pf, per_warp, &warps, &pin, &bytes))) return rc;
  if (LP_SET_SMEM(lp_mlp_splat_fwd_kernel, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
  const int rpb = warps * LP_WARP;
  LP_LAUNCH(lp_mlp_splat_fwd_kernel, dim3((R.n + rpb - 1) / rpb), dim3(rpb), bytes, (cudaStream_t)stream, R, M, S,
            IN, O, weight_grid, valid_mask, mlp_params, pin);
  return lp_check_launch("lp_mlp_splat_forward");
}

int lp_mlp_splat_backward(void* stream, const lp_march_cfg* cfg, const lp_mlp_spec* spec, const lp_rays* rays,
                          const float* valid_mask, const lp_grid_list* input_grid, const float* mlp_params,
                          const lp_grid_list* grad_grid, float* grad_feature, float* grad_mlp_params,
                          float* grad_input_grid) {
  LpRays R; LpMarch M; LpGridSet IN, GG; LpSplatMlp S;
  int rc;
  if (!input_grid || !grad_grid || !mlp_params || !grad_feature || !grad_mlp_params || !grad_input_grid)
    LP_FAIL(LP_ERR_INVALID_ARG, "NULL argument");
  if ((rc = lp_make_march(cfg, &M))) return rc;
  if ((rc = lp_make_gridset(input_grid, &IN, "input_grid"))) return rc;
  if ((rc = lp_make_gridset(grad_grid, &GG, "grad_grid"))) return rc;
  if (IN.g[0].B != GG.g[0].B) LP_FAIL(LP_ERR_INVALID_ARG, "input / gradient grid batch sizes differ");
  if ((rc = lp_make_splat_mlp(spec, IN.C, GG.C, &S))) return rc;
  if ((rc = lp_make_rays(rays, &R, IN.C))) return rc;
  if (R.n == 0) return LP_OK;
  if (lptc::lp_tc_mlp_splat_supported(S, IN, GG)) {
    if ((rc = lptc::lp_tc_mlp_splat_backward((cudaStream_t)stream, R, M, S, IN, GG, valid_mask, mlp_params, grad_feature,
                                             grad_mlp_params, grad_input_grid)))
      LP_FAIL(rc, "tensor-core MLP splatter launch setup failed");
    return lp_check_launch("lp_mlp_splat_backward(tc)");
  }
  const int pf = (S.n_params + 3) & ~3;
  const int per_warp = (S.total + 2 * S.max_dim + 2 * S.c_in) * LP_LS;
  int warps, pin; size_t bytes;
  if ((rc = lp_plan_smem(pf, pf, per_warp, &warps, &pin, &bytes))) return rc;
  if (LP_SET_SMEM(lp_mlp_splat_bwd_kernel, bytes)) LP_FAIL(LP_ERR_CUDA, "cannot raise dynamic smem limit");
  const int rpb = warps * LP_WARP;
  LP_LAUNCH(lp_mlp_splat_bwd_kernel, dim3((R.n + rpb - 1) / rpb), dim3(rpb), bytes, (cudaStream_t)stream, R, M, S,
            IN, GG, valid_mask, mlp_params, pin, grad_feature, grad_mlp_params, grad_input_grid);
  return lp_check_launch("lp_mlp_splat_backward");
}

}  // extern "C"
