/*
 * lightplane_b200 -- C-ABI of the B200-native Renderer / Splatter hot path.
 *
 * This is the drop-in boundary: the entry points below replace the six Triton kernel launches
 * of the reference (facebookresearch/lightplane).  Each one cites the reference launch site it
 * stands in for.  All `float*` / `int32_t*` data pointers are DEVICE pointers to contiguous
 * memory owned by the caller (PyTorch in the shipped binding); structs and size tables are HOST
 * memory, read synchronously during the call.  The library is stateless, allocates nothing that
 * outlives a call, launches on the stream it is given and never synchronises it.  Return value:
 * LP_OK (0) or an LP_ERR_* code; `lp_last_error()` gives a thread-local message.
 *
 * Conventions shared with the reference (docs/feature_grids.md:56-59, grid_sample_util.py:209-283):
 *   grid i has shape [B, D_i, H_i, W_i, C], world x -> W, y -> H, z -> D, coordinates in [-1,1],
 *   texel centres at align_corners=False positions, zero padding outside; a grid with all of
 *   D,H,W > 1 is a voxel grid, D==1 is the XY plane, H==1 the XZ plane, otherwise the YZ plane;
 *   the features of all grids in a list are summed.
 */
#ifndef LIGHTPLANE_B200_H
#define LIGHTPLANE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LP_ABI_VERSION 3
#define LP_MAX_GRIDS 8   /* grids per grid-list */
#define LP_MAX_LAYERS 8  /* layers per MLP */

enum lp_status {
  LP_OK = 0,
  LP_ERR_INVALID_ARG = 1, /* NULL / inconsistent sizes                        */
  LP_ERR_UNSUPPORTED = 2, /* valid request this build cannot serve            */
  LP_ERR_CUDA = 3,        /* a CUDA runtime call or launch failed             */
  LP_ERR_RESOURCE = 4     /* configuration does not fit shared memory         */
};

/* A flat grid-list.  `data` = [sum_i B*D_i*H_i*W_i, channels] fp32 (device).  For gradient /
 * output lists the library accumulates into `data` with atomics: the caller zero-fills it.
 * (reference: misc_utils.py:25-46 flatten_grid; sizes table = `feature_grid_sizes`) */
typedef struct lp_grid_list {
  float* data;
  int32_t num_grids;
  int32_t channels;
  int32_t sizes[LP_MAX_GRIDS][5]; /* (B, D, H, W, C) per grid, host values */
} lp_grid_list;

/* The ray batch (reference: ray_utils.py:19-57 `Rays`; kernel args lightplane_renderer.py:518-523). */
typedef struct lp_rays {
  const float* directions; /* [N,3] */
  const float* origins;    /* [N,3] */
  const int32_t* grid_idx; /* [N], 0 <= idx < B */
  const float* near;       /* [N] */
  const float* far;        /* [N] */
  const float* encoding;   /* [N, encoding_dim]: ray encoding (renderer) / splatted feature (splatter) */
  int32_t num_rays;
  int32_t encoding_dim;
} lp_rays;

/* Ray-march configuration (reference kernel constexprs: renderer_fw.py:115-132). */
typedef struct lp_march_cfg {
  int32_t num_samples;        /* equispaced samples in [near, far]                               */
  int32_t num_samples_inf;    /* extra samples beyond far, equispaced in disparity               */
  float gain;                 /* opacity scale                                                   */
  float disparity_at_inf;
  int32_t mask_out_of_bounds; /* zero samples outside [-1,1]^3                                   */
  int32_t contract_coords;    /* MERF contraction, then x0.5 (ray_util.py:12-45)                 */
  int32_t inject_noise;       /* add sigma * N(0,1) hash noise to raw opacity (rand_util.py:38-79) */
  float noise_sigma;
  int32_t noise_seed;
  int32_t noise_num_rays;     /* ray count used for the 2nd hash index: N rounded up to 16,
                                 as the reference pads rays (renderer_fw.py:290-294)              */
  int32_t ray_image_width;    /* scheduling hint, 0 = none: the N rays are a row-major image of this
                                 width (multiple of 16, N a multiple of 8 rows); the tensor-core
                                 kernels then walk 16x8-pixel tiles instead of 128-ray scan-line runs
                                 (texel-coherent gathers / reductions).  Results do not depend on it
                                 beyond floating-point summation order.                            */
} lp_march_cfg;

/* Decoder layout inside the flat `mlp_params` vector (reference: mlp_utils.py:390-456 and
 * lightplane_renderer.py:764-784): trunk, opacity, colour; per MLP all weights [in,out]
 * row-major, then all biases.  Trunk: ReLU after every layer incl. the last; opacity / colour:
 * ReLU between layers, linear last layer (renderer_mlp_util.py:100-112).  Opacity out dim = 1. */
typedef struct lp_decoder_spec {
  int32_t n_layers_trunk, n_layers_opacity, n_layers_color; /* trunk may be 0 (colour-grid mode) */
  int32_t dim_hidden_trunk, dim_hidden_opacity, dim_hidden_color;
  int32_t dim_in_trunk, dim_in_opacity, dim_in_color;
  int32_t dim_out_trunk;
  int32_t dim_out_color;  /* width of the last colour layer in the layout (16 when padded)      */
  int32_t num_color_used; /* channels rendered & written, 1..dim_out_color                       */
} lp_decoder_spec;

/* Single MLP of the MLP-splatter (reference: splatter_mlp_util.py; ReLU between layers only). */
typedef struct lp_mlp_spec {
  int32_t n_layers;
  int32_t dim_in, dim_hidden, dim_out;
} lp_mlp_spec;

int lp_abi_version(void);
const char* lp_last_error(void);
/* 1 if the library was compiled for the GPU (sm_100a), 0 for the test-only host emulation. */
int lp_is_device_build(void);

/* Renderer forward.  Replaces `fw_kernel[grid](...)`, lightplane_renderer.py:505-555 /
 * renderer_fw.py:85-375.  Outputs are fully written (no pre-zeroing needed).
 *   out_ray_length [N], out_neg_log_transmittance [N],
 *   out_features [N, features_stride] (first num_color_used columns written).
 * color_grid: NULL, or the separate colour grid-list (then n_layers_trunk must be 0).
 * scaffold:   NULL, or a 1-grid list [B,D,H,W,1] of 0/1 occupancy. */
int lp_render_forward(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                      const lp_rays* rays, const lp_grid_list* grid,
                      const lp_grid_list* color_grid, const lp_grid_list* scaffold,
                      const float* mlp_params, float* out_ray_length,
                      float* out_neg_log_transmittance, float* out_features,
                      int32_t features_stride);

/* Renderer backward.  Replaces `bw_kernel[grid](...)`, lightplane_renderer.py:657-711 /
 * renderer_bw.py:89-627.  Like the reference it stores nothing per sample and recomputes the
 * forward inside the kernel.  Unlike the reference it marches in FORWARD sample order: with
 * p_j = colour_j . g_feat + t_j * g_len and render weights w_j = T_{j-1} - T_j the opacity
 * gradient is  dL/d(delta_j*gain*o_j) = T_j p_j - sum_{k>j} w_k p_k + g_nlt,  and the suffix sum is
 * obtained as (g_feat . features + g_len * ray_length) - sum_{k<=j} w_k p_k from the saved
 * forward OUTPUTS.  The reference instead walks backwards and unrolls T_j by subtracting from the
 * saved final NLT (renderer_bw.py:429-433), which loses the low bits whenever later samples carry
 * huge step lengths (background samples: its Triton path is ~1e-2 off its own naive path there).
 * Same gradient, better conditioned.
 *   ray_length [N], features [N, features_stride]: the forward outputs.
 * grad_grid / grad_color_grid / grad_mlp_params are accumulated into (caller zero-fills);
 * grad_encoding [N, dim_in_color] is fully written. */
int lp_render_backward(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                       const lp_rays* rays, const lp_grid_list* grid,
                       const lp_grid_list* color_grid, const lp_grid_list* scaffold,
                       const float* mlp_params, const float* ray_length, const float* features,
                       int32_t features_stride, const float* grad_ray_length,
                       const float* grad_neg_log_transmittance, const float* grad_features,
                       int32_t grad_features_stride, float* grad_grid, float* grad_color_grid,
                       float* grad_mlp_params, float* grad_encoding);

/* Renderer backward with gradients w.r.t. the ray geometry (an extension; the reference has no
 * such gradients).  Arguments and outputs of lp_render_backward, plus
 *   grad_origins [N,3], grad_directions [N,3]: fully written; either may be NULL (not wanted).
 * With a sample at p_j = o + t_j d read at x_j = c(p_j) (c = the contraction or the identity) and
 * a_j the gradient w.r.t. its sampled feature row, g_j = sum_grids sum_taps <v_t, a_j> grad w_t(x_j),
 * dL/do = sum_j J_c(p_j)^T g_j and dL/dd = sum_j t_j J_c(p_j)^T g_j.  The OOB mask, scaffold and
 * noise are piecewise constant in position and add no terms; near / far get no gradient. */
int lp_render_backward_rays(void* stream, const lp_march_cfg* cfg, const lp_decoder_spec* spec,
                            const lp_rays* rays, const lp_grid_list* grid,
                            const lp_grid_list* color_grid, const lp_grid_list* scaffold,
                            const float* mlp_params, const float* ray_length, const float* features,
                            int32_t features_stride, const float* grad_ray_length,
                            const float* grad_neg_log_transmittance, const float* grad_features,
                            int32_t grad_features_stride, float* grad_grid, float* grad_color_grid,
                            float* grad_mlp_params, float* grad_encoding, float* grad_origins,
                            float* grad_directions);

/* Splatter forward.  Replaces BOTH launches of `fw_kernel` (features, then unit weights),
 * lightplane_splatter.py:503-539 / splatter_fw.py:71-165, in one pass: accumulates
 * encoding*valid into out->data [.., C] and valid into weight_grid [..] (may be NULL).
 * valid_mask [N] may be NULL (= all ones). */
int lp_splat_forward(void* stream, const lp_march_cfg* cfg, const lp_rays* rays,
                     const float* valid_mask, const lp_grid_list* out, float* weight_grid);

/* Splatter backward.  Replaces `bw_kernel`, lightplane_splatter.py:664 / splatter_bw.py:75-180:
 * grad_feature[r] = valid[r] * sum_j sample(grad_grid, x_rj); fully written.  grad_grid is the
 * upstream gradient already divided by the clamped weight grid (lightplane_splatter.py:608). */
int lp_splat_backward(void* stream, const lp_march_cfg* cfg, const lp_rays* rays,
                      const float* valid_mask, const lp_grid_list* grad_grid,
                      float* grad_feature);

/* MLP-splatter forward.  Replaces `fw_kernel_wMLP` + the weight launch, splatter_fw.py:168-309:
 * splat MLP(sample(input_grid, x) + encoding) * valid. */
int lp_mlp_splat_forward(void* stream, const lp_march_cfg* cfg, const lp_mlp_spec* spec,
                         const lp_rays* rays, const float* valid_mask,
                         const lp_grid_list* input_grid, const float* mlp_params,
                         const lp_grid_list* out, float* weight_grid);

/* MLP-splatter backward.  Replaces `bw_kernel_wMLP`, splatter_bw.py:183-394.  grad_feature is
 * fully written; grad_mlp_params / grad_input_grid accumulate (caller zero-fills). */
int lp_mlp_splat_backward(void* stream, const lp_march_cfg* cfg, const lp_mlp_spec* spec,
                          const lp_rays* rays, const float* valid_mask,
                          const lp_grid_list* input_grid, const float* mlp_params,
                          const lp_grid_list* grad_grid, float* grad_feature,
                          float* grad_mlp_params, float* grad_input_grid);

/* In-place `feat[r, :] /= max(weight[r], 1e-5)` and `weight[r] = max(weight[r], 1e-5)`.
 * Replaces the torch ops at lightplane_splatter.py:541,584. */
int lp_splat_normalize(void* stream, float* feature_grid, float* weight_grid, int64_t num_rows,
                       int32_t channels);

/* Hash -> Box-Muller normal noise of the opacity-noise feature, for the RNG parity test
 * (reference: rand_util.py:19-35 int_to_randn_kernel).  x1, x2 int32 [n]; out fp32 [n]. */
int lp_int_to_randn(void* stream, const int32_t* x1, const int32_t* x2, int32_t seed,
                    float* out, int64_t n);

/* ---- glue of the reference's renderer MODULE, fused (optional: the ops above do not need them) ----
 *
 * Ray encoding  encoding[r, :] = weight @ embed(normalize(directions[r])) + bias  with the harmonic
 * embedding  [sin(2^k d) | sin(2^k d + pi/2) | d]  (k < n_harmonics; per phase: x, y, z blocks of
 * n_harmonics columns).  Replaces, in one launch, `F.normalize` + `calc_harmonic_embedding`
 * (ray_utils.py:181-212) + `harmonic_ray_embedding_linear` (renderer_module.py:578-601).
 * weight fp32 [encoding_dim, 3 + 6 * n_harmonics] row-major (torch.nn.Linear layout), bias fp32
 * [encoding_dim] or NULL, encoding fp32 [num_rays, encoding_dim] fully written, 16-byte aligned. */
int lp_ray_embed_forward(void* stream, int64_t num_rays, const float* directions, int32_t n_harmonics,
                         const float* weight, const float* bias, int32_t encoding_dim, float* encoding);

/* Its backward: grad_weight [encoding_dim, 3 + 6 * n_harmonics] and grad_bias [encoding_dim] (may be
 * NULL) ACCUMULATE the sums over rays (caller zero-fills); directions get no gradient. */
int lp_ray_embed_backward(void* stream, int64_t num_rays, const float* directions, int32_t n_harmonics,
                          const float* grad_encoding, int32_t encoding_dim, float* grad_weight,
                          float* grad_bias);

/* Background epilogue of the module (renderer_module.py:552-563):
 *   T = exp(-nlt);  out = features + T * bg_color;  alpha = return_log_transmittance ? -nlt : 1 - T.
 * nlt, alpha fp32 [num_rays]; features, out fp32 [num_rays, channels]; bg_color fp32 [channels]. */
int lp_bg_composite_forward(void* stream, int64_t num_rays, int32_t channels, const float* nlt,
                            const float* features, const float* bg_color,
                            int32_t return_log_transmittance, float* alpha, float* out);

/* Its backward: grad_nlt [num_rays] fully written from grad_alpha [num_rays] and grad_out
 * [num_rays, channels] (either may be NULL = zero); d features = grad_out (no kernel needed). */
int lp_bg_composite_backward(void* stream, int64_t num_rays, int32_t channels, const float* nlt,
                             const float* bg_color, int32_t return_log_transmittance,
                             const float* grad_alpha, const float* grad_out, float* grad_nlt);

#ifdef __cplusplus
}
#endif
#endif /* LIGHTPLANE_B200_H */
