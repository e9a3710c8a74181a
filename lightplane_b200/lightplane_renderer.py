"""Functional Lightplane Renderer bound to the sm_100a CUDA library.

Replaces the reference's `lightplane/lightplane_renderer.py`: `lightplane_renderer` (:33-293)
keeps its signature and return values; `LightplaneFunction` (:296-756) is the
`torch.autograd.Function` whose forward / backward now call `lp_render_forward` /
`lp_render_backward` of `include/lightplane_b200.h` instead of launching Triton kernels.

Extension: gradients w.r.t. the ray origins and directions (`lp_render_backward_rays`) when either
requires grad -- e.g. for refining camera poses from a photometric loss; the reference returns none.

Differences a caller can observe, all deliberate (DESIGN.md "Boundary"):
  * no host synchronisation: shapes are validated from metadata only; `grid_idx` range is
    clamped in the kernel (set `lightplane_renderer.VALIDATE_INPUTS = True` for the
    reference's device-side asserts, lightplane_renderer.py:464-467);
  * rays are not padded to a multiple of 16 and the padded colour channels are neither computed
    nor stored (the reference crops them right after the launch, :284-291);
  * `regenerate_code`, `triton_block_size`, `triton_num_warps` are accepted and ignored;
  * `rays.origins` / `rays.directions` that require grad receive their gradient (the reference's
    backward returns None for them); `near` / `far` still get none.
"""

from __future__ import annotations

import random
import warnings
from typing import List, Optional, Sequence, Tuple

import torch

from . import _cabi
from .misc_utils import check_grid_and_color_grid, process_and_flatten_grid
from .mlp_utils import MIN_BLOCK_SIZE, DecoderParams, get_triton_function_input_dims

# Opt-in device-side validation (costs host syncs, like the reference's asserts).
VALIDATE_INPUTS = False

import weakref

# id(tensor) -> (weakref to the tensor, _version, dims): an entry is valid only while the SAME tensor object is alive and
# unmodified, so a recycled address or id can never serve another decoder's dims (ADVICE r1).
_DIMS_CACHE: dict = {}


def _tensor_dims(t: torch.Tensor) -> List[int]:
    """`t.tolist()` as ints.  CPU tensors are read directly; device tensors are read back once per tensor object and
    version (the reference `.item()`s them every call, lightplane_renderer.py:221-233)."""
    if t.device.type == "cpu":
        return [int(v) for v in t.tolist()]
    ent = _DIMS_CACHE.get(id(t))
    if ent is not None and ent[0]() is t and ent[1] == t._version:
        return ent[2]
    dims = [int(v) for v in t.tolist()]
    key = id(t)
    _DIMS_CACHE[key] = (weakref.ref(t, lambda _r, k=key: _DIMS_CACHE.pop(k, None)), t._version, dims)
    return dims


def _decoder_dims(dp: DecoderParams):
    """Host copy of the decoder layer dims: `(triton-style dims, n_hidden_trunk, n_hidden_opacity, n_hidden_color)`."""
    nt, no, nc = (_tensor_dims(t) for t in (dp.n_hidden_trunk, dp.n_hidden_opacity, dp.n_hidden_color))
    return get_triton_function_input_dims(nt, no, nc), nt, no, nc


def _mlp_numel(d_in, d_hid, d_out, n_layers) -> int:
    """Parameter count of one MLP (reference: lightplane_renderer.py:764-784)."""
    if n_layers == 0:
        return 0
    if n_layers == 1:
        return d_in * d_out + d_out
    return d_in * d_hid + d_hid * d_hid * (n_layers - 2) + d_hid * d_out + d_hid * (n_layers - 1) + d_out


def lightplane_renderer(
    rays,
    grid,
    decoder_params: DecoderParams,
    # ------ config keys ------
    num_samples: int,
    gain: float,
    num_samples_inf: int = 0,
    mask_out_of_bounds_samples: bool = False,
    contract_coords: bool = False,
    disparity_at_inf: float = 1e-5,
    inject_noise_sigma: float = 0.0,
    inject_noise_seed: Optional[int] = None,
    scaffold: Optional[torch.Tensor] = None,
    color_grid=None,
    grid_sizes: Optional[List[List[int]]] = None,
    color_grid_sizes: Optional[List[List[int]]] = None,
    regenerate_code: bool = False,
    triton_block_size: int = 16,
    triton_num_warps: int = 4,
    ray_image_width: Optional[int] = None,
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Render `rays` through the feature grid-list `grid` (emission-absorption ray march).

    For each of `num_samples` equispaced depths in [near, far] (+ `num_samples_inf` samples
    beyond far, equispaced in disparity) the grid-list is tri/bi-linearly sampled, decoded by
    trunk -> (opacity, colour) MLPs and alpha-composited.  Arguments and semantics are those
    of the reference (lightplane_renderer.py:54-211).

    `ray_image_width` (extension, optional): when the N rays are a row-major image of that width
    (a multiple of 16, with a multiple of 8 rows) the kernels walk them in 16x8-pixel tiles, which
    makes the gathers / gradient reductions of a warp texel-coherent.  A scheduling hint only:
    results are those of the default order up to floating-point summation order.

    Returns `(ray_length_render [N], negative_log_transmittance [N], feature_render [N, color_chn])`.
    """
    del regenerate_code, triton_block_size, triton_num_warps  # Triton-era knobs: ignored
    grid, color_grid, grid_sizes, color_grid_sizes = check_grid_and_color_grid(
        grid, color_grid, grid_sizes, color_grid_sizes
    )
    grid, color_grid, grid_sizes, color_grid_sizes = process_and_flatten_grid(
        grid, color_grid, grid_sizes, color_grid_sizes
    )
    (hid_t, hid_o, hid_c, n_t, n_o, n_c, chn_layout), _, _, _ = _decoder_dims(decoder_params)

    if inject_noise_sigma > 0.0:
        if inject_noise_seed is None:
            inject_noise_seed = int(random.randint(0, 1000000))
    else:
        inject_noise_seed = 0

    return LightplaneFunction.apply(
        grid,
        decoder_params.mlp_params,
        rays.encoding,
        color_grid,
        # ---- non-differentiable ----
        grid_sizes,
        color_grid_sizes,
        rays.directions,
        rays.origins,
        rays.grid_idx,
        rays.near,
        rays.far,
        scaffold,
        (hid_t, hid_o, hid_c, n_t, n_o, n_c, chn_layout, int(decoder_params.color_chn)),
        int(num_samples),
        int(num_samples_inf),
        float(gain),
        bool(mask_out_of_bounds_samples),
        bool(contract_coords),
        float(disparity_at_inf),
        float(inject_noise_sigma),
        int(inject_noise_seed),
        int(ray_image_width or 0),
    )


class LightplaneFunction(torch.autograd.Function):
    """autograd binding of the fused ray-march kernels.

    Differentiable inputs: flat feature grid, mlp_params, ray encoding, flat colour grid
    (as in the reference, lightplane_renderer.py:724-756) and, as an extension, the ray directions
    and origins: when either requires grad the backward calls `lp_render_backward_rays`, which adds
    dL/d origin = sum_j J_c(p_j)^T g_j and dL/d direction = sum_j t_j J_c(p_j)^T g_j over the samples
    p_j = o + t_j d (g_j: the gradient w.r.t. the grid-space sample point; J_c: the contraction's
    Jacobian).  Without it the backward is exactly `lp_render_backward`.
    Only per-ray tensors are saved for backward (the forward outputs `ray_length`, `features`
    and the inputs) -- the backward kernel recomputes every per-sample quantity.
    """

    @staticmethod
    def forward(
        ctx,
        feature_grid: torch.Tensor,  # [sum BDHW, C]
        mlp_params: torch.Tensor,  # [P]
        ray_encoding: torch.Tensor,  # [N, dim_in_color]
        color_feature_grid: Optional[torch.Tensor],
        grid_sizes: Sequence[Sequence[int]],
        color_grid_sizes: Optional[Sequence[Sequence[int]]],
        directions: torch.Tensor,
        origins: torch.Tensor,
        grid_idx: torch.Tensor,
        near: torch.Tensor,
        far: torch.Tensor,
        scaffold: Optional[torch.Tensor],  # [B, D, H, W]
        mlp_dims: Tuple[int, ...],
        num_samples: int,
        num_samples_inf: int,
        gain: float,
        mask_out_of_bounds_samples: bool,
        contract_coords: bool,
        disparity_at_inf: float,
        inject_noise_sigma: float,
        inject_noise_seed: int,
        ray_image_width: int = 0,
    ):
        lib = _cabi.get_lib()
        device = feature_grid.device
        if device.type != "cuda":
            raise _cabi.LightplaneB200Error(
                "lightplane_renderer runs on CUDA tensors only (no CPU fallback); "
                f"got feature grid on {device}"
            )
        hid_t, hid_o, hid_c, n_t, n_o, n_c, chn_layout, color_chn = mlp_dims
        use_color_grid = color_feature_grid is not None
        num_rays = int(directions.shape[0])
        num_grid_channels = int(feature_grid.shape[-1])

        if mask_out_of_bounds_samples and contract_coords:
            warnings.warn(
                "The renderer has been configured to contract the coordinates lying outside the"
                " [-1,1] cube (contract_coords=True) and to also mask out all such points"
                " (mask_out_of_bounds_samples=True)."
            )

        # ---- layer dims exactly as the reference derives them (:383-401) ----
        if use_color_grid:
            assert n_t == 0, "mlp_n_layers_trunk has to be 0 when use_separate_color_grid"
            dim_in_trunk = dim_out_trunk = 0
            dim_in_opacity = dim_in_color = num_grid_channels
        else:
            assert n_t > 0, "a trunk MLP is required unless a separate color grid is given"
            dim_in_trunk, dim_out_trunk = num_grid_channels, hid_t
            dim_in_opacity = dim_in_color = hid_t
        assert 1 <= color_chn <= chn_layout

        # ---- metadata-only validation (reference asserts :403-467, minus the device reads) ----
        assert feature_grid.ndim == 2 and mlp_params.ndim == 1
        assert all(int(s[4]) == num_grid_channels for s in grid_sizes)
        batch = int(grid_sizes[0][0])
        assert all(int(s[0]) == batch for s in grid_sizes), "all grids must share the batch size"
        assert tuple(directions.shape) == (num_rays, 3) and tuple(origins.shape) == (num_rays, 3)
        for t in (grid_idx, near, far):
            assert tuple(t.shape) == (num_rays,)
        assert ray_encoding is not None and tuple(ray_encoding.shape) == (num_rays, dim_in_color), (
            f"ray_encoding should be [{num_rays}, {dim_in_color}], got "
            f"{None if ray_encoding is None else tuple(ray_encoding.shape)}"
        )
        expected = (
            _mlp_numel(dim_in_trunk, hid_t, dim_out_trunk, n_t)
            + _mlp_numel(dim_in_opacity, hid_o, 1, n_o)
            + _mlp_numel(dim_in_color, hid_c, chn_layout, n_c)
        )
        assert expected == mlp_params.numel(), (
            f"The number of elements in mlp param should be {expected}. Got {mlp_params.numel()} instead."
        )
        if use_color_grid:
            assert int(color_feature_grid.shape[-1]) == num_grid_channels
        if scaffold is not None:
            assert scaffold.ndim == 4 and int(scaffold.shape[0]) == batch
        if VALIDATE_INPUTS:
            assert int(grid_idx.min()) >= 0, "Negative grid index"
            assert int(grid_idx.max()) <= batch - 1, "A grid index is out of bounds"

        # ---- marshal ----
        feature_grid_c = _cabi.f32c(feature_grid)
        mlp_params_c = _cabi.f32c(mlp_params)
        enc_c = _cabi.f32c(ray_encoding)
        color_c = _cabi.f32c(color_feature_grid) if use_color_grid else None
        dirs_c, orig_c = _cabi.f32c(directions), _cabi.f32c(origins)
        near_c, far_c = _cabi.f32c(near), _cabi.f32c(far)
        gidx_c = grid_idx.to(torch.int32).contiguous()
        scaf_c = _cabi.f32c(scaffold) if scaffold is not None else None

        cfg = _cabi.make_cfg(
            num_samples,
            num_samples_inf,
            gain,
            disparity_at_inf,
            mask_out_of_bounds_samples,
            contract_coords,
            inject_noise_sigma,
            inject_noise_seed,
            num_rays,
            ray_image_width,
        )
        spec = _cabi.DecoderSpec(
            n_t, n_o, n_c, hid_t, hid_o, hid_c, dim_in_trunk, dim_in_opacity, dim_in_color,
            dim_out_trunk, chn_layout, color_chn,
        )
        rays_s = _cabi.make_rays(dirs_c, orig_c, gidx_c, near_c, far_c, enc_c)
        grid_s = _cabi.make_grid_list(feature_grid_c, grid_sizes)
        color_s = _cabi.make_grid_list(color_c, color_grid_sizes) if use_color_grid else None
        scaf_s = (
            _cabi.make_grid_list(scaf_c, [list(scaffold.shape) + [1]]) if scaffold is not None else None
        )

        ray_length = torch.empty(num_rays, device=device, dtype=torch.float32)
        nlt = torch.empty(num_rays, device=device, dtype=torch.float32)
        features = torch.empty(num_rays, color_chn, device=device, dtype=torch.float32)
        if num_rays > 0:
            with torch.cuda.device(device):
                st = _cabi.call(lib, "lp_render_forward",
                    _cabi.stream_ptr(device),
                    _byref(cfg), _byref(spec), _byref(rays_s), _byref(grid_s),
                    _byref(color_s), _byref(scaf_s),
                    mlp_params_c.data_ptr(),
                    ray_length.data_ptr(), nlt.data_ptr(), features.data_ptr(), color_chn,
                )
            _cabi.check(lib, st, "lp_render_forward")

        ctx.save_for_backward(
            ray_length, features, feature_grid_c, mlp_params_c, enc_c, color_c, dirs_c, orig_c,
            gidx_c, near_c, far_c, scaf_c,
        )
        ctx.ray_dtypes = (directions.dtype, origins.dtype)
        ctx.lp = (cfg, spec, grid_sizes, color_grid_sizes,
                  None if scaffold is None else list(scaffold.shape) + [1], color_chn)
        return ray_length, nlt, features

    @staticmethod
    def backward(ctx, grad_ray_length, grad_nlt, grad_features):
        lib = _cabi.get_lib()
        (ray_length, features, feature_grid, mlp_params, enc, color_grid, dirs, orig, gidx, near, far,
         scaf) = ctx.saved_tensors
        cfg, spec, grid_sizes, color_grid_sizes, scaf_size, color_chn = ctx.lp
        device = feature_grid.device
        num_rays = int(dirs.shape[0])

        def _g(t, shape):
            if t is None:
                return torch.zeros(shape, device=device, dtype=torch.float32)
            return _cabi.f32c(t)

        g_len = _g(grad_ray_length, (num_rays,))
        g_nlt = _g(grad_nlt, (num_rays,))
        g_feat = _g(grad_features, (num_rays, color_chn))

        grad_grid = torch.zeros_like(feature_grid)
        grad_mlp = torch.zeros_like(mlp_params)
        grad_enc = torch.empty_like(enc)
        grad_color = torch.zeros_like(color_grid) if color_grid is not None else None

        rays_s = _cabi.make_rays(dirs, orig, gidx, near, far, enc)
        grid_s = _cabi.make_grid_list(feature_grid, grid_sizes)
        color_s = _cabi.make_grid_list(color_grid, color_grid_sizes) if color_grid is not None else None
        scaf_s = _cabi.make_grid_list(scaf, [scaf_size]) if scaf is not None else None

        # inputs 6 / 7 of forward(): directions, origins
        want_dir, want_org = ctx.needs_input_grad[6], ctx.needs_input_grad[7]
        grad_dir = torch.empty_like(dirs) if want_dir else None
        grad_org = torch.empty_like(orig) if want_org else None
        args = (_cabi.stream_ptr(device),
                _byref(cfg), _byref(spec), _byref(rays_s), _byref(grid_s),
                _byref(color_s), _byref(scaf_s),
                mlp_params.data_ptr(), ray_length.data_ptr(), features.data_ptr(), color_chn,
                g_len.data_ptr(), g_nlt.data_ptr(), g_feat.data_ptr(), color_chn,
                grad_grid.data_ptr(), _cabi.ptr(grad_color), grad_mlp.data_ptr(),
                grad_enc.data_ptr())
        entry = "lp_render_backward_rays" if (want_dir or want_org) else "lp_render_backward"
        if entry == "lp_render_backward_rays":
            args += (_cabi.ptr(grad_org), _cabi.ptr(grad_dir))
        if num_rays > 0:
            with torch.cuda.device(device):
                st = _cabi.call(lib, entry, *args)
            _cabi.check(lib, st, entry)
        else:
            grad_enc.zero_()
        if grad_dir is not None:
            grad_dir = grad_dir.to(ctx.ray_dtypes[0])
        if grad_org is not None:
            grad_org = grad_org.to(ctx.ray_dtypes[1])

        return (grad_grid, grad_mlp, grad_enc, grad_color, None, None, grad_dir, grad_org) + (None,) * 14


def _byref(s):
    return _cabi.byref(s)
