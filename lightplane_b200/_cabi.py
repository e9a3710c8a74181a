"""ctypes binding of `include/lightplane_b200.h` (the C-ABI shared library in `csrc/`).

The product path has exactly one implementation: the CUDA library.  If it is missing or was not
built for the GPU, `get_lib()` raises -- there is no CPU or PyTorch fallback.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

LP_MAX_GRIDS = 8
LP_ABI_VERSION = 3

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB_PATH = os.path.join(_HERE, "csrc", "liblightplane_b200.so")


class LightplaneB200Error(RuntimeError):
    pass


class GridList(C.Structure):
    _fields_ = [
        ("data", C.c_void_p),
        ("num_grids", C.c_int32),
        ("channels", C.c_int32),
        ("sizes", (C.c_int32 * 5) * LP_MAX_GRIDS),
    ]


class RaysStruct(C.Structure):
    _fields_ = [
        ("directions", C.c_void_p),
        ("origins", C.c_void_p),
        ("grid_idx", C.c_void_p),
        ("near", C.c_void_p),
        ("far", C.c_void_p),
        ("encoding", C.c_void_p),
        ("num_rays", C.c_int32),
        ("encoding_dim", C.c_int32),
    ]


class MarchCfg(C.Structure):
    _fields_ = [
        ("num_samples", C.c_int32),
        ("num_samples_inf", C.c_int32),
        ("gain", C.c_float),
        ("disparity_at_inf", C.c_float),
        ("mask_out_of_bounds", C.c_int32),
        ("contract_coords", C.c_int32),
        ("inject_noise", C.c_int32),
        ("noise_sigma", C.c_float),
        ("noise_seed", C.c_int32),
        ("noise_num_rays", C.c_int32),
        ("ray_image_width", C.c_int32),
    ]


class DecoderSpec(C.Structure):
    _fields_ = [
        ("n_layers_trunk", C.c_int32),
        ("n_layers_opacity", C.c_int32),
        ("n_layers_color", C.c_int32),
        ("dim_hidden_trunk", C.c_int32),
        ("dim_hidden_opacity", C.c_int32),
        ("dim_hidden_color", C.c_int32),
        ("dim_in_trunk", C.c_int32),
        ("dim_in_opacity", C.c_int32),
        ("dim_in_color", C.c_int32),
        ("dim_out_trunk", C.c_int32),
        ("dim_out_color", C.c_int32),
        ("num_color_used", C.c_int32),
    ]


class MlpSpec(C.Structure):
    _fields_ = [
        ("n_layers", C.c_int32),
        ("dim_in", C.c_int32),
        ("dim_hidden", C.c_int32),
        ("dim_out", C.c_int32),
    ]


_P = C.c_void_p
_PROTOTYPES = {
    "lp_abi_version": (C.c_int, []),
    "lp_last_error": (C.c_char_p, []),
    "lp_is_device_build": (C.c_int, []),
    "lp_render_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int32]),
    "lp_render_backward": (
        C.c_int,
        [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P],
    ),
    "lp_render_backward_rays": (
        C.c_int,
        [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P],
    ),
    "lp_splat_forward": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "lp_splat_backward": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "lp_mlp_splat_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "lp_mlp_splat_backward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "lp_splat_normalize": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32]),
    "lp_int_to_randn": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int64]),
    "lp_ray_embed_forward": (C.c_int, [_P, C.c_int64, _P, C.c_int32, _P, _P, C.c_int32, _P]),
    "lp_ray_embed_backward": (C.c_int, [_P, C.c_int64, _P, C.c_int32, _P, C.c_int32, _P, _P]),
    "lp_bg_composite_forward": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, _P, C.c_int32, _P, _P]),
    "lp_bg_composite_backward": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, C.c_int32, _P, _P, _P]),
}
EXPORTED_SYMBOLS = tuple(_PROTOTYPES)


def load_library(path: str) -> C.CDLL:
    """dlopen `path` and type every entry point `include/lightplane_b200.h` declares."""
    if not os.path.exists(path):
        raise LightplaneB200Error(
            f"lightplane_b200: CUDA library not found at {path}. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C lightplane_b200/csrc`). "
            "There is no CPU fallback."
        )
    lib = C.CDLL(path)
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.lp_abi_version() != LP_ABI_VERSION:
        raise LightplaneB200Error(
            f"lightplane_b200: ABI mismatch (library {lib.lp_abi_version()}, binding {LP_ABI_VERSION})"
        )
    return lib


_LIB: Optional[C.CDLL] = None


def get_lib() -> C.CDLL:
    """The product library (device build).  Raises if absent or if it is not a GPU build."""
    global _LIB
    if _LIB is None:
        lib = load_library(os.environ.get("LIGHTPLANE_B200_LIB", DEFAULT_LIB_PATH))
        if not lib.lp_is_device_build():
            raise LightplaneB200Error("lightplane_b200: library is not a device (sm_100a) build")
        _LIB = lib
    return _LIB


def check(lib: C.CDLL, status: int, what: str) -> None:
    if status != 0:
        msg = lib.lp_last_error()
        raise LightplaneB200Error(
            f"{what} failed with status {status}: {msg.decode() if msg else '?'}"
        )


# ------------------------------------------------------------------------------------------
# marshalling helpers (shared by the product ops and by the tests' low-level calls)
# ------------------------------------------------------------------------------------------
def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def f32c(t: torch.Tensor) -> torch.Tensor:
    """Contiguous fp32 view/copy (no-op for the normal case)."""
    if t.dtype != torch.float32:
        t = t.float()
    t = t if t.is_contiguous() else t.contiguous()
    if t.data_ptr() % 16 != 0:  # a view with an odd storage offset: the kernels use 16-byte vector accesses
        t = t.clone()
    return t


def make_grid_list(data: Optional[torch.Tensor], sizes: Sequence[Sequence[int]], channels=None) -> GridList:
    if len(sizes) > LP_MAX_GRIDS:
        raise LightplaneB200Error(f"at most {LP_MAX_GRIDS} grids per grid-list are supported")
    gl = GridList()
    gl.data = ptr(data)
    gl.num_grids = len(sizes)
    gl.channels = int(sizes[0][4] if channels is None else channels)
    rows = 0
    for i, s in enumerate(sizes):
        assert len(s) == 5
        for j in range(5):
            gl.sizes[i][j] = int(s[j])
        gl.sizes[i][4] = gl.channels
        rows += int(s[0]) * int(s[1]) * int(s[2]) * int(s[3])
    if data is not None:
        assert data.numel() == rows * gl.channels, (
            f"grid tensor has {data.numel()} elements, sizes imply {rows * gl.channels}"
        )
    return gl


def make_rays(directions, origins, grid_idx, near, far, encoding) -> RaysStruct:
    r = RaysStruct()
    r.directions, r.origins, r.grid_idx = ptr(directions), ptr(origins), ptr(grid_idx)
    r.near, r.far, r.encoding = ptr(near), ptr(far), ptr(encoding)
    r.num_rays = int(directions.shape[0])
    r.encoding_dim = 0 if encoding is None else int(encoding.shape[1])
    return r


def make_cfg(
    num_samples,
    num_samples_inf=0,
    gain=1.0,
    disparity_at_inf=1e-5,
    mask_out_of_bounds=False,
    contract_coords=False,
    noise_sigma=0.0,
    noise_seed=0,
    num_rays=0,
    ray_image_width=0,
) -> MarchCfg:
    c = MarchCfg()
    c.num_samples, c.num_samples_inf = int(num_samples), int(num_samples_inf)
    c.gain, c.disparity_at_inf = float(gain), float(disparity_at_inf)
    c.mask_out_of_bounds, c.contract_coords = int(bool(mask_out_of_bounds)), int(bool(contract_coords))
    c.inject_noise = int(noise_sigma > 0.0)
    c.noise_sigma = float(noise_sigma)
    # the hash works on int32 (rand_util.py:38-79): wrap python ints like a C cast would
    seed = int(noise_seed) & 0xFFFFFFFF
    c.noise_seed = seed - (1 << 32) if seed >= (1 << 31) else seed
    c.noise_num_rays = ((int(num_rays) + 15) // 16) * 16
    c.ray_image_width = int(ray_image_width or 0)
    return c


def stream_ptr(device: torch.device) -> Optional[int]:
    if device.type != "cuda":
        return None
    return torch.cuda.current_stream(device).cuda_stream


def byref(s: Optional[C.Structure]):
    """Pointer to a ctypes struct as c_void_p (None -> NULL)."""
    return None if s is None else C.cast(C.pointer(s), C.c_void_p)


# ------------------------------------------------------------------------------------------
# optional per-launch device timing (used by bench.py for the roofline numbers)
# ------------------------------------------------------------------------------------------
_PROFILE: Optional[list] = None


def profile_begin() -> None:
    """Start recording a CUDA-event pair around every C-ABI launch."""
    global _PROFILE
    _PROFILE = []


def profile_end():
    """Stop recording; returns `[(entry_point, milliseconds), ...]` (synchronises)."""
    global _PROFILE
    rec, _PROFILE = _PROFILE or [], None
    torch.cuda.synchronize()
    return [(name, a.elapsed_time(b)) for name, a, b in rec]


def call(lib, name: str, *args) -> int:
    """Invoke C-ABI entry point `name`; when profiling is on, bracket it with CUDA events recorded
    on the current stream (the one the launch goes to)."""
    fn = getattr(lib, name)
    if _PROFILE is None:
        return fn(*args)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    st = fn(*args)
    b.record()
    _PROFILE.append((name, a, b))
    return st
