"""Gradients w.r.t. the ray origins and directions (`lp_render_backward_rays`, an extension over the reference)
against fp64 autograd through the oracle, which forms the sample points as origins + depths * directions and
interpolates with differentiable fractions.  CPU tests run the kernels in the host emulation (tests/hostsim/) on the
tensor-core path and, with LP_ONLY_GENERIC=1, on the generic path; `-m gpu` tests go through the autograd op."""
import os
import subprocess

import pytest
import torch

from _golden import case_names, coherent_case, load_case, rel_err, renderer_cfg, synthetic_case
from _lowlevel import decoder_spec
from lightplane_b200 import _cabi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "hostsim", "liblp_hostsim.so")
CSRC = os.path.join(os.path.dirname(HERE), "lightplane_b200", "csrc")

TOL_RAYS = {"tc": 1e-3, "generic": 2e-4}  # ray-geometry gradients; the other outputs keep the renderer tests' bounds


def _tol(k, path):
    if k in ("g_origins", "g_directions"):
        return TOL_RAYS[path]
    return 6e-3 if k == "g_mlp" else (1e-3 if k.startswith("g_") else 2e-4)


def oracle_rays_case(c, dtype=torch.float64):
    """Oracle outputs and gradients of a renderer case, origins and directions included."""
    from oracle import lightplane_oracle as O

    f = lambda t: t.detach().to(dtype=dtype, device="cpu")
    grid, mlp, enc = (f(c[k]).requires_grad_(True) for k in ("grid", "mlp_params", "encoding"))
    dirs, orig = f(c["directions"]).requires_grad_(True), f(c["origins"]).requires_grad_(True)
    cgrid = f(c["color_grid"]).requires_grad_(True) if "color_grid" in c else None
    sizes = [[int(v) for v in s] for s in c["grid_sizes"]]
    color_chn = int(c["color_chn"])
    outs = O.render(
        dirs, orig, c["grid_idx"].cpu().long(), f(c["near"]), f(c["far"]), enc, grid, sizes, mlp,
        [int(v) for v in c["n_hidden_trunk"]], [int(v) for v in c["n_hidden_opacity"]], [int(v) for v in c["n_hidden_color"]],
        scaffold=f(c["scaffold"]) if "scaffold" in c else None, color_grid_flat=cgrid,
        color_grid_sizes=sizes if cgrid is not None else None, **renderer_cfg(c),
    )
    ray_length, nlt, feats = outs[0], outs[1], outs[2][:, :color_chn]
    loss = (f(c["cot_ray_length"]) * ray_length).sum() + (f(c["cot_nlt"]) * nlt).sum() + (f(c["cot_features"]) * feats).sum()
    leaves = [grid, mlp, enc, orig, dirs] + ([cgrid] if cgrid is not None else [])
    g = torch.autograd.grad(loss, leaves)
    res = dict(ray_length=ray_length, nlt=nlt, features=feats, g_grid=g[0], g_mlp=g[1], g_enc=g[2], g_origins=g[3],
               g_directions=g[4])
    if cgrid is not None:
        res["g_color_grid"] = g[5]
    return {k: v.detach() for k, v in res.items()}


def render_rays_case(lib, c, device, want_origins=True, want_directions=True):
    """forward + lp_render_backward_rays of a renderer case through the raw C-ABI."""
    f = lambda k: c[k].to(device=device, dtype=torch.float32).contiguous()
    cfgd = renderer_cfg(c)
    n = c["directions"].shape[0]
    color_chn = int(c["color_chn"])
    sizes = [[int(v) for v in s] for s in c["grid_sizes"]]
    dirs, orig, near, far, enc = f("directions"), f("origins"), f("near"), f("far"), f("encoding")
    gidx = c["grid_idx"].to(device=device, dtype=torch.int32).contiguous()
    grid, mlp = f("grid"), f("mlp_params")
    cgrid = f("color_grid") if "color_grid" in c else None
    scaf = f("scaffold") if "scaffold" in c else None
    cfg = _cabi.make_cfg(cfgd["num_samples"], cfgd["num_samples_inf"], cfgd["gain"], cfgd["disparity_at_inf"],
                         cfgd["mask_out_of_bounds_samples"], cfgd["contract_coords"], cfgd["inject_noise_sigma"],
                         cfgd["inject_noise_seed"], n)
    spec = decoder_spec(c)
    rays = _cabi.make_rays(dirs, orig, gidx, near, far, enc)
    gl = _cabi.make_grid_list(grid, sizes)
    cl = _cabi.make_grid_list(cgrid, sizes) if cgrid is not None else None
    sl = _cabi.make_grid_list(scaf, [list(scaf.shape) + [1]]) if scaf is not None else None
    B = _cabi.byref
    stream = _cabi.stream_ptr(torch.device(device))
    out_len, out_nlt, out_feat = torch.empty(n, device=device), torch.empty(n, device=device), torch.empty(n, color_chn, device=device)
    st = lib.lp_render_forward(stream, B(cfg), B(spec), B(rays), B(gl), B(cl), B(sl), mlp.data_ptr(),
                               out_len.data_ptr(), out_nlt.data_ptr(), out_feat.data_ptr(), color_chn)
    _cabi.check(lib, st, "lp_render_forward")
    g_grid, g_mlp, g_enc = torch.zeros_like(grid), torch.zeros_like(mlp), torch.empty_like(enc)
    g_cgrid = torch.zeros_like(cgrid) if cgrid is not None else None
    g_org = torch.full_like(orig, float("nan")) if want_origins else None
    g_dir = torch.full_like(dirs, float("nan")) if want_directions else None
    cl2, cn, cf = f("cot_ray_length"), f("cot_nlt"), f("cot_features")
    st = lib.lp_render_backward_rays(stream, B(cfg), B(spec), B(rays), B(gl), B(cl), B(sl), mlp.data_ptr(),
                                     out_len.data_ptr(), out_feat.data_ptr(), color_chn, cl2.data_ptr(), cn.data_ptr(),
                                     cf.data_ptr(), color_chn, g_grid.data_ptr(), _cabi.ptr(g_cgrid), g_mlp.data_ptr(),
                                     g_enc.data_ptr(), _cabi.ptr(g_org), _cabi.ptr(g_dir))
    _cabi.check(lib, st, "lp_render_backward_rays")
    res = dict(ray_length=out_len, nlt=out_nlt, features=out_feat, g_grid=g_grid, g_mlp=g_mlp, g_enc=g_enc)
    if g_org is not None:
        res["g_origins"] = g_org
    if g_dir is not None:
        res["g_directions"] = g_dir
    if g_cgrid is not None:
        res["g_color_grid"] = g_cgrid
    return res


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["make", "-s", "-C", CSRC, "hostsim"], check=True)
    lib = _cabi.load_library(LIB)
    assert lib.lp_is_device_build() == 0
    return lib


def _cases():
    out = [(name, lambda name=name: load_case(name)) for name in case_names("render_")]
    out.append(("coherent_mask_scaffold_c32", lambda: coherent_case(load_case("render_c32_b1"), n=64, pixel=0.03, mask_oob=1,
                                                                    scaffold_res=6)))
    out.append(("coherent_mask_scaffold_c16", lambda: coherent_case(load_case("render_triplane_inf_gain"), n=64, pixel=0.08,
                                                                    mask_oob=1, scaffold_res=8)))
    out.append(("empty_space_folding", lambda: coherent_case(load_case("render_triplane_inf_gain"), n=160, pixel=0.01, mask_oob=0,
                                                             origin=(1.3, -0.2, -3.0), near=0.3, far=6.0)))
    return out


CASES = dict(_cases())


def _check(got, want, path, label):
    for k, v in got.items():
        assert torch.isfinite(v).all(), (label, k)
        err = rel_err(v, want[k])
        assert err < _tol(k, path), (label, path, k, err)


@pytest.mark.parametrize("path", ["tc", "generic"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_hostsim_ray_grads_vs_oracle(lib, monkeypatch, name, path):
    if path == "generic":
        monkeypatch.setenv("LP_ONLY_GENERIC", "1")
    c = CASES[name]()
    want = oracle_rays_case(c)
    assert float(want["g_origins"].abs().sum()) > 0 and float(want["g_directions"].abs().sum()) > 0, name
    _check(render_rays_case(lib, c, "cpu"), want, path, name)


@pytest.mark.parametrize("path", ["tc", "generic"])
def test_hostsim_ray_grads_one_pointer(lib, monkeypatch, path):
    """Either output may be NULL; the other is still fully written."""
    if path == "generic":
        monkeypatch.setenv("LP_ONLY_GENERIC", "1")
    c = coherent_case(load_case("render_triplane_inf_gain"), n=64, pixel=0.05, mask_oob=0)
    want = oracle_rays_case(c)
    got = render_rays_case(lib, c, "cpu", want_directions=False)
    assert "g_directions" not in got
    _check(got, want, path, "origins only")
    got = render_rays_case(lib, c, "cpu", want_origins=False)
    assert "g_origins" not in got
    _check(got, want, path, "directions only")


@pytest.mark.parametrize("kind", ["color_grid", "hidden64", "layers_424"])
def test_hostsim_ray_grads_other_decoders_take_generic_kernel(lib, kind):
    """Decoders served by the other tensor-core kernels: ray-geometry requests run the generic kernel."""
    if kind == "color_grid":
        c = synthetic_case(n=64, C=16, sigma=0.5)
    elif kind == "hidden64":
        c = synthetic_case(n=64, C=16, hidden=64, layers=(2, 2, 2), color_grid=False)
    else:
        c = synthetic_case(n=64, C=16, hidden=32, layers=(4, 2, 4), color_grid=False)
    _check(render_rays_case(lib, c, "cpu"), oracle_rays_case(c), "generic", kind)


def test_hostsim_ray_grads_contraction(lib, monkeypatch):
    """Contracted coordinates with rays that leave the unit cube: J_c's off-diagonal terms through the max-norm."""
    c = coherent_case(load_case("render_triplane_inf_gain"), n=64, pixel=0.06, mask_oob=0, origin=(0.4, -0.3, -1.6),
                      near=0.2, far=4.0)
    cfg = c["cfg"].copy()
    cfg[3] = 1
    c["cfg"] = cfg
    want = oracle_rays_case(c)
    _check(render_rays_case(lib, c, "cpu"), want, "tc", "contract")
    monkeypatch.setenv("LP_ONLY_GENERIC", "1")
    _check(render_rays_case(lib, c, "cpu"), want, "generic", "contract")


# =====================================================================================================================
# GPU: the autograd op
# =====================================================================================================================
def _op_vs_oracle(c, dev="cuda", ray_image_width=None):
    """lightplane_renderer with requires_grad on origins and directions vs the oracle; returns relative errors."""
    import numpy as np

    import lightplane_b200 as lp

    want = oracle_rays_case(c)
    f = lambda k: c[k].to(dev).float()
    sizes = [[int(v) for v in s] for s in c["grid_sizes"]]
    rows = [int(np.prod(s[:4])) for s in sizes]
    grid = f("grid").requires_grad_(True)
    grids = [g.reshape(s) for g, s in zip(torch.split(grid, rows), sizes)]
    cgrid = f("color_grid").requires_grad_(True) if "color_grid" in c else None
    cgrids = [g.reshape(s) for g, s in zip(torch.split(cgrid, rows), sizes)] if cgrid is not None else None
    mlp, enc = f("mlp_params").requires_grad_(True), f("encoding").requires_grad_(True)
    dirs, orig = f("directions").requires_grad_(True), f("origins").requires_grad_(True)
    dp = lp.DecoderParams(mlp, torch.as_tensor(c["n_hidden_trunk"]), torch.as_tensor(c["n_hidden_opacity"]),
                          torch.as_tensor(c["n_hidden_color"]), int(c["color_chn"]))
    rays = lp.Rays(directions=dirs, origins=orig, grid_idx=c["grid_idx"].to(dev), near=f("near"), far=f("far"), encoding=enc)
    cfg = renderer_cfg(c)
    scaf = f("scaffold") if "scaffold" in c else None
    outs = lp.lightplane_renderer(rays, grids, dp, scaffold=scaf, color_grid=cgrids, ray_image_width=ray_image_width, **cfg)
    loss = (f("cot_ray_length") * outs[0]).sum() + (f("cot_nlt") * outs[1]).sum() + (f("cot_features") * outs[2]).sum()
    leaves = [grid, mlp, enc, orig, dirs] + ([cgrid] if cgrid is not None else [])
    g = torch.autograd.grad(loss, leaves)
    got = dict(ray_length=outs[0], nlt=outs[1], features=outs[2], g_grid=g[0], g_mlp=g[1], g_enc=g[2], g_origins=g[3],
               g_directions=g[4])
    if cgrid is not None:
        got["g_color_grid"] = g[5]
    return {k: rel_err(v, want[k]) for k, v in got.items()}


def _gpu_cases():
    return {
        **{name: (lambda name=name: load_case(name)) for name in case_names("render_")},
        "color_grid": lambda: synthetic_case(n=256, C=16, sigma=0.5),
        "hidden64": lambda: synthetic_case(n=256, C=32, hidden=64, layers=(2, 2, 2), color_grid=False),
        "layers_424": lambda: synthetic_case(n=256, C=16, hidden=32, layers=(4, 2, 4), color_grid=False),
    }


GPU_CASES = _gpu_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GPU_CASES))
def test_gpu_ray_grads_vs_oracle(name):
    errs = _op_vs_oracle(GPU_CASES[name]())
    print(name, {k: f"{v:.1e}" for k, v in errs.items()})
    for k, v in errs.items():
        tol = 1e-3 if k in ("g_origins", "g_directions") else (3e-3 if k == "g_mlp" else (1e-3 if k.startswith("g_") else 2e-4))
        assert v < tol, (name, k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("tile_walk", [False, True])
def test_gpu_ray_grads_bench_camera(tile_walk):
    """The bench-camera baseline of test_gpu_baseline_configs.py: 4096 rays x 128 samples, 64^2 x 16 triplane."""
    import lightplane_b200 as lp
    from bench import camera_rays
    from oracle import lightplane_oracle as O

    dev, side, S, C, H = "cuda", 64, 128, 16, 32
    torch.manual_seed(0)
    dp = lp.init_decoder_params(dev, 2, 2, 2, input_chn=C, hidden_chn=H, color_chn=3, opacity_init_bias=-1.0)
    shapes = [[1, 1, 64, 64, C], [1, 64, 1, 64, C], [1, 64, 64, 1, C]]
    grids = [0.5 * torch.randn(s, device=dev) for s in shapes]
    d, o, gi, nr, fr = [t.to(dev) for t in camera_rays(side, side, 1000, "cpu")]
    n = side * side
    g = torch.Generator().manual_seed(11)
    enc = torch.randn(n, H, generator=g).to(dev)
    target = torch.rand(n, 3, generator=g).to(dev)
    dd, oo = d.clone().requires_grad_(True), o.clone().requires_grad_(True)
    rays = lp.Rays(directions=dd, origins=oo, grid_idx=gi, near=nr, far=fr, encoding=enc)
    outs = lp.lightplane_renderer(rays, grids, dp, num_samples=S, gain=1.0, ray_image_width=side if tile_walk else None)
    g_o, g_d = torch.autograd.grad(((outs[2] - target) ** 2).mean(), [oo, dd])
    f = lambda t: t.detach().double().cpu()
    od, oorg = f(d).requires_grad_(True), f(o).requires_grad_(True)
    og = f(torch.cat([x.reshape(-1, C) for x in grids], 0))
    res = O.render(od, oorg, gi.cpu().long(), f(nr), f(fr), f(enc), og, shapes, f(dp.mlp_params), [C, H, H], [H, H, 1],
                   [H, H, 16], num_samples=S, gain=1.0)
    w_o, w_d = torch.autograd.grad(((res[2][:, :3] - f(target)) ** 2).mean(), [oorg, od])
    errs = dict(g_origins=rel_err(g_o, w_o), g_directions=rel_err(g_d, w_d))
    print("bench camera 4096x128 ray-geometry gradients vs fp64 oracle:", {k: f"{v:.1e}" for k, v in errs.items()})
    assert max(errs.values()) < 1e-3, errs


@pytest.mark.gpu
def test_gpu_ray_grads_routing():
    """Without a geometry gradient the backward is lp_render_backward; with one it is lp_render_backward_rays."""
    import lightplane_b200 as lp

    c = load_case("render_triplane_inf_gain")
    dev = "cuda"
    f = lambda k: c[k].to(dev).float()
    sizes = [[int(v) for v in s] for s in c["grid_sizes"]]
    import numpy as np

    rows = [int(np.prod(s[:4])) for s in sizes]
    grid = f("grid").requires_grad_(True)
    dp = lp.DecoderParams(f("mlp_params"), torch.as_tensor(c["n_hidden_trunk"]), torch.as_tensor(c["n_hidden_opacity"]),
                          torch.as_tensor(c["n_hidden_color"]), int(c["color_chn"]))
    for geo in (False, True):
        orig = f("origins").requires_grad_(geo)
        rays = lp.Rays(directions=f("directions"), origins=orig, grid_idx=c["grid_idx"].to(dev), near=f("near"), far=f("far"),
                       encoding=f("encoding"))
        grids = [g.reshape(s) for g, s in zip(torch.split(grid, rows), sizes)]
        outs = lp.lightplane_renderer(rays, grids, dp, **renderer_cfg(c))
        _cabi.profile_begin()
        leaves = [grid, orig] if geo else [grid]
        grads = torch.autograd.grad(outs[2].sum(), leaves)
        names = [nm for nm, _ in _cabi.profile_end()]
        assert ("lp_render_backward_rays" in names) == geo and ("lp_render_backward" in names) == (not geo), names
        if geo:
            assert grads[1].dtype == orig.dtype and grads[1].shape == orig.shape and bool(torch.isfinite(grads[1]).all())


@pytest.mark.gpu
def test_gpu_eval_opacity_at_points_gradient():
    """d opacity / d pts (density normals) through eval_opacity_at_points' zero-direction rays."""
    import lightplane_b200 as lp
    from oracle import lightplane_oracle as O

    dev = "cuda"
    torch.manual_seed(2)
    C, H = 16, 32
    m = lp.LightplaneRenderer(num_samples=8, color_chn=3, grid_chn=C, mlp_hidden_chn=H, opacity_init_bias=-1.0).to(dev)
    shapes = [[1, 1, 12, 13, C], [1, 11, 1, 13, C], [1, 11, 12, 1, C]]
    grids = [torch.randn(s, device=dev) for s in shapes]
    pts = (torch.rand(7, 50, 3, device=dev) * 1.8 - 0.9).requires_grad_(True)
    idx = torch.zeros(7, dtype=torch.long, device=dev)
    opa = m.eval_opacity_at_points(pts, idx, grids)
    (g_pts,) = torch.autograd.grad(opa.sum(), [pts])

    f = lambda t: t.detach().double().cpu()
    p = f(pts).reshape(-1, 3).requires_grad_(True)
    n = p.shape[0]
    nt, no, nc = (m.n_hidden_trunk.tolist(), m.n_hidden_opacity.tolist(), m.n_hidden_color.tolist())
    res = O.render(torch.zeros(n, 3, dtype=torch.float64), p, torch.zeros(n, dtype=torch.long), torch.zeros(n, dtype=torch.float64),
                   torch.ones(n, dtype=torch.float64), torch.zeros(n, m.rays_encoding_dim, dtype=torch.float64),
                   f(torch.cat([x.reshape(-1, C) for x in grids], 0)), shapes, f(m.mlp_params), nt, no, nc, num_samples=2,
                   gain=float(m.gain))
    (w,) = torch.autograd.grad((0.5 * res[1]).sum(), [p])
    err = rel_err(g_pts.reshape(-1, 3), w)
    print("eval_opacity_at_points d/d pts error vs fp64 oracle:", f"{err:.1e}")
    assert err < 1e-3, err


@pytest.mark.gpu
def test_gpu_pose_refinement_reduces_error():
    """A learnable offset on the origins of one view, started from a perturbed value, converges back towards the offset
    the target view was rendered with (photometric MSE, Adam)."""
    import lightplane_b200 as lp
    from bench import camera_rays

    dev, side, S, C, H = "cuda", 48, 64, 16, 32
    torch.manual_seed(7)
    dp = lp.init_decoder_params(dev, 2, 2, 2, input_chn=C, hidden_chn=H, color_chn=3, opacity_init_bias=-1.0)
    shapes = [[1, 1, 32, 32, C], [1, 32, 1, 32, C], [1, 32, 32, 1, C]]
    # smooth planes (bilinear upsampling of 6x6 noise): the photometric loss is smooth in the camera position over the
    # perturbation's range
    up = lambda: torch.nn.functional.interpolate(torch.randn(1, C, 6, 6, device=dev), size=(32, 32), mode="bilinear")
    grids = [(2.0 * up()[0].permute(1, 2, 0)).reshape(s).contiguous() for s in shapes]
    d, o, gi, nr, fr = [t.to(dev) for t in camera_rays(side, side, 1000, "cpu")]
    enc = torch.zeros(side * side, H, device=dev)

    def render(offset):
        rays = lp.Rays(directions=d, origins=o + offset, grid_idx=gi, near=nr, far=fr, encoding=enc)
        return lp.lightplane_renderer(rays, grids, dp, num_samples=S, gain=1.0, ray_image_width=side)[2]

    true_off = torch.tensor([0.03, -0.02, 0.01], device=dev)
    with torch.no_grad():
        target = render(true_off)
    off = (true_off + torch.tensor([0.08, 0.06, -0.07], device=dev)).requires_grad_(True)
    opt = torch.optim.Adam([off], lr=0.01)
    err0 = float((off - true_off).norm())
    for _ in range(40):
        opt.zero_grad()
        loss = ((render(off) - target) ** 2).mean()
        loss.backward()
        opt.step()
    err1 = float((off.detach() - true_off).norm())
    print(f"pose offset error {err0:.4f} -> {err1:.4f}")
    assert err1 < 0.3 * err0, (err0, err1)
