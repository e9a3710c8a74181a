"""Cost of the ray-geometry gradients on the headline workload: 1920x1080 camera rays, 128 samples, 64^2 x 16 triplane,
2/2/2 x 32 decoder, image MSE through `LightplaneRenderer`, `ray_image_width` tile walk.  Forward + backward timed with
CUDA events three ways, alternating within one process:
  plain    -- no geometry gradient (lp_render_backward)
  rays     -- origins and directions require grad (lp_render_backward_rays, tensor-core kernel)
  generic  -- the same with LP_ONLY_GENERIC=1 (generic fp32 kernels), on a smaller image (--generic-height rows)
Per-launch backward times come from the C-ABI's event profile.  Prints one JSON line; --out writes markdown too.

    python tools/bench_ray_grads.py --rounds 5 --out profiles/ray_grads.md
"""
import argparse
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--generic-height", type=int, default=64, help="rows of the image the generic-kernel variant renders")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import lightplane_b200 as lp
    from bench import camera_rays
    from lightplane_b200 import _cabi

    dev = torch.device("cuda")
    S, C, H, PLANE = 128, 16, 32, 64
    torch.manual_seed(0)
    model = lp.LightplaneRenderer(num_samples=S, color_chn=3, grid_chn=C, mlp_hidden_chn=H, opacity_init_bias=-1.0).to(dev)
    shapes = [[1, 1, PLANE, PLANE, C], [1, PLANE, 1, PLANE, C], [1, PLANE, PLANE, 1, C]]
    rows = sum(s[0] * s[1] * s[2] * s[3] for s in shapes)
    grid = (0.5 * torch.randn(rows, C, device=dev)).requires_grad_(True)

    def problem(h):
        rays = [t.to(dev) for t in camera_rays(args.width, h, 1000, "cpu")]
        return rays, torch.rand(rays[0].shape[0], 3, generator=torch.Generator().manual_seed(0)).to(dev)

    full, small = problem(args.height), problem(args.generic_height)

    def step(data, geo):
        (d, o, gi, nr, fr), tgt = data
        if geo:
            d, o = d.detach().requires_grad_(True), o.detach().requires_grad_(True)
        rays = lp.Rays(directions=d, origins=o, grid_idx=gi, near=nr, far=fr)
        _, _, feat = model(rays, grid, grid_sizes=shapes, ray_image_width=args.width)
        loss = ((feat - tgt) ** 2).mean()
        leaves = [grid] + list(model.parameters()) + ([o, d] if geo else [])
        return torch.autograd.grad(loss, leaves)

    variants = {"plain": (full, False, False), "rays": (full, True, False), "generic": (small, True, True)}

    def run(name, iters):
        data, geo, generic = variants[name]
        if generic:
            os.environ["LP_ONLY_GENERIC"] = "1"
        try:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            _cabi.profile_begin()
            a.record()
            for _ in range(iters):
                step(data, geo)
            b.record()
            prof = _cabi.profile_end()
        finally:
            os.environ.pop("LP_ONLY_GENERIC", None)
        bwd = [ms for nm, ms in prof if nm.startswith("lp_render_backward")]
        names = sorted({nm for nm, _ in prof if nm.startswith("lp_render_backward")})
        return a.elapsed_time(b) / iters, sum(bwd) / len(bwd), names

    for name in variants:  # warm-up of every shape
        run(name, 2)
    res = {name: {"step_ms": [], "bwd_ms": [], "entry": None} for name in variants}
    for _ in range(args.rounds):
        for name in variants:
            step_ms, bwd_ms, names = run(name, args.iters if name != "generic" else 1)
            res[name]["step_ms"].append(step_ms)
            res[name]["bwd_ms"].append(bwd_ms)
            res[name]["entry"] = names
    q = "--query-gpu=name,power.limit,clocks.max.sm"
    gpu = subprocess.run(["nvidia-smi", q, "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n_full, n_small = args.width * args.height, args.width * args.generic_height
    out = {"gpu": gpu, "rays_full": n_full, "rays_generic": n_small, "samples": S}
    for name, r in res.items():
        r["bwd_ms_median"] = sorted(r["bwd_ms"])[len(r["bwd_ms"]) // 2]
        r["step_ms_median"] = sorted(r["step_ms"])[len(r["step_ms"]) // 2]
        out[name] = r
    # the generic kernel ran on fewer rays: its backward time scaled to the full image (it is linear in the ray count)
    out["generic"]["bwd_ms_scaled_to_full"] = out["generic"]["bwd_ms_median"] * n_full / n_small
    out["rays_over_plain_bwd"] = out["rays"]["bwd_ms_median"] / out["plain"]["bwd_ms_median"]
    out["generic_over_rays_bwd"] = out["generic"]["bwd_ms_scaled_to_full"] / out["rays"]["bwd_ms_median"]
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(f"# Ray-geometry gradients: cost on the headline workload\n\nGPU: {gpu} (name, power limit, max SM clock)\n\n")
            fh.write(f"{args.width}x{args.height} rays, {S} samples, 64^2 x 16 triplane, image MSE through LightplaneRenderer, "
                     f"ray_image_width tile walk; medians of {args.rounds} alternating rounds (CUDA events).\n\n")
            fh.write("| variant | backward entry | backward launch ms | forward+backward step ms |\n|---|---|---|---|\n")
            for name in variants:
                r = out[name]
                extra = f" ({args.width}x{args.generic_height} rays; {r['bwd_ms_scaled_to_full']:.1f} ms scaled to the full image)" if name == "generic" else ""
                fh.write(f"| {name} | {', '.join(r['entry'])} | {r['bwd_ms_median']:.2f}{extra} | {r['step_ms_median']:.2f} |\n")
            fh.write(f"\nbackward with ray gradients / plain backward: {out['rays_over_plain_bwd']:.2f}x; "
                     f"generic route / tensor-core route (per ray): {out['generic_over_rays_bwd']:.1f}x\n")


if __name__ == "__main__":
    main()
