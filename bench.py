#!/usr/bin/env python
"""Headline benchmark: forward+backward rays/s of the Lightplane Renderer at 128 samples on a
64^2 x 16-channel triplane (BASELINE.json `metric`), synthetic 1920x1080 ray batches.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W  # CPU arm: the oracle port of the
                                                           # reference's naive path, on host cores

A "step" = one forward + backward pass of the public API (`LightplaneRenderer` module, MSE loss to
a random target image) over the whole ray batch; at N>1 every rank renders its own FullHD batch
(weak scaling) and the grid / MLP gradients are SUM-all-reduced over NCCL inside the step.
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for how every field is derived.

`--dump-outputs DIR` writes what the last timed step returned to its caller (rendered features, loss, and the
gradient of every trained tensor) as DIR/<name>.npy in float32.  The inputs depend only on the arguments (fixed
seeds), so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402

METRIC = "renderer_fwd_bwd_rays_per_s"
UNIT = "rays/s"
S = 128
C, H, COLOR = 16, 32, 3
PLANE = 64
# algorithmic per-sample costs (SURVEY.md 8d): MACs fwd = C*H + H*H + H*H + H + H*H + H*3
MAC_FWD = C * H + H * H + (H * H + H) + (H * H + H * COLOR)
FLOP_FWD_PER_SAMPLE = 2 * MAC_FWD            # 7 424
FLOP_BWD_PER_SAMPLE = 2 * FLOP_FWD_PER_SAMPLE  # dX + dW, recompute NOT counted: 14 848
BYTES_PER_RAY_FWD = 36 + 4 * H + 4 + 4 + 4 * COLOR            # rays+enc in, 3 outputs out
BYTES_PER_RAY_BWD = 36 + 4 * H + 4 + 4 * COLOR + 4 + 4 + 4 * COLOR + 4 * H  # + outputs, grads in, g_enc out


def load_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="MEASURED_PEAKS.json (sustained bf16)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback of B200_PROFILING.md")


def camera_rays(width, height, seed, device, fov=0.62, clip_to_volume=False):
    """Pinhole camera on a sphere of radius 2.6 looking at the origin.  Default (`fov` 0.62): the
    [-1,1]^3 volume spans most of the image height and near/far bracket the cube, so many samples lie
    in empty space (what a scene render looks like).  `clip_to_volume`: a narrower view (`fov` 0.2:
    every ray crosses the cube) with near/far = the ray's entry/exit of the cube, i.e. EVERY sample is
    inside the volume and touches all three planes (the heaviest gather / scatter load)."""
    g = torch.Generator().manual_seed(seed)
    ang = float(torch.rand(1, generator=g)) * 6.28318
    elev = 0.3 + 0.4 * float(torch.rand(1, generator=g))
    eye = 2.6 * torch.tensor([torch.cos(torch.tensor(ang)) * torch.cos(torch.tensor(elev)),
                              torch.sin(torch.tensor(elev)),
                              torch.sin(torch.tensor(ang)) * torch.cos(torch.tensor(elev))])
    fwd = -eye / eye.norm()
    up = torch.tensor([0.0, 1.0, 0.0])
    right = torch.linalg.cross(fwd, up)
    right = right / right.norm()
    up = torch.linalg.cross(right, fwd)
    aspect = width / height
    ys, xs = torch.meshgrid(torch.linspace(fov, -fov, height), torch.linspace(-fov * aspect, fov * aspect, width),
                            indexing="ij")
    dirs = fwd[None, None] + xs[..., None] * right + ys[..., None] * up
    dirs = (dirs / dirs.norm(dim=-1, keepdim=True)).reshape(-1, 3).contiguous()
    n = dirs.shape[0]
    origins = eye.expand(n, 3).contiguous()
    if clip_to_volume:
        inv = 1.0 / dirs
        t0, t1 = (-1.0 - origins) * inv, (1.0 - origins) * inv
        tn = torch.minimum(t0, t1).max(dim=1).values
        tf = torch.maximum(t0, t1).min(dim=1).values
        miss = tf <= tn
        near = torch.where(miss, torch.full_like(tn, 2.6), tn + 1e-4)
        far = torch.where(miss, torch.full_like(tf, 2.6), tf - 1e-4)
    else:
        near = torch.full((n,), 2.6 - 1.75)
        far = torch.full((n,), 2.6 + 1.75)
    grid_idx = torch.zeros(n, dtype=torch.int32)
    return dirs, origins, grid_idx, near, far


DUMP_BYTES = 64 << 20


def dump_outputs(outdir, arrays):
    """Write every array as `outdir/<name>.npy` in float32, at most DUMP_BYTES in all.  Smallest first, an array larger
    than an equal share of what is left keeps a sample of its rows (first axis) drawn with a fixed seed, so the sample
    depends only on the array's shape."""
    import numpy as np

    os.makedirs(outdir, exist_ok=True)
    budget, left = DUMP_BYTES - (1 << 20), len(arrays)  # 1 MB for the .npy headers
    for name, v in sorted(arrays.items(), key=lambda kv: kv[1].numel()):
        v = v.detach().float().cpu()
        share = budget // left
        if v.numel() * 4 > share:
            rows = max(1, share // (v[0].numel() * 4))
            v = v[torch.randperm(v.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values]
        np.save(os.path.join(outdir, name + ".npy"), v.numpy())
        budget -= v.numel() * 4
        left -= 1


def workload_stats(rays_t, width, samples, plane, tile_walk, device):
    """What the ray batch asks of the kernels (VERDICT r1 item 5): share of samples inside [-1,1]^3, planes touched
    per sample (0..3), and the share of 128-ray group-steps whose samples ALL miss every plane (folded by the
    tensor-core kernels).  Evaluated on the device, chunked over ray tiles."""
    d, o, _, near, far = [t.to(device) for t in rays_t]
    n = d.shape[0]
    tiles = n // 128
    if tile_walk and width % 16 == 0 and n % (width * 8) == 0:  # the kernels' 16x8-pixel tile walk (lp_tile_ray)
        idx = torch.arange(tiles * 128, device=device)
        tile, s = idx // 128, idx % 128
        tpr = width // 16
        w, l = s // 32, s % 32
        ray = ((tile // tpr) * 8 + (w // 2) * 4 + l // 8) * width + (tile % tpr) * 16 + (w % 2) * 8 + l % 8
    else:
        ray = torch.arange(tiles * 128, device=device)
    frac = torch.linspace(0, 1, samples, device=device)
    lim = 1.0 + 1.0 / plane  # a bilinear footprint reaches half a texel beyond the plane's edge
    inside = planes = folded = 0.0
    chunk = 2048  # tiles per chunk
    for lo in range(0, tiles, chunk):
        r = ray[lo * 128:(lo + chunk) * 128]
        t = near[r, None] + (far[r] - near[r])[:, None] * frac[None]
        p = o[r, None, :] + t[..., None] * d[r, None, :]
        a = p.abs()
        inside += float((a.max(-1).values <= 1).sum())
        hit = [(a[..., i] < lim) & (a[..., j] < lim) for i, j in ((0, 1), (0, 2), (1, 2))]
        ph = hit[0].float() + hit[1].float() + hit[2].float()
        planes += float(ph.sum())
        folded += float((ph.reshape(-1, 128, samples).sum(1) == 0).sum())
    tot = tiles * 128 * samples
    return {"samples_in_volume_frac": round(inside / tot, 4), "planes_hit_per_sample": round(planes / tot, 4),
            "folded_group_steps_frac": round(folded / (tiles * samples), 4)}


class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        busy = [v for v in sm if v > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(busy) if busy else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle (a port of the reference's naive PyTorch path) on the host cores
# ---------------------------------------------------------------------------------------------
def host_threads():
    """Threads for the CPU arm: the cores this process may run on, at most 64 (beyond that the chunked PyTorch oracle
    only thrashes: 128 threads measured 50x slower than 64 on the GPU box)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


def oracle_problem(n_rays, seed=0):
    """A small instance of the bench workload on CPU tensors (same camera model, grid, decoder init)."""
    import lightplane_b200 as lp

    torch.manual_seed(seed)
    dp = lp.init_decoder_params("cpu", 2, 2, 2, input_chn=C, hidden_chn=H, color_chn=COLOR, opacity_init_bias=-1.0)
    shapes = [[1, 1, PLANE, PLANE, C], [1, PLANE, 1, PLANE, C], [1, PLANE, PLANE, 1, C]]
    rows = sum(s[1] * s[2] * s[3] for s in shapes)
    grid = 0.5 * torch.randn(rows, C)
    side = int(n_rays ** 0.5)
    d, o, gi, nr, fr = camera_rays(side, n_rays // side, seed, "cpu")
    n = d.shape[0]
    return dict(dp=dp, shapes=shapes, grid=grid, mlp=dp.mlp_params.detach().clone(), rays=(d, o, gi, nr, fr),
                enc=torch.randn(n, H), target=torch.rand(n, COLOR), n=n, side=side)


def oracle_fwd_bwd(prob, chunk):
    """fwd+bwd of the problem through oracle/lightplane_oracle.py, chunked over rays (the naive formulation keeps
    every per-sample activation); returns (seconds, features, grad_grid, grad_mlp)."""
    from oracle import lightplane_oracle as O

    d, o, gi, nr, fr = prob["rays"]
    grid = prob["grid"].clone().requires_grad_(True)
    mlp = prob["mlp"].clone().requires_grad_(True)
    n = prob["n"]
    feats = []
    t0 = time.perf_counter()
    for lo in range(0, n, chunk):
        sl = slice(lo, min(lo + chunk, n))
        _, _, feat = O.render(d[sl], o[sl], gi[sl].long(), nr[sl], fr[sl], prob["enc"][sl], grid, prob["shapes"], mlp,
                              [C, H, H], [H, H, 1], [H, H, 16], num_samples=S, gain=1.0)
        loss = ((feat[:, :COLOR] - prob["target"][sl]) ** 2).sum() / (n * COLOR)
        loss.backward()
        feats.append(feat[:, :COLOR].detach())
    return time.perf_counter() - t0, torch.cat(feats), grid.grad, mlp.grad


def gpu_parity(prob, dev, ofeat, ogrid, omlp):
    """The CUDA path on the oracle leg's own rays: mean|d|/mean|ref| of the rendered features and of the grid / MLP
    gradients (the numbers behind `parity_err`)."""
    import lightplane_b200 as lp

    dp = prob["dp"]
    mp = prob["mlp"].to(dev).requires_grad_(True)
    dpp = lp.DecoderParams(mp, dp.n_hidden_trunk, dp.n_hidden_opacity, dp.n_hidden_color, dp.color_chn)
    rows = [s[1] * s[2] * s[3] for s in prob["shapes"]]
    parts = torch.split(prob["grid"].to(dev), rows)
    grids = [g.reshape(s).clone().requires_grad_(True) for g, s in zip(parts, prob["shapes"])]
    d, o, gi, nr, fr = [t.to(dev) for t in prob["rays"]]
    rays = lp.Rays(directions=d, origins=o, grid_idx=gi, near=nr, far=fr, encoding=prob["enc"].to(dev))
    _, _, feat = lp.lightplane_renderer(rays, grids, dpp, num_samples=S, gain=1.0, ray_image_width=prob["side"])
    ((feat - prob["target"].to(dev)) ** 2).mean().backward()
    gg = torch.cat([g.grad.reshape(-1, C) for g in grids], 0)

    def rel(a, b):
        a, b = a.detach().double().cpu(), b.detach().double().cpu()
        return float((a - b).abs().mean() / b.abs().mean())

    return {"features": rel(feat, ofeat), "g_grid": rel(gg, ogrid), "g_mlp": rel(mp.grad, omlp)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    torch.set_num_threads(threads)  # torchrun exports OMP_NUM_THREADS=1: pin the arm to the box's cores explicitly
    n_rays, chunk = 8192, 2048
    for _ in range(args.warmup):
        oracle_fwd_bwd(oracle_problem(2048), 2048)
    t = 0.0
    n = 0
    for k in range(args.steps):
        prob = oracle_problem(n_rays, seed=k)
        dt = oracle_fwd_bwd(prob, chunk)[0]
        t += dt
        n += prob["n"]
    value = n / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"renderer fwd+bwd, {S} samples, triplane {PLANE}^2x{C}ch, MLP 2/2/2 h{H}",
                   "note": "reference is a Python package (no compiled CPU path): this arm is the oracle "
                           "port of its naive PyTorch renderer, chunked over rays, on the host cores "
                           f"(torch.set_num_threads({threads}))"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n_rays} rays x {S} samples per step, chunks of {chunk}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-in-volume", action="store_true", help="skip the second timed workload (all samples inside the volume)")
    ap.add_argument("--no-tile-walk", dest="tile_walk", action="store_false",
                    help="do not pass the image width (ray_image_width): the kernels then walk 128-ray scan-line runs instead "
                         "of 16x8-pixel tiles (measured: profiles/bench_r2_ablation.md)")
    ap.add_argument("--per-rank-cameras", action="store_true",
                    help="N>1: a different camera per rank (default: the same view on every rank, so that the scaling "
                         "number measures the machine and not the spread of per-view work)")
    ap.add_argument("--workload", default="headline", choices=["headline", "cfg5"],
                    help="cfg5 = BASELINE.json configs[4]: 256 samples, 128^2 x 32 triplane, Renderer + Splatter per step")
    # non-default shapes
    ap.add_argument("--samples", type=int, default=None)
    ap.add_argument("--plane", type=int, default=None)
    ap.add_argument("--grid-chn", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's features, loss and gradients as DIR/<name>.npy (float32, at most "
                         "64 MB: larger outputs keep a fixed seeded sample of their rows)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repository's CUDA path (--impl ours)")
    cfg5 = args.workload == "cfg5"
    globals().update(S=args.samples or (256 if cfg5 else S), PLANE=args.plane or (128 if cfg5 else PLANE),
                     C=args.grid_chn or (32 if cfg5 else C))
    globals().update(MAC_FWD=C * H + H * H + (H * H + H) + (H * H + H * COLOR))
    globals().update(FLOP_FWD_PER_SAMPLE=2 * MAC_FWD, FLOP_BWD_PER_SAMPLE=4 * MAC_FWD)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist

    import lightplane_b200 as lp
    from lightplane_b200 import _cabi
    from lightplane_b200.distributed import all_reduce_gradients

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD if world > 1 else None

    # ---- model (replicated) + data (per rank) ----
    torch.manual_seed(0)
    model = lp.LightplaneRenderer(num_samples=S, color_chn=COLOR, grid_chn=C, mlp_hidden_chn=H,
                                  opacity_init_bias=-1.0).to(dev)
    shapes = [[1, 1, PLANE, PLANE, C], [1, PLANE, 1, PLANE, C], [1, PLANE, PLANE, 1, C]]
    # the three planes live in ONE flat [rows, C] parameter + a host size table (the reference API's flat form,
    # misc_utils.py:201-234): no per-call concatenation, one tensor to all-reduce
    grid_rows = sum(s[0] * s[1] * s[2] * s[3] for s in shapes)
    grids = [(0.5 * torch.randn(grid_rows, C, device=dev)).requires_grad_(True)]
    params = grids + list(model.parameters())
    cam_seed = 1000 + (rank if args.per_rank_cameras else 0)
    hint = args.width if args.tile_walk else None

    def make_data(**cam_kw):
        host = [t.pin_memory() for t in camera_rays(args.width, args.height, cam_seed, "cpu", **cam_kw)]
        return host, [t.to(dev) for t in host]

    host, resident = make_data()
    n_rays = host[0].shape[0]
    target_host = torch.rand(n_rays, COLOR, generator=torch.Generator().manual_seed(rank)).pin_memory()
    target = target_host.to(dev)
    h2d_bytes = sum(t.numel() * t.element_size() for t in host) + target_host.numel() * 4
    out_host = torch.empty(n_rays, COLOR).pin_memory()
    loss_host = torch.empty(1).pin_memory()
    d2h_bytes = out_host.numel() * 4 + 4
    splat_feat = torch.rand(n_rays, C, device=dev, requires_grad=True) if cfg5 else None
    comm_events = []

    def step(rays_t, tgt):
        for p in params:
            p.grad = None
        rays = lp.Rays(directions=rays_t[0], origins=rays_t[1], grid_idx=rays_t[2], near=rays_t[3], far=rays_t[4])
        _, _, feat = model(rays, grids[0], grid_sizes=shapes, ray_image_width=hint)
        loss = ((feat - tgt) ** 2).mean()
        if cfg5:  # configs[4]: the Splatter runs on the same sharded rays; its accumulators are all-reduced inside the op
            srays = lp.Rays(directions=rays_t[0], origins=rays_t[1], grid_idx=rays_t[2], near=rays_t[3], far=rays_t[4],
                            encoding=splat_feat)
            sp = lp.lightplane_splatter(srays, [tuple(s) for s in shapes], num_samples=S, return_list=False,
                                        process_group=group)
            loss = loss + (sp ** 2).mean()
            splat_feat.grad = None
        loss.backward()
        if world > 1:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            all_reduce_gradients(params)
            b.record()
            comm_events.append((a, b))
        return feat, loss

    # End-to-end step = what a training loop with a prefetching input pipeline does: the pinned host batch of step i+1 is
    # copied on a side stream while step i's kernels run, the step's result is read back on a second side stream.  Every
    # step's input bytes and result bytes move inside the timed region (K steps issue K+1 input copies).
    h2d_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    pipe = {"next": None}

    def prefetch():
        with torch.cuda.stream(h2d_stream):
            bufs = [t.to(dev, non_blocking=True) for t in host] + [target_host.to(dev, non_blocking=True)]
            ev = torch.cuda.Event()
            ev.record(h2d_stream)
        return bufs, ev

    def e2e_step():
        cur = torch.cuda.current_stream(dev)
        if pipe["next"] is None:
            pipe["next"] = prefetch()
        bufs, ev = pipe["next"]
        cur.wait_event(ev)
        for t in bufs:
            t.record_stream(cur)
        pipe["next"] = prefetch()
        feat, loss = step(bufs[:-1], bufs[-1])
        done = torch.cuda.Event()
        done.record(cur)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(done)
            feat.record_stream(d2h_stream)
            loss.record_stream(d2h_stream)
            out_host.copy_(feat.detach(), non_blocking=True)
            loss_host.copy_(loss.detach().reshape(1), non_blocking=True)

    def e2e_finish():  # the timed region ends only when the last result has reached the host
        cur = torch.cuda.current_stream(dev)
        cur.wait_stream(d2h_stream)
        cur.wait_stream(h2d_stream)
        pipe["next"] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(args.warmup):
        step(resident, target)
        e2e_step()
    e2e_finish()

    last = {}

    def timed_step():
        feat, loss = step(resident, target)
        last["features"], last["loss"] = feat.detach(), loss.detach()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    comm_events.clear()
    _cabi.profile_begin()
    try:
        ms = timed(timed_step, args.steps)
        launches = _cabi.profile_end()
    finally:  # nvidia-smi must not outlive a failed step
        clocks = sampler.stop() if sampler else None
    # taken before the later timed regions, which run the step again and overwrite the gradients
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = {"features": last["features"], "loss": last["loss"], "grad_grid": grids[0].grad}
        outputs.update({"grad_" + k.replace(".", "_"): p.grad for k, p in model.named_parameters()})
        if cfg5:
            outputs["grad_splat_features"] = splat_feat.grad
        outputs = {k: v.cpu() for k, v in outputs.items()}
    comm_ms = sum(a.elapsed_time(b) for a, b in comm_events) / max(len(comm_events), 1) if comm_events else 0.0
    ms_e2e = timed(e2e_step, args.steps, e2e_finish)

    value = world * n_rays * args.steps / (ms * 1e-3)
    e2e_value = world * n_rays * args.steps / (ms_e2e * 1e-3)

    per = {}
    for name, t in launches:
        per.setdefault(name, []).append(t)
    avg = {k: sum(v) / len(v) for k, v in per.items()}
    bwd_ms = avg.get("lp_render_backward", float("nan"))
    fwd_ms = avg.get("lp_render_forward", float("nan"))

    # ---- second timed workload: every sample inside the volume (3 planes per sample, nothing to fold) ----
    in_volume = None
    if not args.skip_in_volume and not cfg5:
        host_v, resident_v = make_data(fov=0.2, clip_to_volume=True)
        for _ in range(2):
            step(resident_v, target)
        _cabi.profile_begin()
        ms_v = timed(lambda: step(resident_v, target), args.steps)
        lv = {}
        for name, t in _cabi.profile_end():
            lv.setdefault(name, []).append(t)
        in_volume = {"value": world * n_rays * args.steps / (ms_v * 1e-3), "unit": UNIT, "ms_per_step": ms_v / args.steps,
                     "launch_ms": {k: sum(v) / len(v) for k, v in lv.items() if k.startswith("lp_render")},
                     "camera": "fov 0.2, near/far = ray-cube intersection"}
        if rank == 0:
            in_volume.update(workload_stats(host_v, args.width, S, PLANE, args.tile_walk, dev))

    # ---- N>1: per-rank kernel times and the share of the step spent in the collective ----
    comm = None
    if world > 1:
        mine = torch.tensor([fwd_ms, bwd_ms, comm_ms, ms / args.steps], device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        allr = torch.stack(allr).cpu()
        comm = {"what": "SUM all-reduce of grid + MLP gradients (one NCCL bucket) inside the step; ms = event pair around it "
                        "(includes waiting for the slowest rank)",
                "bytes_per_step": int(sum(p.numel() for p in params) * 4),
                "per_rank_ms": {"forward": [round(float(v), 3) for v in allr[:, 0]], "backward": [round(float(v), 3) for v in allr[:, 1]],
                                "all_reduce": [round(float(v), 3) for v in allr[:, 2]], "step": [round(float(v), 3) for v in allr[:, 3]]},
                "cameras": "one per rank" if args.per_rank_cameras else "same view on every rank"}

    if rank == 0:
        peaks = load_peaks()
        samples = n_rays * S
        ach_tflops = samples * FLOP_BWD_PER_SAMPLE / (bwd_ms * 1e-3) / 1e12
        traffic = None
        tp = os.path.join(REPO, "profiles", "traffic.json")
        if os.path.exists(tp) and not cfg5:
            traffic = json.load(open(tp)).get("lp_render_backward_dram_bytes_per_launch")
        roofline = {
            "kernel": "lp_render_backward", "bound": "tensor", "achieved": ach_tflops, "peak": peaks["tflops"],
            "unit": "TFLOP/s", "frac": ach_tflops / peaks["tflops"], "traffic": traffic,
            "peak_source": peaks["source"],
            "algorithmic_flops_per_launch": samples * FLOP_BWD_PER_SAMPLE,
            "launch_ms": {k: v for k, v in avg.items()},
            "kernel_share_of_step": sum(avg.values()) * args.steps / ms,
            "hbm": {"algorithmic_bytes_per_launch": n_rays * BYTES_PER_RAY_BWD,
                    "achieved_gbs": n_rays * BYTES_PER_RAY_BWD / (bwd_ms * 1e-3) / 1e9,
                    "peak_gbs": peaks["hbm_gbs"],
                    "frac": n_rays * BYTES_PER_RAY_BWD / (bwd_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]},
            "forward": {"achieved_tflops": samples * FLOP_FWD_PER_SAMPLE / (fwd_ms * 1e-3) / 1e12,
                        "frac": samples * FLOP_FWD_PER_SAMPLE / (fwd_ms * 1e-3) / 1e12 / peaks["tflops"]},
        }
        cpu = None
        if world == 1 and not args.skip_cpu_baseline and not cfg5:
            torch.set_num_threads(host_threads())
            oracle_fwd_bwd(oracle_problem(4096), 2048)  # warm-up
            prob = oracle_problem(16384, seed=1)
            dt, ofeat, ogrid, omlp = oracle_fwd_bwd(prob, 2048)
            cpu = {"value": prob["n"] / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                   "sample": "16384 rays x %d samples of the same workload, chunks of 2048 rays, 1 warm-up" % S,
                   "parity_err": gpu_parity(prob, dev, ofeat, ogrid, omlp),
                   "parity_note": "mean|d|/mean|ref| of this repo's CUDA path vs the oracle on the sample's rays (fp32 oracle)"}
        stats = workload_stats(host, args.width, S, PLANE, args.tile_walk, dev)
        what = "fwd+bwd of LightplaneRenderer + MSE" + (" + LightplaneSplatter fwd+bwd into the same triplane shape" if cfg5 else "")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": f"{args.width}x{args.height} rays/GPU, {S} samples, triplane 3x[{PLANE}x{PLANE}]x{C}ch, "
                            f"MLP trunk/opacity/colour 2/2/2 hidden {H}, colour {COLOR}; {what}",
                "rays_per_gpu": n_rays, "num_samples": S,
                "camera": "pinhole at radius 2.6, fov 0.62, near/far 0.85/4.35 bracket the cube (scene-render view)",
                **stats,
                "ray_order": "row-major image, walked in 16x8-pixel tiles (ray_image_width hint)" if args.tile_walk else "row-major image, 128-ray scan-line runs",
                "l2_policy": "inputs larger than L2: per-step ray/encoding/gradient tensors ~%d MB" % (n_rays * (BYTES_PER_RAY_BWD) // 1e6),
                "parallelism": f"rays sharded x{world}, grid+MLP replicated, grad all-reduce (NCCL)" if world > 1 else "single GPU",
            },
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "pipeline": "pinned-host inputs of step i+1 copied on a side stream during step i, result of step i read back "
                                "on a second side stream; the region ends when the last result is on the host"},
            "gpu_launches": len(launches),
            "clocks": clocks,
            "roofline": roofline,
        }
        if in_volume is not None:
            line["value_in_volume"] = in_volume["value"]
            line["in_volume"] = in_volume
        if comm is not None:
            line["comm"] = comm
        if cpu is not None:
            line["cpu_baseline"] = cpu
        gc = os.path.join(REPO, "profiles", "gpu_comparator_r2.json")
        if os.path.exists(gc) and not cfg5:  # the reference's own Triton kernels on the same B200 (tools/gpu_comparator.py)
            try:
                rows = json.load(open(gc)).get("timing", [])
                line["gpu_comparator"] = {r["workload"].split(" rays")[0]: r.get("reference_triton", {}).get("rays_per_s") for r in rows}
            except Exception:
                pass
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
