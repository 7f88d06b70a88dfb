#!/usr/bin/env python
"""
bench.py -- rays/sec of the pixelNeRF render hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4] [--scaling weak|strong]
                  [--impl ours|reference|reference-gpu|torch-eager] [--dump-outputs DIR]
  torchrun --nproc-per-node N ... bench.py --gpus N ...   (one rank per GPU, NCCL)

A "step" renders one batch of synthetic rays (coarse + fine pass) of a BASELINE.json workload:
  c2 (default, the headline)  SRN-car 128x128, 2 source views, 64+32 samples   16 384 rays = one frame
  c3                          ShapeNet-NMR 64x64, 1 source view, 64+16 samples   4 096 rays = one frame
  c4                          DTU 400x300, 3 source views, 96+48 samples       120 000 rays = one frame
all with ResnetFC d=512 x 5 blocks, random-init weights with re-randomised fc_1 (synth.bench_mlp_weights: lin_z scaled
so the random network renders a non-blank, semi-transparent volume), and a real resnet34 trunk for the latent.  `value` = rays/s of the whole job with inputs resident in HBM; `e2e` = the same through the public API
(`NeRFRenderer.bind_parallel(net)(rays)`) from pinned HOST rays to HOST pixels.

Ranks shard rays (render/sharding.py, torch.chunk order): `--scaling weak` (default) gives every GPU one frame,
`--scaling strong` splits ONE frame over the N GPUs (BASELINE configs C3 / C4: "8xB200 ray-sharded").  The scene is
broadcast from rank 0 once (NCCL) and rendered pixels are gathered to rank 0 every step inside the timed region.

The line also carries a `parity` block: the benchmarked model + frame, 256 rays with injected noise, CUDA vs the CPU
oracle (outside the timed region).

`--dump-outputs DIR` writes the rgb / depth of the last timed step, so that two builds run with the same arguments
(hence the same seeded scene, rays and sample noise) can be compared output for output.  Nothing is written into the
source tree: no bytecode either, so the tree may be read-only.

`--impl reference` times the UNMODIFIED reference (oracle/_ref, installed by build(); falls back to the
oracle port when absent) on the HOST CPU cores through its own public API, on a bounded sample of the same workload;
`--impl reference-gpu` runs the same unmodified reference eagerly on the B200(s) (fp32, TF32 off; DataParallel at N>1) --
the denominator of north_star's ">= 10x the reference's own 1xGPU PyTorch rays/sec".
"""
import argparse
import importlib.util
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pixel-nerf_b200")
SRC = os.path.join(PKG, "src")


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


synth = _load("pnr_synth", os.path.join(PKG, "synth.py"))

WORKLOADS = {
    "c2": dict(metric="rays/sec (64c+32f samples, 2 src views)", frame_rays=128 * 128, cpu_rays=1024,
               text="C2 SRN-car 128x128, 2 src views, 64 coarse + 32 fine (16 depth) samples, ResnetFC d=512 x5 blocks, "
                    "resnet34 latent 2x512x64x64"),
    "c3": dict(metric="rays/sec (64c+16f samples, 1 src view)", frame_rays=64 * 64, cpu_rays=1024,
               text="C3 ShapeNet-NMR 64x64, 1 src view, 64 coarse + 16 fine (8 depth) samples, ResnetFC d=512 x5 blocks, "
                    "resnet34 (no first pool) latent 1x512x32x32"),
    "c4": dict(metric="rays/sec (96c+48f samples, 3 src views)", frame_rays=400 * 300, cpu_rays=512,
               text="C4 DTU 400x300, 3 src views, 96 coarse + 48 fine (16 depth) samples, ResnetFC d=512 x5 blocks, "
                    "resnet34 latent 3x512x150x200"),
}


def profile_file(workload):
    for name in (f"r2_k_field_tc_{workload}.txt", "r2_k_field_tc.txt", "r1_final_k_field_tc.txt"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p) and (workload == "c2" or name.startswith(f"r2_k_field_tc_{workload}")):
            return p
    return None


def profiled_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu capture of this command; None if absent."""
    p = profile_file(workload)
    if p is None:
        return None, None
    n, tot = 0, 0.0
    for line in open(p):
        if "dram__bytes_read.sum [" in line or "dram__bytes_write.sum [" in line:
            unit = line.split("[")[1].split("]")[0]
            val = float(line.split("=")[1])
            tot += val * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
            n += 1
    return (tot / (n / 2) if n else None), os.path.relpath(p, ROOT)


def profiled_tensor_active(workload):
    p = profile_file(workload)
    if p is None:
        return None
    vals = [float(l.split("=")[1]) for l in open(p)
            if "sm__pipe_tensor_cycles_active_realtime.avg.pct_of_peak_sustained_elapsed" in l]
    return sum(vals) / len(vals) if vals else None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md sustained)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.samples = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,power.limit")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
               "samples": len(sm)}
        try:    # board power next to the clocks: the kernel runs against the power limit, not the clock limit
            pw = sorted(float(s[6]) for s in self.samples if len(s) >= 8)
            if pw:
                out["power_w"] = pw[len(pw) // 2]
                out["power_limit_w"] = float(self.samples[0][7])
        except ValueError:
            pass
        return out


def model_conf(cfg):
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    from util import hocon
    conf = hocon.parse_file(os.path.join(PKG, "conf", "exp", "srn.conf"))
    conf.put("model.encoder.pretrained", False)          # no network: random-init trunk
    conf.put("model.encoder.use_first_pool", cfg["use_first_pool"])
    conf.put("model.mlp_coarse.d_hidden", cfg["d_hidden"])
    conf.put("model.mlp_fine.d_hidden", cfg["d_hidden"])
    conf.put("renderer.n_coarse", cfg["n_coarse"])
    conf.put("renderer.n_fine", cfg["n_fine"])
    conf.put("renderer.n_fine_depth", cfg["n_fine_depth"])
    conf.put("renderer.white_bkgd", cfg["white_bkgd"])
    return conf


def build_scene(cfg, device, engine):
    """net (encoded, on device) + renderer through the public classes."""
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    from model import make_model
    from render import NeRFRenderer
    conf = model_conf(cfg)
    torch.manual_seed(0)
    net = make_model(conf["model"])
    net.mlp_coarse.load_state_dict(synth.bench_mlp_weights(11, cfg["d_hidden"]))
    net.mlp_fine.load_state_dict(synth.bench_mlp_weights(12, cfg["d_hidden"]))
    net = net.to(device).eval()
    net.engine = engine
    renderer = NeRFRenderer.from_conf(conf["renderer"], eval_batch_size=50000).to(device).eval()
    src, _, focal, c = synth.make_cameras(cfg)
    images = synth.make_images(cfg, seed=0)
    with torch.no_grad():
        net.encode(images[None].to(device), src[None].to(device), focal.to(device), c=c[None].to(device))
    return net, renderer


def scene_tensors(net):
    """Everything the render path reads (latent + cameras + weights): the ONE broadcast per scene that replaces
    DataParallel's per-call module replication (reference src/render/nerf.py:370)."""
    return [net.encoder.latent, net.poses, net.focal, net.c, *[p.data for p in net.mlp_coarse.parameters()],
            *[p.data for p in net.mlp_fine.parameters()]]


def parity_block(net, renderer, cfg, rays_dev, n=256):
    """CUDA (the benchmarked model, engine and frame) vs the CPU oracle on n rays spread over the frame, same injected
    noise; outside the timed region.  flipped = rays whose merged fine samples differ (a 1-ulp searchsorted bin flip
    moves an importance sample by a bin, SURVEY 7.3)."""
    oracle = _load("pnr_oracle", os.path.join(ROOT, "oracle", "pnr_oracle.py"))
    R = rays_dev.shape[1]
    idx = torch.linspace(0, R - 1, min(n, R)).long()
    sub = rays_dev[:, idx.to(rays_dev.device)].contiguous()
    nr = sub.shape[1]
    noise = synth.draw_noise(7, nr, cfg["n_coarse"], cfg["n_fine"], cfg["n_fine_depth"])
    with torch.no_grad():
        out = renderer._forward_fused(net, sub, want_weights=False,
                                      noise_in={k: v.to(sub.device) for k, v in noise.items()}, want_z=True)
    src, _, focal, c = synth.make_cameras(cfg)
    state = oracle.encode_state(src, focal, c[None], cfg["W"], cfg["H"])
    sd = lambda m: {k: v.detach().float().cpu() for k, v in m.state_dict().items()}
    t0 = time.perf_counter()
    with torch.no_grad():
        ref = oracle.render(sub.cpu(), noise, state, net.encoder.latent.detach().float().cpu(), sd(net.mlp_coarse),
                            sd(net.mlp_fine), cfg["NS"], cfg["n_coarse"], cfg["n_fine"], cfg["n_fine_depth"],
                            white_bkgd=cfg["white_bkgd"], eval_batch_size=50000)
    t_oracle = time.perf_counter() - t0
    best = "fine" if cfg["n_fine"] > 0 else "coarse"
    rgb = out[best].rgb.reshape(-1, 3).cpu()
    d = (rgb - ref[best]["rgb"]).abs().max(-1).values
    dz = (out[best].z.reshape(nr, -1).cpu() - ref[best]["z"]).abs().max(-1).values
    flipped = dz > 1e-4 * (cfg["z_far"] - cfg["z_near"])
    keep = ~flipped
    mse = ((rgb - ref[best]["rgb"]) ** 2).mean().item()
    dc = (out.coarse.rgb.reshape(-1, 3).cpu() - ref["coarse"]["rgb"]).abs().max().item()
    ddep = (out[best].depth.reshape(-1).cpu() - ref[best]["depth"])[keep].abs().max().item() if keep.any() else None
    q = lambda t, p: float(torch.quantile(t, p)) if t.numel() else None
    return {"vs": "oracle/pnr_oracle.py (CPU fp32 restatement pinned on reference-generated goldens)", "rays": nr,
            "psnr_db": (-10 * math.log10(mse)) if mse > 0 else float("inf"),
            "max_abs_drgb_coarse": dc, "max_abs_drgb": float(d[keep].max()) if keep.any() else None,
            "p999_abs_drgb": q(d[keep], 0.999), "max_abs_drgb_incl_flipped": float(d.max()),
            "max_abs_ddepth": ddep, "flipped_rays": int(flipped.sum()), "tolerance": 1e-4,
            "oracle_seconds": t_oracle}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """arrays: name -> (1, rays, ...) tensor, written as out_dir/<name>.npy in float32.  Above DUMP_LIMIT_BYTES in all,
    a fixed, seeded sample of rays (the same rays for every array, in ray order) is written instead."""
    import numpy as np
    n = next(iter(arrays.values())).shape[1]
    per_ray = sum(t[0, :1].numel() * 4 for t in arrays.values())
    keep = None
    if n * per_ray > DUMP_LIMIT_BYTES:
        keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_LIMIT_BYTES // per_ray].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t if keep is None else t[:, keep]).numpy())


def run_ours(args):
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    import pnr_native as pn
    from render import sharding
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the render path has no CPU fallback)")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    wl = WORKLOADS[args.workload]
    cfg = synth.CONFIGS[args.workload]
    net, renderer = build_scene(cfg, device, args.engine)
    if dist is not None:
        with torch.no_grad():
            sharding.broadcast_state(scene_tensors(net), dist, src=0)
            net.encoder.latent.add_(0)  # bump version -> derived state (channels-last copy, P maps) is rebuilt
    render_par = renderer.bind_parallel(net, [local], simple_output=True).eval()

    frame = args.rays if args.rays else wl["frame_rays"]
    strong = args.scaling == "strong"
    total = frame if strong else frame * world           # rays of the whole job per step
    n_target = max(8, total // (cfg["W"] * cfg["H"]) + 1)
    all_rays = synth.make_rays(cfg, total, n_target=n_target)[None]          # (1, total, 8)
    my_rays_host = sharding.local_shard(all_rays, rank, world, dim=1)[0].contiguous().pin_memory()
    n_mine = my_rays_host.shape[0]
    rays_dev = my_rays_host.to(device)[None]                      # (1, n_mine, 8) resident
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)  # > 126 MB L2

    def gather(rgb, depth):
        if dist is None:
            return rgb, depth
        return (sharding.gather_rays(rgb, total, dist, rank, world, dst=0, dim=1),
                sharding.gather_rays(depth, total, dist, rank, world, dst=0, dim=1))

    def step_resident():
        flush.zero_()
        with torch.no_grad():
            rgb, depth = render_par(rays_dev)
        return gather(rgb, depth)

    host_rgb = torch.empty(1, total if rank == 0 else 1, 3).pin_memory()
    host_dep = torch.empty(1, total if rank == 0 else 1).pin_memory()

    def step_e2e():
        flush.zero_()
        with torch.no_grad():
            r = my_rays_host.to(device, non_blocking=True)[None]
            rgb, depth = render_par(r)
        rgb, depth = gather(rgb, depth)
        if rank == 0:
            host_rgb.copy_(rgb, non_blocking=True)
            host_dep.copy_(depth, non_blocking=True)

    def timed(fn, steps):
        """(device ms of `steps` calls of fn, what the last call returned)"""
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if dist is not None:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_resident()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = pn.launch_count()
    pn.profile_begin()
    ms_total, (last_rgb, last_depth) = timed(step_resident, args.steps)
    kern_ms, kern_launches = pn.profile_end()
    if os.environ.get("PNR_TC_COUNTERS"):
        names = ["mma_total", "mma_wait_a_first_chunk", "mma_wait_b", "mma_wait_bpeer", "unused4", "unused5",
                 "mma_wait_a_later_chunks", "stream_wait_empty"]
        print("tc_counters", dict(zip(names, pn.tc_counters())), file=sys.stderr)
    launches = pn.launch_count() - launches0
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    sampler.stop_flag = True
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rgb": last_rgb, "depth": last_depth})

    value = total * args.steps / (ms_total / 1e3)
    e2e_value = total * args.steps / (ms_e2e / 1e3)
    fl = synth.flops_per_ray(cfg["n_coarse"], cfg["n_fine"], cfg["NS"], cfg["d_hidden"])
    peak, peak_src = peaks()
    rays_rank = n_mine * args.steps
    kern_tflops = (rays_rank * fl / 1e12) / (kern_ms / 1e3) if kern_ms > 0 else None

    # fp16 tensor work the tensor engine actually issues: 3 split products over lin_in (K padded to 48) and the
    # 10 fc layers; the three lin_z GEMMs are folded into the per-scene projected-latent maps (DESIGN.md 3.1)
    d = cfg["d_hidden"]
    pts = cfg["n_coarse"] + ((cfg["n_coarse"] + cfg["n_fine"]) if cfg["n_fine"] > 0 else 0)
    exec_fl = 2 * 3 * pts * (cfg["NS"] * (48 * d + 6 * d * d) + 4 * d * d)
    exec_tflops = (rays_rank * exec_fl / 1e12) / (kern_ms / 1e3) if kern_ms > 0 else None
    tensor_engine = net._fused.mlp.get("mlp_coarse", (0, 0, 0, None))[3] is not None

    parity = None
    cpu_base = None
    if rank == 0 and not args.no_parity:
        try:
            parity = parity_block(net, renderer, cfg, rays_dev)
        except Exception as e:     # the throughput line must still be printed
            parity = {"error": repr(e)[:300]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline_subprocess(args.workload, args.cpu_rays or wl["cpu_rays"])

    if rank == 0:
        traffic, traffic_src = profiled_traffic(args.workload)
        line = {
            "metric": wl["metric"], "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32 (fp16 hi/lo split products, fp32 accumulate)" if tensor_engine else "f32",
            "data": "synthetic",
            "config": {"workload": wl["text"], "rays_per_step": total, "rays_per_step_per_gpu": n_mine,
                       "engine": args.engine, "l2_flush_between_steps": True,
                       "weights": f"synthetic kaiming (synth.bench_mlp_weights, lin_z x{synth.BENCH_LATENT_GAIN}), "
                                  "random-init resnet34 trunk",
                       "parallelism": f"ray-sharded x{world} ({args.scaling})", "flop_per_ray": fl},
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": total * 8 * 4,
                    "d2h_bytes_per_step": total * 4 * 4},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": kern_tflops, "peak": peak, "unit": "TFLOP/s",
                         "frac": (kern_tflops / peak) if kern_tflops else None, "traffic": traffic,
                         "peak_source": peak_src, "kernel_launches": int(kern_launches),
                         "ncu_tensor_pipe_active_pct": profiled_tensor_active(args.workload),
                         "traffic_note": f"dram bytes per launch from {traffic_src} (same command under ncu); see "
                                         "DESIGN.md section 7 for what they consist of",
                         "kernel_ms_per_step": kern_ms / args.steps,
                         "executed_fp16_mma_tflops": exec_tflops if tensor_engine else None,
                         "executed_frac_of_peak": (exec_tflops / peak) if (tensor_engine and exec_tflops) else None,
                         "note": "algorithmic fp32-model FLOPs of the reference (SURVEY 8d) / device time of the "
                                 "MLP-contraction kernel(s), CUDA events on the launch stream"},
            "clocks": sampler.summary(),
        }
        if parity is not None:
            line["parity"] = parity
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
# reference arms: the UNMODIFIED reference through its own public API (oracle/_ref)
# ------------------------------------------------------------------------------------------
def reference_root():
    for root in (os.environ.get("PIXELNERF_REF"), os.path.join(ROOT, "oracle", "_ref")):
        if root and os.path.isdir(os.path.join(root, "src", "render")):
            return root
    return None


def build_reference_scene(workload, device):
    """The reference's PixelNeRFNet + NeRFRenderer + bind_parallel, weights and scene of the workload; returns
    (net, renderer) or None when oracle/_ref is absent."""
    root = reference_root()
    if root is None:
        return None
    os.environ["PIXELNERF_REF"] = root
    rh = _load("pnr_ref_harness", os.path.join(ROOT, "oracle", "ref_harness.py"))
    cfg = synth.CONFIGS[workload]
    torch.manual_seed(0)
    net, renderer = rh.build_reference(cfg["d_hidden"], synth.bench_mlp_weights(11, cfg["d_hidden"]),
                                       synth.bench_mlp_weights(12, cfg["d_hidden"]), cfg["n_coarse"], cfg["n_fine"],
                                       cfg["n_fine_depth"], white_bkgd=cfg["white_bkgd"], eval_batch_size=50000,
                                       use_first_pool=cfg["use_first_pool"])
    net = net.to(device).eval()
    renderer = renderer.to(device).eval()
    src, _, focal, c = synth.make_cameras(cfg)
    images = synth.make_images(cfg, seed=0)
    with torch.no_grad():
        net.encode(images[None].to(device), src[None].to(device), focal.to(device), c=c[None].to(device))
    return net, renderer


def cpu_threads_probe(render_once, candidates):
    """Thread count for the CPU arm: time a small render at each candidate, keep the fastest."""
    best, best_t, table = None, None, {}
    for t in candidates:
        torch.set_num_threads(t)
        render_once()
        t0 = time.perf_counter()
        render_once()
        dt = time.perf_counter() - t0
        table[t] = dt
        if best_t is None or dt < best_t:
            best, best_t = t, dt
    torch.set_num_threads(best)
    return best, table


_cpu_arm_cache = {}


def cpu_arm(workload):
    """(render(rays (1,n,8)) callable, kind, description, threads, probe) for the host-CPU arm."""
    if workload in _cpu_arm_cache:
        return _cpu_arm_cache[workload]
    cfg = synth.CONFIGS[workload]
    ref = build_reference_scene(workload, torch.device("cpu"))
    if ref is not None:
        net, renderer = ref
        render_par = renderer.bind_parallel(net, None, simple_output=True).eval()

        def render(rays):
            with torch.no_grad():
                return render_par(rays)
        kind, what = "reference", "unmodified reference (oracle/_ref) NeRFRenderer.bind_parallel(net)(rays), torch CPU fp32"
    else:
        oracle = _load("pnr_oracle", os.path.join(ROOT, "oracle", "pnr_oracle.py"))
        src, _, focal, c = synth.make_cameras(cfg)
        latent = synth.make_latent(5, cfg["NS"], cfg["H"] // 2, cfg["W"] // 2)
        state = oracle.encode_state(src, focal, c[None], cfg["W"], cfg["H"])
        wc, wf = synth.bench_mlp_weights(11, cfg["d_hidden"]), synth.bench_mlp_weights(12, cfg["d_hidden"])

        def render(rays):
            noise = synth.draw_noise(3, rays.shape[1], cfg["n_coarse"], cfg["n_fine"], cfg["n_fine_depth"])
            with torch.no_grad():
                return oracle.render(rays, noise, state, latent, wc, wf, cfg["NS"], cfg["n_coarse"], cfg["n_fine"],
                                     cfg["n_fine_depth"], white_bkgd=cfg["white_bkgd"], eval_batch_size=50000)
        kind, what = "port", "oracle/pnr_oracle.py (oracle/_ref absent), torch CPU fp32"
    ncpu = os.cpu_count() or 1
    cands = sorted({t for t in (8, 16, 32, 64, 128, ncpu) if t <= ncpu})
    probe_rays = synth.make_rays(cfg, 64)[None]
    threads, table = cpu_threads_probe(lambda: render(probe_rays), cands)
    _cpu_arm_cache[workload] = (render, kind, what, threads, {str(k): round(v, 4) for k, v in table.items()})
    return _cpu_arm_cache[workload]


def cpu_reference_run(workload, sample_rays, warm_rays=0):
    """One timed pass of the reference's CPU path over `sample_rays` rays of the workload."""
    cfg = synth.CONFIGS[workload]
    render, kind, what, threads, probe = cpu_arm(workload)
    if warm_rays:
        render(synth.make_rays(cfg, warm_rays)[None])
    rays = synth.make_rays(cfg, sample_rays)[None]
    t0 = time.perf_counter()
    render(rays)
    dt = time.perf_counter() - t0
    return {"value": sample_rays / dt, "unit": "rays/s", "cores": threads, "kind": kind,
            "sample": f"{sample_rays} rays of the same {workload.upper()} workload per pass; {what}",
            "host_cpus": os.cpu_count(), "thread_probe_seconds_64_rays": probe}


def cpu_baseline_subprocess(workload, sample_rays):
    """`cpu_baseline` of the default run: one bounded pass of `--impl reference` in a child process (the reference's
    packages are called `model` / `render` / `util` like this repo's, so the two cannot share an interpreter)."""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--steps", "1",
           "--warmup", "1", "--cpu-rays", str(sample_rays)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        for line in reversed(out.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)["cpu_baseline"]
        return {"error": (out.stderr or out.stdout)[-300:]}
    except Exception as e:   # the bench line must still be printed
        return {"error": repr(e)[:300]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    n = args.cpu_rays or wl["cpu_rays"]
    for _ in range(max(args.warmup, 0)):
        cpu_reference_run(args.workload, max(64, n // 8))
    stats = [cpu_reference_run(args.workload, n) for _ in range(args.steps)]
    v = sum(s["value"] for s in stats) / len(stats)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = {"impl": "reference", "metric": wl["metric"], "value": v, "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": n / v * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["text"], "rays_per_step": n},
            "cpu_baseline": {**stats[0], "value": v},
            "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def run_reference_gpu(args):
    """Context arm: the unmodified reference, eager PyTorch fp32 (TF32 off), on the B200(s): `net.cuda()`,
    `bind_parallel(net, gpus)` = nn.DataParallel(dim=1) when N > 1 (reference src/render/nerf.py:354-371), rays split in
    `ray_batch_size` = 50 000 pieces like eval/gen_video.py:213-216.  Single process (rank 0 only under torchrun)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    cfg = synth.CONFIGS[args.workload]
    if reference_root() is None:
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref not installed (build() with a reference checkout)"}))
        return
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    gpus = list(range(args.gpus))
    device = torch.device("cuda", 0)
    net, renderer = build_reference_scene(args.workload, device)
    render_par = renderer.bind_parallel(net, gpus, simple_output=True).eval()
    frame = args.rays if args.rays else wl["frame_rays"]
    total = frame if args.scaling == "strong" else frame * args.gpus
    rays = synth.make_rays(cfg, total, n_target=max(8, total // (cfg["W"] * cfg["H"]) + 1)).to(device)

    def step():
        with torch.no_grad():
            out = [render_par(r[None])[0] for r in torch.split(rays, 50000, dim=0)]
        return torch.cat(out, dim=1)
    for _ in range(max(args.warmup, 1)):
        step()
    for g in gpus:
        torch.cuda.synchronize(g)
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    for g in gpus:
        torch.cuda.synchronize(g)
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = max(e0.elapsed_time(e1), 0.0)
    v = total * args.steps / (ms / 1e3)
    print(json.dumps({"impl": "reference-gpu", "metric": wl["metric"], "value": v, "unit": "rays/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": ms / args.steps,
                      "wall_ms_per_step": wall_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
                      "dtype": "f32 (TF32 off)", "data": "synthetic",
                      "config": {"workload": wl["text"], "rays_per_step": total, "ray_batch_size": 50000,
                                 "parallelism": "single GPU" if args.gpus == 1 else f"nn.DataParallel(dim=1) x{args.gpus}",
                                 "note": "unmodified reference (oracle/_ref), PyTorch eager"}}))


def run_torch_eager(args):
    """Context number: the composed torch-op path of THIS repo (the same ATen op sequence as the reference's PyTorch
    code) on ONE GPU in fp32 (TF32 off, 50 000-point chunks).  `--impl reference-gpu` is the real reference."""
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    device = torch.device("cuda", 0)
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = synth.CONFIGS[args.workload]
    net, renderer = build_scene(cfg, device, "simt")
    n = args.rays if args.rays else WORKLOADS[args.workload]["frame_rays"]
    rays = synth.make_rays(cfg, n).to(device)[None]

    class TorchField:            # a generic `model` callable for NeRFRenderer's composed path
        use_viewdirs = True

        def __call__(self, xyz, coarse=True, viewdirs=None):
            return net._forward_autograd(xyz, coarse, viewdirs)

    field = TorchField()

    def step():
        with torch.no_grad():
            return renderer._forward_torch(field, rays, False)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    print(json.dumps({"impl": "torch-eager", "metric": WORKLOADS[args.workload]["metric"],
                      "value": n * args.steps / (ms / 1e3), "unit": "rays/s", "n_gpus": 1, "steps": args.steps,
                      "ms_per_step": ms / args.steps, "dtype": "f32",
                      "config": {"workload": args.workload.upper(), "rays_per_step": n,
                                 "note": "composed torch ops of this repo's autograd path under no_grad"}}))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu", "torch-eager"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--engine", default=os.environ.get("PNR_ENGINE", "auto"), choices=["auto", "simt", "tc"])
    ap.add_argument("--rays", type=int, default=0,
                    help="rays per step per GPU (weak) / per job (strong); default = one frame of the workload")
    ap.add_argument("--cpu-rays", type=int, default=0, help="rays per CPU-reference pass (default per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rgb / depth the last timed step rendered as DIR/<name>.npy (float32, at most 64 MB "
                         "in all: a fixed sample of rays above that); the same arguments give the same inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours renders")
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "reference-gpu":
        run_reference_gpu(a)
    elif a.impl == "torch-eager":
        run_torch_eager(a)
    else:
        run_ours(a)
