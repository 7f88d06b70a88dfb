#!/usr/bin/env python
"""Training-step throughput (SURVEY 8f-1): the reference's step -- encode(SB objects x NS views), render SB x B rays
with want_weights=True, MSE coarse + MSE fine, backward through MLPs and the encoder trunk, Adam step
(train/train.py:117-233, SB = 4 and B = 128 are its defaults) -- through this package's classes.

    python scripts/bench_train.py --mode render     # the package default: pnr_render + pnr_render_backward in one node
    python scripts/bench_train.py --mode field      # PNR_FUSED_BACKWARD=1: torch renderer, fused field fwd + pnr_field_backward
    python scripts/bench_train.py --mode torch      # PNR_FUSED_BACKWARD=0: composed-torch grad path of this package
    python scripts/bench_train.py --mode reference  # the UNMODIFIED reference (oracle/_ref), same step, same GPU

`--device cpu --tiny` checks the script itself (torch mode)."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "pixel-nerf_b200", "src"))
sys.path.insert(0, os.path.join(ROOT, "pixel-nerf_b200"))
import synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["torch", "field", "render", "reference"], default="render")
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--SB", type=int, default=4)
    ap.add_argument("--B", type=int, default=128)
    ap.add_argument("--tiny", action="store_true", help="d_hidden 32, 8+4 samples, 32x32 images: a script self-check")
    a = ap.parse_args()
    os.environ["PNR_FUSED_BACKWARD"] = {"torch": "0", "field": "1", "render": "2", "reference": "0"}[a.mode]
    dev = torch.device(a.device)
    W = H = 128
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    if a.mode == "reference":
        # the reference's own classes (packages `model` / `render` / `util` of oracle/_ref instead of this repo's)
        sys.path.remove(os.path.join(ROOT, "pixel-nerf_b200", "src"))
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_harness as rh
        model, render, _ = rh.import_reference()
        torch.manual_seed(0)
        net = model.make_model(rh.model_conf(512, True)).to(dev).train()
        NeRFRenderer = render.NeRFRenderer
        renderer = NeRFRenderer(n_coarse=64, n_fine=32, n_fine_depth=16, depth_std=0.01, white_bkgd=True).to(dev).train()
    else:
        import util
        from model import make_model
        from render import NeRFRenderer
        conf = util.hocon.parse_file(os.path.join(ROOT, "pixel-nerf_b200", "conf", "exp", "srn.conf"))
        conf.put("model.encoder.pretrained", False)
        if a.tiny:
            W = H = 32
            for k in ("model.mlp_coarse.d_hidden", "model.mlp_fine.d_hidden"):
                conf.put(k, 32)
            conf.put("renderer.n_coarse", 8)
            conf.put("renderer.n_fine", 4)
            conf.put("renderer.n_fine_depth", 2)
        torch.manual_seed(0)
        net = make_model(conf["model"]).to(dev).train()
        renderer = NeRFRenderer.from_conf(conf["renderer"], lindisp=False).to(dev).train()
    with torch.no_grad():                       # the reference zero-initialises fc_1: give every layer a gradient
        for mlp in (net.mlp_coarse, net.mlp_fine):
            for blk in mlp.blocks:
                blk.fc_1.weight.normal_(0, 0.03)
    render_par = renderer.bind_parallel(net, None).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    NS, SB, B = 2, a.SB, a.B
    z_near, z_far, focal = 0.8, 1.8, torch.tensor(131.25 * W / 128.0)
    g = torch.Generator().manual_seed(1)

    def batch():
        images = torch.rand(SB, NS, 3, H, W, generator=g) * 2 - 1
        src = torch.stack([torch.stack([synth.pose_spherical(40.0 * v + 25.0 * o, -30.0, 1.3) for v in range(NS)])
                           for o in range(SB)])
        tgt = torch.stack([synth.pose_spherical(100.0 + 70.0 * o, -10.0, 1.3) for o in range(SB)])
        all_rays = synth.gen_rays(tgt, W, H, float(focal), z_near, z_far).reshape(SB, -1, 8)
        pix = torch.randint(0, W * H, (SB, B), generator=g)
        rays = torch.stack([all_rays[o][pix[o]] for o in range(SB)])
        gt = torch.rand(SB, B, 3, generator=g)
        return images.to(dev), src.to(dev), rays.to(dev), gt.to(dev)

    def step():
        images, src, rays, gt = batch()
        net.encode(images, src, focal.to(dev))
        out = render_par(rays, want_weights=True)
        loss = torch.nn.functional.mse_loss(out["coarse"]["rgb"], gt)
        if "fine" in out and len(out["fine"]) > 0:
            loss = loss + torch.nn.functional.mse_loss(out["fine"]["rgb"], gt)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return float(loss.detach())

    sync = torch.cuda.synchronize if dev.type == "cuda" else (lambda *x: None)
    for _ in range(a.warmup):
        step()
    sync()
    t0 = time.perf_counter()
    losses = [step() for _ in range(a.steps)]
    sync()
    dt = time.perf_counter() - t0
    print(json.dumps({"metric": "training rays/s (encode + render fwd/bwd + Adam)", "mode": a.mode,
                      "value": SB * B * a.steps / dt, "ms_per_step": dt / a.steps * 1e3, "SB": SB, "B": B,
                      "loss_first": losses[0], "loss_last": losses[-1], "finite": bool(np.isfinite(losses).all())}))


if __name__ == "__main__":
    main()
