"""Recipes shared by the reference-parity tests and by tests/ref_probe.py, which ran the reference on the same inputs to
write tests/golden/ref_*.npz: seeded scenes and networks, tensor digests, the element sample of large outputs, and the
flattened form of a parsed conf.  Nothing here needs the reference."""
import hashlib
import importlib.util
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


synth = load_by_path("pnr_synth_for_ref_recipes", os.path.join(ROOT, "pixel-nerf_b200", "synth.py"))

# name, use_first_pool, (SB, NS, H, W)
ENCODER_CASES = (("pool", True, (2, 2, 48, 64)), ("nopool", False, (1, 3, 40, 40)))
N_SAMPLE = 2048


def scene(seed, SB, NS, H, W):
    g = torch.Generator().manual_seed(seed)
    images = torch.rand(SB, NS, 3, H, W, generator=g) * 2 - 1
    poses = torch.eye(4).repeat(SB, NS, 1, 1)
    poses[..., :3, :3] = torch.linalg.qr(torch.randn(SB, NS, 3, 3, generator=g))[0]
    poses[..., :3, 3] = torch.randn(SB, NS, 3, generator=g)
    focal = torch.rand(SB, 2, generator=g) * 50 + 40
    c = torch.rand(SB, 2, generator=g) * 4 + torch.tensor([W / 2.0, H / 2.0])
    return images, poses, focal, c


def digest(t):
    """sha256 over dtype, shape and bytes of a tensor."""
    t = t.detach().contiguous()
    h = hashlib.sha256(f"{t.dtype} {tuple(t.shape)}".encode())
    h.update(t.numpy().tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def state_digests(sd):
    return np.array(list(sd.keys())), np.stack([digest(v) for v in sd.values()])


def sample_index(numel, seed):
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:N_SAMPLE]


def encoder_net(make_model, model_conf, use_first_pool):
    """Seed-3 init (the reference and this package build bit-identical resnet34 trunks from one seed), BatchNorm running
    stats moved away from their (0, 1) initial values so that eval-mode BN does real work, synthetic MLP weights."""
    torch.manual_seed(3)
    net = make_model(model_conf(64, use_first_pool)).eval()
    with torch.no_grad():
        for m in net.encoder.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    net.mlp_coarse.load_state_dict(synth.make_mlp_weights(31, 64))
    net.mlp_fine.load_state_dict(synth.make_mlp_weights(32, 64))
    return net


def encoder_uv(SB, NS, H, W):
    g = torch.Generator().manual_seed(8)
    return torch.rand(SB * NS, 33, 2, generator=g) * torch.tensor([W * 1.2, H * 1.2]) - 3.0


def checkpoint_net(make_model, model_conf):
    """The network whose checkpoint the reference writes: seed-11 init, non-degenerate synthetic MLP weights."""
    torch.manual_seed(11)
    net = make_model(model_conf(512, True)).eval()
    net.mlp_coarse.load_state_dict(synth.bench_mlp_weights(41, 512))
    net.mlp_fine.load_state_dict(synth.bench_mlp_weights(42, 512))
    return net


def checkpoint_points():
    g = torch.Generator().manual_seed(12)
    xyz = torch.randn(1, 64, 3, generator=g) * 0.4
    dirs = torch.nn.functional.normalize(torch.randn(1, 64, 3, generator=g), dim=-1)
    return xyz, dirs


def flatten(c, prefix=""):
    out = {}
    for k in c.keys():
        v = c[k]
        if hasattr(v, "keys"):
            out.update(flatten(v, prefix + k + "."))
        else:
            out[prefix + k] = v
    return out
