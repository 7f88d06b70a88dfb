"""TEST INFRASTRUCTURE: runs the UNMODIFIED reference in its own interpreter (its packages are called `model`, `render`,
`util` like this repo's, so the two cannot share one) and writes the golden data that tests/test_ref_state_parity.py
and tests/test_host_logic.py compare against:

  python tests/ref_probe.py tests/golden      # the reference: $PIXELNERF_REF, else oracle/_ref (oracle/ref_harness.py)

  ref_encoder.npz     SpatialEncoder / encode() state on two small scenes  (SURVEY 8a row a19)
  ref_checkpoint.npz  what the reference's own save_weights writes, and its field values for that checkpoint (row f-4)
  ref_confs.json      the reference's conf/exp/*.conf and expconf.conf, parsed with this package's HOCON reader

The networks are rebuilt at test time from the recipes in tests/ref_recipes.py (same seeds, same code path); the
stored per-tensor digests prove that the rebuilt weights are the ones the reference ran with.  Large outputs are stored as a fixed,
seeded sample of elements plus per-channel means and the full tensor's max |value|.
"""
import json
import os
import sys

import numpy as np
import torch

from ref_recipes import (ENCODER_CASES, ROOT, checkpoint_net, checkpoint_points, digest, encoder_net, encoder_uv,
                         flatten, load_by_path, sample_index, scene, state_digests)

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness as rh  # noqa: E402


def sampled(prefix, t, seed, mean_dims):
    """Seeded sample, per-channel means (float64) and max |value| of a large tensor."""
    t = t.detach()
    idx = sample_index(t.numel(), seed)
    return {prefix + "_shape": np.array(t.shape), prefix + "_max": np.array(t.abs().max().item()),
            prefix + "_sample": t.reshape(-1)[idx].numpy(), prefix + "_mean": t.double().mean(mean_dims).numpy()}


class _Args:
    def __init__(self, d, name="probe", resume=True):
        self.checkpoints_path, self.name, self.resume = d, name, resume


def write_encoder(out):
    model, _, _ = rh.import_reference()
    rec = {}
    for name, use_first_pool, (SB, NS, H, W) in ENCODER_CASES:
        net = encoder_net(model.make_model, rh.model_conf, use_first_pool)
        images, poses, focal, c = scene(7, SB, NS, H, W)
        uv = encoder_uv(SB, NS, H, W)
        with torch.no_grad():
            net.encode(images, poses, focal, c=c)
            idx = net.encoder.index(uv, None, net.image_shape)
        keys, dig = state_digests(net.state_dict())
        rec.update({f"{name}/sd_keys": keys, f"{name}/sd_digest": dig, f"{name}/uv": uv.numpy(),
                    f"{name}/inputs_digest": np.stack([digest(t) for t in (images, poses, focal, c)]),
                    f"{name}/latent_scaling": net.encoder.latent_scaling.numpy(),
                    f"{name}/poses_state": net.poses.numpy(), f"{name}/focal_state": net.focal.numpy(),
                    f"{name}/c_state": net.c.numpy(), f"{name}/image_shape": net.image_shape.numpy(),
                    f"{name}/num_views_per_obj": np.array(net.num_views_per_obj)})
        rec.update(sampled(f"{name}/latent", net.encoder.latent, 1, (2, 3)))
        rec.update(sampled(f"{name}/index", idx, 2, (1,)))
    np.savez_compressed(out, **rec)


def write_checkpoint(out, tmp):
    """The reference's own `save_weights` (models.py:300-316), twice so that the backup file is rolled, and the field
    values its own forward gives for that checkpoint on a small scene."""
    model, _, _ = rh.import_reference()
    net = checkpoint_net(model.make_model, rh.model_conf)
    os.makedirs(os.path.join(tmp, "probe"), exist_ok=True)
    net.save_weights(_Args(tmp))
    net.save_weights(_Args(tmp))
    written = torch.load(os.path.join(tmp, "probe", "pixel_nerf_latest"))
    keys, dig = state_digests(written)
    images, poses, focal, c = scene(5, 1, 2, 32, 32)
    xyz, dirs = checkpoint_points()
    with torch.no_grad():
        net.encode(images, poses, focal, c=c)
        out_c = net(xyz, coarse=True, viewdirs=dirs)
        out_f = net(xyz, coarse=False, viewdirs=dirs)
    assert out_c[..., 3].std() > 0 and out_f[..., :3].std() > 0, "degenerate field values"
    np.savez_compressed(out, sd_keys=keys, sd_digest=dig, files=np.array(sorted(os.listdir(os.path.join(tmp, "probe")))),
                        inputs_digest=np.stack([digest(t) for t in (images, poses, focal, c)]),
                        xyz=xyz.numpy(), dirs=dirs.numpy(), out_coarse=out_c.numpy(), out_fine=out_f.numpy())


def write_confs(out):
    hocon = load_by_path("pnr_hocon_for_probe", os.path.join(ROOT, "pixel-nerf_b200", "src", "util", "hocon.py"))
    names = ["conf/exp/" + n for n in sorted(os.listdir(os.path.join(rh.REF_ROOT, "conf", "exp")))] + ["expconf.conf"]
    with open(out, "w") as f:
        json.dump({n: flatten(hocon.parse_file(os.path.join(rh.REF_ROOT, n))) for n in names}, f, indent=1,
                  sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    import tempfile
    dest = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    torch.set_num_threads(os.cpu_count())
    write_encoder(os.path.join(dest, "ref_encoder.npz"))
    with tempfile.TemporaryDirectory() as tmp:
        write_checkpoint(os.path.join(dest, "ref_checkpoint.npz"), tmp)
    write_confs(os.path.join(dest, "ref_confs.json"))
    for n in ("ref_encoder.npz", "ref_checkpoint.npz", "ref_confs.json"):
        print(n, os.path.getsize(os.path.join(dest, n)), "bytes")
