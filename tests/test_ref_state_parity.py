"""State producer and checkpoint compatibility against the UNMODIFIED reference, through the golden data that
tests/ref_probe.py wrote by running it (tests/golden/ref_encoder.npz, ref_checkpoint.npz); the seeded recipes both
share are in tests/ref_recipes.py:

  * a19: `SpatialEncoder.forward` / `PixelNeRFNet.encode` -- same state_dict, same images -> the same latent, camera
    state and `index()` values as the reference (src/model/encoder.py:111-164, src/model/models.py:89-144);
  * f-4: a checkpoint as the reference's own `save_weights` writes it strict-loads here and gives the reference's field
    values; a checkpoint written here has the names, order, shapes and values the reference's strict
    `load_weights` needs (src/model/models.py:268-316).
"""
import os

import numpy as np
import torch

import golden_util as gu
import gpu_util
import ref_recipes

ENC = np.load(os.path.join(gu.GOLD, "ref_encoder.npz"))
CKPT = np.load(os.path.join(gu.GOLD, "ref_checkpoint.npz"))


class Args:
    def __init__(self, d, name, resume=True):
        self.checkpoints_path, self.name, self.resume = d, name, resume


def assert_same_state(sd, keys, digests):
    """Same names in the same order, and bit-identical tensors, as the reference's state_dict."""
    assert list(sd.keys()) == keys.tolist()
    bad = [k for k, d in zip(keys, digests) if not np.array_equal(ref_recipes.digest(sd[k]), d)]
    assert not bad, f"tensors differ from the reference's: {bad[:5]}"


def assert_sampled(t, z, prefix, seed, rel, mean_dims):
    """|t - ref| <= rel * max|ref| on the stored sample of elements and on the per-channel means (ref_probe.sampled)."""
    tol = rel * float(z[prefix + "_max"])
    assert tuple(t.shape) == tuple(z[prefix + "_shape"]), prefix
    idx = ref_recipes.sample_index(t.numel(), seed)
    assert (t.reshape(-1)[idx] - torch.from_numpy(z[prefix + "_sample"])).abs().max() <= tol, prefix
    assert (t.double().mean(mean_dims) - torch.from_numpy(z[prefix + "_mean"])).abs().max() <= tol, prefix


def test_encoder_and_encode_state_match_the_reference():
    from model import make_model
    for name, use_first_pool, (SB, NS, H, W) in ref_recipes.ENCODER_CASES:
        g = lambda k: ENC[f"{name}/{k}"]
        net = ref_recipes.encoder_net(make_model, gpu_util.model_conf, use_first_pool)
        assert_same_state(net.state_dict(), g("sd_keys"), g("sd_digest"))
        images, poses, focal, c = ref_recipes.scene(7, SB, NS, H, W)
        assert np.array_equal(np.stack([ref_recipes.digest(t) for t in (images, poses, focal, c)]), g("inputs_digest"))
        uv = ref_recipes.encoder_uv(SB, NS, H, W)
        assert torch.equal(uv, torch.from_numpy(g("uv")))
        with torch.enable_grad():     # CPU tensors: the composed-torch path (encode() itself has no fused part)
            net.encode(images, poses, focal, c=c)
            idx = net.encoder.index(uv, None, net.image_shape)
        assert_sampled(net.encoder.latent.detach(), ENC, f"{name}/latent", 1, 1e-6, (2, 3))
        assert torch.equal(net.encoder.latent_scaling, torch.from_numpy(g("latent_scaling")))
        assert torch.equal(net.poses, torch.from_numpy(g("poses_state")))
        assert torch.equal(net.focal, torch.from_numpy(g("focal_state")))
        assert torch.equal(net.c, torch.from_numpy(g("c_state")))
        assert torch.equal(net.image_shape, torch.from_numpy(g("image_shape")))
        assert net.num_views_per_obj == int(g("num_views_per_obj"))
        assert_sampled(idx.detach(), ENC, f"{name}/index", 2, 1e-5, (1,))


def test_checkpoints_round_trip_with_the_reference(tmp_path):
    from model import make_model
    d = str(tmp_path)
    # the checkpoint the reference's save_weights wrote: torch.save(state_dict) at <checkpoints>/<name>/pixel_nerf_latest
    src = ref_recipes.checkpoint_net(make_model, gpu_util.model_conf).state_dict()
    assert_same_state(src, CKPT["sd_keys"], CKPT["sd_digest"])
    os.makedirs(os.path.join(d, "probe"))
    torch.save(src, os.path.join(d, "probe", "pixel_nerf_latest"))
    net = make_model(gpu_util.model_conf(512, True)).eval()
    before = net.mlp_coarse.lin_in.weight.clone()
    assert net.load_weights(Args(d, "probe"), strict=True) is net
    assert not torch.equal(before, net.mlp_coarse.lin_in.weight), "checkpoint was not loaded"
    images, poses, focal, c = ref_recipes.scene(5, 1, 2, 32, 32)
    assert np.array_equal(np.stack([ref_recipes.digest(t) for t in (images, poses, focal, c)]), CKPT["inputs_digest"])
    xyz, dirs = torch.from_numpy(CKPT["xyz"]), torch.from_numpy(CKPT["dirs"])
    with torch.enable_grad():                                      # CPU: composed-torch field
        net.encode(images, poses, focal, c=c)
        oc = net(xyz.requires_grad_(True), coarse=True, viewdirs=dirs).detach()
        of = net(xyz, coarse=False, viewdirs=dirs).detach()
    assert (oc - torch.from_numpy(CKPT["out_coarse"])).abs().max() < 1e-5
    assert (of - torch.from_numpy(CKPT["out_fine"])).abs().max() < 1e-5
    # and back: our save_weights writes the files the reference's writes, and what the reference's
    # load_weights(strict=True) reads from them is the state it computed out_coarse / out_fine with
    os.makedirs(os.path.join(d, "ours"), exist_ok=True)
    net.save_weights(Args(d, "ours"))
    net.save_weights(Args(d, "ours"))
    assert sorted(os.listdir(os.path.join(d, "ours"))) == CKPT["files"].tolist()
    assert_same_state(torch.load(os.path.join(d, "ours", "pixel_nerf_latest")), CKPT["sd_keys"], CKPT["sd_digest"])
    # opt_init semantics (models.py:276-283): no resume + opt_init -> nothing is loaded, returns None
    assert net.load_weights(Args(d, "probe", resume=False), opt_init=True) is None
