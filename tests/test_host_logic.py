"""Host-side logic on CPU: HOCON reader, conf files, model/renderer construction, state_dict
compatibility, unsupported-flag errors, schedule, DotMap, no-CPU-fallback guard."""
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pixel-nerf_b200")
sys.path.insert(0, os.path.join(PKG, "src"))

from util import hocon  # noqa: E402
import golden_util as gu  # noqa: E402
import gpu_util  # noqa: E402
import ref_recipes  # noqa: E402


def test_hocon_subset():
    c = hocon.parse_string('''
      # comment
      a { b = 1, c = [1, 2.5, x]  // trailing
          d { e = True } }
      a.b = 2
      a { d { f = "s t" } }
      g : null
      h = some bare words
    ''')
    assert c.get_int("a.b") == 2 and c["a.c"] == [1, 2.5, "x"]
    assert c.get_bool("a.d.e") is True and c.get_string("a.d.f") == "s t"
    assert c.get("g") is None and c["h"] == "some bare words"
    assert "a.d.e" in c and "a.zz" not in c
    assert c.get_int("missing", 7) == 7
    with pytest.raises(KeyError):
        c.get_int("missing")


@pytest.mark.parametrize("name", ["srn", "sn64", "dtu", "sn64_unseen", "multi_obj"])
def test_conf_files_resolve_includes(name):
    c = hocon.parse_file(os.path.join(PKG, "conf", "exp", name + ".conf"))
    assert c.get_int("model.mlp_coarse.n_blocks") == 5 and c.get_int("model.mlp_coarse.combine_layer") == 3
    assert c.get_int("renderer.n_coarse") == 64 and c.get_list("renderer.sched") == []
    assert c.get_float("renderer.white_bkgd") == (0.0 if name == "dtu" else 1.0)
    assert c.get_bool("model.encoder.use_first_pool", True) == (name not in ("sn64", "sn64_unseen"))
    assert c.get_string("data.format") == {"srn": "srn", "sn64": "dvr", "dtu": "dvr_dtu", "sn64_unseen": "dvr_gen",
                                           "multi_obj": "multi_obj"}[name]


def test_shipped_confs_equal_the_reference_confs():
    """Every exp conf and expconf.conf of this package parses to the same tree as the reference's own file (read with
    the same in-repo HOCON reader; the reference's files are the schema, stored parsed in tests/golden/ref_confs.json
    by tests/ref_probe.py)."""
    with open(os.path.join(gu.GOLD, "ref_confs.json")) as f:
        theirs = json.load(f)
    assert len(theirs) == 6 and "expconf.conf" in theirs
    for name, tree in theirs.items():
        assert ref_recipes.flatten(hocon.parse_file(os.path.join(PKG, name))) == tree, name


def test_model_state_dict_keys_and_shapes():
    case = gu.load_case("tiny")
    net = gpu_util.build_net(case, device="cpu", engine="simt")
    sd = net.state_dict()
    for k in ("code._freqs", "code._phases", "mlp_coarse.lin_in.weight", "mlp_coarse.lin_z.2.bias",
              "mlp_coarse.blocks.4.fc_1.weight", "mlp_fine.lin_out.bias", "encoder.model.conv1.weight"):
        assert k in sd, k
    assert sd["mlp_coarse.lin_in.weight"].shape == (32, 42)
    assert not any(k.startswith(("poses", "focal", "image_shape")) for k in sd)  # non-persistent buffers
    assert net.d_in == 42 and net.d_latent == 512 and net.use_viewdirs


def test_reference_init_zeroes_fc1():
    from model.resnetfc import ResnetFC
    m = ResnetFC(42, d_latent=512, d_hidden=64, combine_layer=3)
    assert all(float(b.fc_1.weight.abs().sum()) == 0.0 for b in m.blocks)
    assert len(m.lin_z) == 3


def test_unsupported_flags_raise_by_name():
    from model import make_model
    conf = gpu_util.model_conf(32)
    conf.put("use_code_viewdirs", True)
    with pytest.raises(NotImplementedError, match="use_code_viewdirs"):
        make_model(conf)
    conf = gpu_util.model_conf(32)
    conf.put("mlp_coarse.combine_type", "max")
    with pytest.raises(NotImplementedError, match="combine_type"):
        make_model(conf)
    from render import NeRFRenderer
    with pytest.raises(NotImplementedError, match="lindisp"):
        NeRFRenderer(lindisp=True)
    # the fused kernels compute the shipped positional code (6 frequencies x 1.5, input included) in registers:
    # any other code is refused by name instead of being trained with one encoding and rendered with another
    for key, val in (("code.freq_factor", 3.14159), ("code.num_freqs", 4), ("code.include_input", False)):
        conf = gpu_util.model_conf(32)
        conf.put(key, val)
        with pytest.raises((NotImplementedError, AssertionError, RuntimeError), match="code|size|shape|mat1"):
            make_model(conf)


def test_scene_epoch_and_contiguous_camera_state():
    """encode() / set_scene() bump the epoch that keys per-GPU replicas, and the camera buffers whose raw pointers go
    to the kernels are contiguous whatever layout the caller's focal / c tensors have."""
    from model import make_model
    net = make_model(gpu_util.model_conf(32)).eval()
    e0 = net._scene_epoch
    poses = torch.eye(4).repeat(2, 2, 1, 1)
    focal = (torch.rand(2, 4) * 10 + 30)[:, ::2]      # non-contiguous (SB, 2) view
    c = torch.rand(2, 4)[:, 1::2]                      # non-contiguous (SB, 2) view
    net.set_scene(torch.rand(4, 512, 8, 8), poses, focal, c, 16, 16)
    assert net._scene_epoch == e0 + 1
    assert net.focal.is_contiguous() and net.c.is_contiguous() and net.poses.is_contiguous()
    assert not focal.is_contiguous() and not c.is_contiguous()
    assert torch.equal(net.focal[:, 1], -focal[:, 1]) and torch.equal(net.c, c)
    net.set_cameras(poses.reshape(-1, 4, 4), focal, c, 16, 16)
    assert net._scene_epoch == e0 + 2


def test_renderer_conf_schedule_and_state():
    from render import NeRFRenderer
    conf = hocon.from_dict(dict(n_coarse=8, n_fine=4, n_fine_depth=2, white_bkgd=True, sched=[[2, 4], [16, 32], [8, 16]]))
    r = NeRFRenderer.from_conf(conf, eval_batch_size=123)
    assert (r.n_coarse, r.n_fine, r.n_fine_depth, r.eval_batch_size, r.using_fine) == (8, 4, 2, 123, True)
    assert r.white_bkgd == 1.0 and set(r.state_dict().keys()) == {"iter_idx", "last_sched"}
    r.sched_step(2)
    assert (r.n_coarse, r.n_fine, int(r.last_sched)) == (16, 8, 1)
    r.sched_step(2)
    assert (r.n_coarse, r.n_fine, int(r.last_sched)) == (32, 16, 2)


def test_no_cpu_fallback_in_inference():
    case = gu.load_case("tiny")
    net = gpu_util.build_net(case, device="cpu", engine="simt")
    renderer = gpu_util.build_renderer(case)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="CUDA"):
            net(case["ref"]["field_xyz"], coarse=True, viewdirs=case["ref"]["field_dirs"])
        with pytest.raises(RuntimeError, match="CUDA"):
            renderer(net, case["rays"])


def test_autograd_path_matches_reference_goldens():
    """The documented grad-mode (training) path: composed torch ops, seeded like the reference."""
    case = gu.load_case("tiny")
    net = gpu_util.build_net(case, device="cpu", engine="simt")
    renderer = gpu_util.build_renderer(case)
    torch.manual_seed(case["seed"] + 4)
    out = renderer(net, case["rays"], want_weights=True)
    assert (out.fine.rgb - case["ref"]["fine_rgb"]).abs().max() < 1e-6
    out.fine.rgb.sum().backward()
    assert net.mlp_fine.lin_in.weight.grad is not None


@pytest.mark.parametrize("name", gu.GRAD_CASE_NAMES)
def test_training_step_gradients_match_reference(name):
    """train/train.py:199-215 through this package's classes in grad mode (`render_par(rays, want_weights=True)`,
    MSE coarse + MSE fine, backward): the gradients of every MLP parameter and of the latent equal the ones the
    reference computed for the same inputs and seed (tests/golden/grad_*.npz)."""
    case, g = gu.load_case(name), gu.load_grad_case(name)
    net = gpu_util.build_net(case, device="cpu", engine="simt").train()
    net.encoder.latent = case["latent"].clone().requires_grad_(True)
    renderer = gpu_util.build_renderer(case).train()
    render_par = renderer.bind_parallel(net, None).train()
    torch.manual_seed(case["seed"] + 4)
    out = render_par(case["rays"], want_weights=True)
    crit = torch.nn.MSELoss()
    loss = crit(out["coarse"]["rgb"], g["rgb_gt"])
    if case["cfg"]["n_fine"] > 0:
        loss = loss * 1.0 + crit(out["fine"]["rgb"], g["rgb_gt"]) * 1.0
    assert abs(loss.item() - g["loss"]) < 1e-6
    loss.backward()

    def close(a, ref):
        return (a - ref).abs().max() <= 1e-4 * ref.abs().max() + 1e-9

    assert close(net.encoder.latent.grad, g["g_latent"])
    for k, p in net.mlp_coarse.named_parameters():
        assert close(p.grad, g["gc"][k]), ("coarse", k)
    if net.mlp_fine is not None:
        for k, p in net.mlp_fine.named_parameters():
            assert close(p.grad, g["gf"][k]), ("fine", k)


def test_dotmap_compat():
    from render.dotmap_compat import DotMap
    d = DotMap(coarse=DotMap(rgb=1))
    d.fine.depth = 2
    assert d.coarse.rgb == 1 and d.toDict() == {"coarse": {"rgb": 1}, "fine": {"depth": 2}}


def test_parse_args_with_expconf(tmp_path, monkeypatch):
    from util import args as uargs
    monkeypatch.chdir(tmp_path)
    a, conf = uargs.parse_args(argv=["-n", "srn_car", "--gpu_id", "0 1", "-R", "1000"])
    assert a.conf.endswith("conf/exp/srn.conf") and a.gpu_id == [0, 1] and a.ray_batch_size == 1000
    assert a.dataset_format == "srn" and conf.get_int("model.mlp_fine.d_hidden") == 512


def test_shard_bounds_follow_torch_chunk():
    from render.sharding import shard_bounds
    for n in (0, 1, 7, 8, 9, 50000):
        for w in (1, 2, 3, 8):
            sizes = [b - a for a, b in shard_bounds(n, w)]
            ref = [t.shape[0] for t in torch.chunk(torch.zeros(n), w)] if n else []
            assert [s for s in sizes if s] == ref
            assert sum(sizes) == n
