"""The reference's UNMODIFIED eval/gen_video.py and train/train.py, run end to end on the GPU against this package through
the overlay tree (scripts/install_ref.py): synthetic SRN-format dataset on disk, reference conf/exp/srn.conf with the
ImageNet download switched off.  The reference comes from oracle/_ref (installed by build())."""
import glob
import os

import numpy as np
import pytest
import torch

import dropin_util as du

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(du.reference_root() is None, reason="no reference checkout (oracle/_ref: build() with one present, or PIXELNERF_REF)")]


def test_gen_video_main_runs_unmodified(tmp_path):
    overlay = du.make_overlay(tmp_path)
    data = du.make_srn_dataset(str(tmp_path / "data" / "cars"), n_obj=1, n_views=4, size=64)
    conf = du.write_test_conf(overlay, str(tmp_path / "test.conf"))
    # a checkpoint for `net.load_weights(args)` (gen_video.py:104): the reference's own init zeroes every fc_1 and
    # mostly renders sigma = 0 (a blank frame), so store the synthetic weights of the benchmarks under the name the
    # script will look for -- this also runs the checkpoint ingest (SURVEY 8f-4) through the unmodified script
    import gpu_util
    import golden_util as gu
    from model import make_model
    net = make_model(gpu_util.model_conf(512))
    net.mlp_coarse.load_state_dict(gu.synth.bench_mlp_weights(31, 512))
    net.mlp_fine.load_state_dict(gu.synth.bench_mlp_weights(32, 512))
    os.makedirs(str(tmp_path / "checkpoints" / "dropin"), exist_ok=True)
    torch.save(net.state_dict(), str(tmp_path / "checkpoints" / "dropin" / "pixel_nerf_latest"))
    r = du.run_script(overlay, "eval/gen_video.py",
                      ["-n", "dropin", "-c", conf, "-D", data, "-F", "srn", "--split", "test", "-S", "0", "--source", "0 2",
                       "--num_views", "3", "--scale", "0.25", "--ray_batch_size", "2000", "--gpu_id", "0"],
                      cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "Wrote to" in r.stdout and "Load checkpoints/dropin/pixel_nerf_latest" in r.stdout
    vids = glob.glob(str(tmp_path / "visuals" / "dropin" / "videot0000_v000_002.mp4.npy"))
    assert len(vids) == 1, os.listdir(str(tmp_path / "visuals" / "dropin"))
    frames = np.load(vids[0])
    assert frames.shape == (3, 32, 32, 3) and frames.dtype == np.uint8
    assert frames.std() > 0                                    # not a constant image
    assert os.path.exists(str(tmp_path / "visuals" / "dropin" / "videot0000_v000_002_view.jpg"))


def test_train_main_runs_unmodified(tmp_path):
    """Two epochs of two batches (SB = 2 objects, 2 source views, 128 rays each): training steps through the fused
    backward, the no-grad eval and visualisation steps through the fused forward, checkpoints written on the way."""
    overlay = du.make_overlay(tmp_path)
    data = du.make_srn_dataset(str(tmp_path / "data" / "cars"), n_obj=4, n_views=5, size=128)
    conf = du.write_test_conf(overlay, str(tmp_path / "test.conf"),
                              extra="train {\n  print_interval = 1\n  save_interval = 2\n  vis_interval = 2\n  eval_interval = 2\n}\n")
    r = du.run_script(overlay, "train/train.py",
                      ["-n", "dropin_train", "-c", conf, "-D", data, "-F", "srn", "-B", "2", "-V", "2", "--epochs", "2",
                       "--gpu_id", "0", "--lr", "1e-4"], cwd=tmp_path, timeout=1500)
    assert r.returncode == 0, (r.stderr[-3000:], r.stdout[-1000:])
    assert "*** Eval:" in r.stdout and "generating visualization" in r.stdout and "saving" in r.stdout
    losses = [float(l.split("t:")[1].split()[0]) for l in r.stdout.splitlines() if l.startswith("E ") and " t:" in l]
    assert len(losses) == 4 and all(np.isfinite(losses))
    ck = str(tmp_path / "checkpoints" / "dropin_train")
    for f in ("pixel_nerf_latest", "_renderer", "_optim", "_iter"):
        assert os.path.exists(os.path.join(ck, f)), os.listdir(ck)
    sd = torch.load(os.path.join(ck, "pixel_nerf_latest"), map_location="cpu")
    assert all(torch.isfinite(v).all() for v in sd.values() if v.is_floating_point())
    assert glob.glob(str(tmp_path / "visuals" / "dropin_train" / "*_vis.png"))
