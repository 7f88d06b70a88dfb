"""Test infrastructure for the drop-in tests: the overlay tree (scripts/install_ref.py), a tiny SRN-format dataset on
disk, and a conf that switches the ImageNet download off.  The reference scripts themselves run UNMODIFIED."""
import importlib.util
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIMS = os.path.join(ROOT, "tests", "shims")


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


install_ref = _load("pnr_install_ref", os.path.join(ROOT, "scripts", "install_ref.py"))


def reference_root():
    """The reference checkout for tests: $PIXELNERF_REF, else the copy build() installs in oracle/_ref; None if neither."""
    return install_ref.find_reference()


def make_overlay(tmp):
    ref = reference_root()
    if ref is None:
        return None
    return install_ref.make_overlay(os.path.join(str(tmp), "overlay"), ref_root=ref)


def env_for_scripts():
    env = dict(os.environ)
    env["PYTHONPATH"] = SHIMS + os.pathsep + env.get("PYTHONPATH", "")
    ref = reference_root()
    if ref:
        env["PIXELNERF_REF"] = ref
    return env


def run_script(overlay, rel, argv, cwd, timeout=900):
    return subprocess.run([sys.executable, os.path.join(overlay, rel), *argv], cwd=str(cwd), env=env_for_scripts(),
                          capture_output=True, text=True, timeout=timeout)


def write_test_conf(overlay, path, extra=""):
    """exp conf = the reference's conf/exp/srn.conf, minus the ImageNet download (no network in the test image)."""
    with open(path, "w") as f:
        f.write('include required("%s")\n' % os.path.join(overlay, "conf", "exp", "srn.conf"))
        f.write("model {\n  encoder {\n    pretrained = False\n  }\n}\n")
        f.write(extra)
    return path


def _pose(theta_deg, phi_deg, radius):
    synth = _load("pnr_synth_for_dropin", os.path.join(ROOT, "pixel-nerf_b200", "synth.py"))
    return synth.pose_spherical(theta_deg, phi_deg, radius).numpy()


def make_srn_dataset(base, n_obj=2, n_views=4, size=128, seed=0):
    """<base>_{train,val,test}/<obj>/{rgb/*.png, pose/*.txt, intrinsics.txt} in the layout SRNDataset reads
    (reference src/data/SRNDataset.py:37-107).  White background with a coloured disc so every image has a bbox."""
    import cv2
    rng = np.random.RandomState(seed)
    flip = np.diag([1.0, -1.0, -1.0, 1.0])   # SRNDataset multiplies poses by this (its own inverse)
    for stage in ("train", "val", "test"):
        for o in range(n_obj):
            d = f"{base}_{stage}/obj{o:03d}"
            os.makedirs(d + "/rgb", exist_ok=True)
            os.makedirs(d + "/pose", exist_ok=True)
            with open(d + "/intrinsics.txt", "w") as f:
                f.write(f"{131.25 * size / 128:.4f} {size / 2:.1f} {size / 2:.1f} 0.\n0. 0. 0.\n1.\n{size} {size}\n")
            for v in range(n_views):
                img = np.full((size, size, 3), 255, np.uint8)
                yy, xx = np.mgrid[:size, :size]
                cx, cy, r = rng.randint(size // 3, 2 * size // 3, 2).tolist() + [size // 5]
                mask = (xx - cx) ** 2 + (yy - cy) ** 2 < r * r
                img[mask] = rng.randint(0, 200, 3)
                img[mask] = (img[mask] * (0.5 + 0.5 * rng.rand(int(mask.sum()), 1))).astype(np.uint8)
                cv2.imwrite(f"{d}/rgb/{v:06d}.png", img)
                pose = _pose(360.0 * v / n_views + 17.0 * o, -20.0, 1.3) @ flip
                np.savetxt(f"{d}/pose/{v:06d}.txt", pose.reshape(1, 16))
    return base
