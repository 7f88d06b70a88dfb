"""north_star: "eval/gen_video.py and train/train.py drop in unchanged".  The reference's scripts start with
`sys.path.insert(0, <script dir>/../src)`, so the supported install is the overlay tree of scripts/install_ref.py
(the reference's eval/ train/ conf/ next to THIS package's src/).  These CPU tests execute the UNMODIFIED scripts'
module tops (all their imports, then `util.args.parse_args` -> `--help`) against the overlay of the reference copy that
build() installs in oracle/_ref, and check which files the names resolve to (against a stand-in checkout written by the
test, so that check needs no reference).
Running the scripts' main loops needs a GPU: tests/test_gpu_dropin_scripts.py."""
import os
import subprocess
import sys

import pytest

import dropin_util as du

SCRIPTS = ["train/train.py", "eval/gen_video.py", "eval/eval.py", "eval/eval_approx.py", "eval/eval_real.py"]

needs_ref = pytest.mark.skipif(du.reference_root() is None,
                               reason="no reference checkout (oracle/_ref: build() with one present, or PIXELNERF_REF)")


@needs_ref
@pytest.mark.parametrize("script", SCRIPTS)
def test_unmodified_script_top_imports_against_the_overlay(tmp_path, script):
    overlay = du.make_overlay(tmp_path)
    r = du.run_script(overlay, script, ["--help"], cwd=tmp_path, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "usage:" in r.stdout and "--conf" in r.stdout


def _stand_in_reference(root):
    """A checkout with the reference's layout whose out-of-scope files are stand-ins: what is checked here is which file
    each name resolves to.  `data/__init__.py` imports a sibling module, as the reference's does."""
    files = {
        "src/render/__init__.py": "",
        "src/model/loss.py": "",
        "src/data/__init__.py": "from .StandInDataset import get_split_dataset\n",
        "src/data/StandInDataset.py": "def get_split_dataset(*args, **kwargs):\n    pass\n",
        "src/util/util.py": "".join(f"def {n}(*args, **kwargs):\n    pass\n\n\n"
                                    for n in ("cmap", "quat_to_rot", "get_image_to_tensor_balanced", "gen_rays")),
    }
    for rel, text in files.items():
        os.makedirs(os.path.dirname(os.path.join(root, rel)), exist_ok=True)
        with open(os.path.join(root, rel), "w") as f:
            f.write(text)
    return root


def test_names_resolve_to_this_package_and_pass_through_the_rest(tmp_path):
    ref = os.path.realpath(_stand_in_reference(str(tmp_path / "reference")))
    overlay = du.install_ref.make_overlay(str(tmp_path / "overlay"), ref_root=ref)
    probe = (
        "import sys, os; sys.path.insert(0, os.path.join(%r, 'src'))\n"
        "import util, render, model, data\n"
        "from model import make_model, loss\n"
        "from data import get_split_dataset\n"
        "from dotmap import DotMap\n"
        "print('NERF', render.nerf.__file__)\n"
        "print('MODELS', model.models.__file__)\n"
        "print('LOSS', loss.__file__)\n"
        "print('DATA', get_split_dataset.__code__.co_filename)\n"
        "print('CMAP', util.cmap.__code__.co_filename)\n"
        "print('QUAT', util.quat_to_rot.__code__.co_filename)\n"
        "print('TOTENSOR', util.get_image_to_tensor_balanced.__code__.co_filename)\n"
        "print('GENRAYS', util.gen_rays.__code__.co_filename)\n"
    ) % overlay
    env = dict(os.environ, PIXELNERF_REF=ref)
    r = subprocess.run([sys.executable, "-c", probe], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    where = dict(line.split(" ", 1) for line in r.stdout.strip().splitlines() if " " in line)
    ours = os.path.join(overlay, "src")
    assert where["NERF"].startswith(ours) and where["MODELS"].startswith(ours) and where["GENRAYS"].startswith(ours)
    for k in ("LOSS", "DATA", "CMAP", "QUAT", "TOTENSOR"):
        assert os.path.realpath(where[k]).startswith(ref), (k, where[k])


def test_pass_through_fails_by_name_without_a_reference(tmp_path):
    """No checkout -> the hot-path classes still import; out-of-scope names raise, naming the missing reference."""
    src = os.path.join(du.ROOT, "pixel-nerf_b200", "src")
    probe = (
        "import sys; sys.path.insert(0, %r)\n"
        "import _pnr_refpath\n"
        "_pnr_refpath.candidates = lambda: []\n"
        "from model import make_model\n"
        "from render import NeRFRenderer\n"
        "import util\n"
        "try:\n    util.cmap\n    raise SystemExit('cmap resolved')\nexcept AttributeError as e:\n    assert 'reference' in str(e)\n"
        "try:\n    import data\n    raise SystemExit('data resolved')\nexcept ImportError as e:\n    assert 'reference' in str(e)\n"
    ) % src
    r = subprocess.run([sys.executable, "-c", probe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-500:]
