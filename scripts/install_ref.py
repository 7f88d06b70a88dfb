#!/usr/bin/env python
"""Install the UNMODIFIED reference (sxyu/pixel-nerf) where this package finds it, and build the "overlay" tree that
lets the reference's own scripts run against this package.

  python scripts/install_ref.py                 # $PIXELNERF_REF or /root/reference -> oracle/_ref/ (oracle/install_ref.py)
  python scripts/install_ref.py --overlay DIR   # DIR/{eval,train,conf,expconf.conf} -> the reference's, DIR/src -> ours

`oracle/_ref/` is git-ignored (the reference is not product source and is never committed); `build()` fills it when a
reference checkout is present.  It is (a) the timing arm `bench.py --impl reference` / `--impl reference-gpu` (the
reference's own code, through its own public API) and (b) the pass-through target of `_pnr_refpath` for everything
outside the hot path (`data`, `model.loss`, ...).

Overlay: the reference's scripts start with `sys.path.insert(0, <dir of script>/../src)` (eval/gen_video.py:4-6,
train/train.py:7-9), which defeats PYTHONPATH.  The one supported drop-in install is therefore a directory that looks
like the reference checkout but whose `src/` is this package's `pixel-nerf_b200/src` -- symlinks only:

    DIR/eval, DIR/train, DIR/conf*, DIR/expconf.conf*  ->  the reference's      (* conf from this package when
    DIR/src                                            ->  pixel-nerf_b200/src     --our-conf is given)

and `python DIR/eval/gen_video.py ...` / `python DIR/train/train.py ...` run the UNMODIFIED scripts on the fused path.
"""
import argparse
import importlib.util
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle_install():
    spec = importlib.util.spec_from_file_location("pnr_oracle_install_ref", os.path.join(REPO, "oracle", "install_ref.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def find_reference():
    """$PIXELNERF_REF, else the copy in oracle/_ref; None if neither holds a reference checkout."""
    for root in (os.environ.get("PIXELNERF_REF"), os.path.join(REPO, "oracle", "_ref")):
        if root and os.path.isdir(os.path.join(root, "src", "render")):
            return root
    return None


def make_overlay(dest, ref_root=None, our_conf=False):
    """Symlink tree described in the module docstring; returns dest."""
    ref_root = ref_root or find_reference()
    if ref_root is None:
        raise RuntimeError("no reference checkout found (set PIXELNERF_REF or run scripts/install_ref.py)")
    os.makedirs(dest, exist_ok=True)
    pkg = os.path.join(REPO, "pixel-nerf_b200")
    links = {"src": os.path.join(pkg, "src"), "eval": os.path.join(ref_root, "eval"),
             "train": os.path.join(ref_root, "train"),
             "conf": os.path.join(pkg if our_conf else ref_root, "conf"),
             "expconf.conf": os.path.join(pkg if our_conf else ref_root, "expconf.conf")}
    for name, target in links.items():
        p = os.path.join(dest, name)
        if os.path.islink(p):
            os.unlink(p)
        elif os.path.exists(p):
            raise RuntimeError(f"{p} exists and is not a symlink")
        os.symlink(os.path.abspath(target), p)
    return dest


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--dest", default=os.path.join(REPO, "oracle", "_ref"))
    ap.add_argument("--overlay", default=None, help="also (or only, if the reference is installed) build an overlay tree")
    ap.add_argument("--our-conf", action="store_true", help="overlay uses this package's conf/ instead of the reference's")
    a = ap.parse_args()
    if a.overlay is None:
        dest = _oracle_install().install(a.dest)
        if dest is None:
            raise SystemExit("no reference checkout found (set PIXELNERF_REF)")
        print("installed the reference in", dest)
    else:
        if find_reference() is None:
            raise SystemExit("no reference checkout found")
        print("overlay at", make_overlay(a.overlay, our_conf=a.our_conf))
    sys.exit(0)
