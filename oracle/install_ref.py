"""
ORACLE TOOLING -- the recipe `__graft_entry__.build()` runs: installs the UNMODIFIED reference (sxyu/pixel-nerf) into
the git-ignored `oracle/_ref/`.

The reference is pure Python (no setup.py / pyproject), so "install" = copy the five trees its scripts use; only files
are copied, nothing is edited.  The source is $PIXELNERF_REF, else /root/reference; without either, nothing is
installed.  `oracle/_ref/` is then what the reference timing arms of bench.py, the drop-in tests (the reference's own
scripts over this package, `scripts/install_ref.py --overlay`) and the pass-through of out-of-scope names
(`_pnr_refpath`) use.  The tests that compare numbers with the reference do not need it: they read tests/golden/.
"""
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
SOURCES = (os.environ.get("PIXELNERF_REF"), "/root/reference")
TREES = ["src", "conf", "eval", "train", "expconf.conf"]


def install(dest=DEST):
    """Copies the first readable reference checkout to dest; returns dest, or None when there is neither a checkout nor
    an earlier copy in dest."""
    src_root = next((s for s in SOURCES if s and os.path.isdir(os.path.join(s, "src", "render"))), None)
    if src_root is None:
        return dest if os.path.isdir(os.path.join(dest, "src", "render")) else None
    if os.path.realpath(src_root) == os.path.realpath(dest):
        return dest
    os.makedirs(dest, exist_ok=True)
    for name in TREES:
        s, d = os.path.join(src_root, name), os.path.join(dest, name)
        if os.path.isdir(s):
            if os.path.exists(d):
                shutil.rmtree(d)
            shutil.copytree(s, d, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        else:
            shutil.copy2(s, d)
    return dest


if __name__ == "__main__":
    print(install() or "no reference checkout found (set PIXELNERF_REF)")
