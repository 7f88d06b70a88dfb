"""Where the reference checkout lives, for the pass-through of everything that is OUT of this package's scope
(SURVEY.md section 2: `data/*`, `model/loss.py`, colour maps / quaternions / image transforms in `util/util.py`).

This package replaces the render hot path only.  The reference's callers (`train/train.py:13-16`,
`eval/gen_video.py:11-16`) also import `data.get_split_dataset`, `model.loss`, `util.cmap`, ... from the same `src/`
directory; those names resolve to the reference's own, unmodified files, located through

    $PIXELNERF_REF  ->  <repo>/oracle/_ref (installed there by build())        (first that has a `src/` directory)

Nothing of the reference is copied into this package; without a reference checkout those names raise ImportError /
AttributeError naming this module, and the hot-path classes still work.
"""
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(os.path.dirname(_HERE))


def candidates():
    env = os.environ.get("PIXELNERF_REF")
    out = [env] if env else []
    out.append(os.path.join(_REPO, "oracle", "_ref"))
    return out


def ref_root():
    """Root of the reference checkout (the directory that holds `src/`), or None."""
    for root in candidates():
        if root and os.path.isdir(os.path.join(root, "src", "render")):
            src = os.path.realpath(os.path.join(root, "src"))
            if src != os.path.realpath(_HERE):       # never resolve to this package itself (overlay installs)
                return root
    return None


def ref_src(*parts):
    """Path below the reference's `src/`, or None when there is no reference checkout."""
    root = ref_root()
    return os.path.join(root, "src", *parts) if root else None


def need(what):
    raise ImportError(f"{what} is outside the render hot path and is passed through to the reference's own file, but no "
                      f"reference checkout was found (tried {candidates()}; set PIXELNERF_REF)")
