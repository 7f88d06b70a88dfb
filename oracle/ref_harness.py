"""
ORACLE TOOLING -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Imports the UNMODIFIED reference (sxyu/pixel-nerf) from $PIXELNERF_REF/src, else from the
copy build() installs in oracle/_ref/src, on CPU so that `make_golden.py` can generate golden vectors and the
restatement in `pnr_oracle.py` can be validated against the real thing.  The reference
needs two pure-Python packages that are not installed here (`dotmap`, `pyhocon`); tiny
stand-ins are injected into sys.modules ONLY for that import -- no reference source is
copied or changed.  The tests do not use it: they compare with golden data it helped write.
bench.py's reference timing arms do, when oracle/_ref is installed.
"""
import os
import sys
import types

import torch

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_ref():
    """$PIXELNERF_REF, else oracle/_ref (oracle/install_ref.py, run by build())."""
    installed = os.path.join(_REPO, "oracle", "_ref")
    for root in (os.environ.get("PIXELNERF_REF"), installed):
        if root and os.path.isdir(os.path.join(root, "src")):
            return root
    return installed


REF_ROOT = _find_ref()


class _DotMap(dict):
    """Minimal dotmap.DotMap stand-in: attribute access, auto-vivify, toDict()."""

    def __init__(self, *a, **kw):
        super().__init__()
        for k, v in dict(*a, **kw).items():
            self[k] = v

    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        if k not in self:
            self[k] = _DotMap()
        return self[k]

    def __setattr__(self, k, v):
        self[k] = v

    def toDict(self):
        return {k: (v.toDict() if isinstance(v, _DotMap) else v) for k, v in self.items()}


class DictConf(dict):
    """pyhocon.ConfigTree look-alike over a nested dict (get_int/get_float/...)."""

    def _get(self, key, default, conv):
        cur = self
        for part in key.split("."):
            if not isinstance(cur, dict) or part not in cur:
                if default is _MISSING:
                    raise KeyError(key)
                return default
            cur = dict.__getitem__(cur, part)
        return conv(cur)

    def __getitem__(self, key):
        v = self._get(key, _MISSING, lambda x: x)
        return DictConf(v) if isinstance(v, dict) and not isinstance(v, DictConf) else v

    def get_int(self, k, d=None):
        return self._get(k, d if d is not None else _MISSING, int)

    def get_float(self, k, d=None):
        return self._get(k, d if d is not None else _MISSING, float)

    def get_bool(self, k, d=None):
        return self._get(k, d if d is not None else _MISSING,
                         lambda v: v if isinstance(v, bool) else str(v).lower() in ("true", "1", "yes"))

    def get_string(self, k, d=None):
        return self._get(k, d if d is not None else _MISSING, str)

    def get_list(self, k, d=None):
        if d is None:
            try:
                return self._get(k, _MISSING, list)
            except KeyError:
                return None
        return self._get(k, d, list)


_MISSING = object()


def import_reference():
    """Returns (model_pkg, render_pkg, util_pkg) of the reference."""
    src = os.path.join(REF_ROOT, "src")
    if not os.path.isdir(src):
        raise RuntimeError(f"reference not found at {REF_ROOT}")
    if "dotmap" not in sys.modules:
        try:
            import dotmap  # noqa: F401
        except ImportError:
            m = types.ModuleType("dotmap")
            m.DotMap = _DotMap
            sys.modules["dotmap"] = m
    if "pyhocon" not in sys.modules:
        try:
            import pyhocon  # noqa: F401
        except ImportError:
            m = types.ModuleType("pyhocon")

            class ConfigFactory:  # only referenced by util/args.py:parse_args, unused here
                @staticmethod
                def parse_file(path):
                    raise RuntimeError("pyhocon stub")

            m.ConfigFactory = ConfigFactory
            sys.modules["pyhocon"] = m
    for name in ("model", "render", "util"):
        if name in sys.modules and not getattr(sys.modules[name], "__file__", "").startswith(src):
            raise RuntimeError(f"module '{name}' already imported from elsewhere; "
                               "the reference must be imported in its own process")
    if src not in sys.path:
        sys.path.insert(0, src)
    import model
    import render
    import util
    return model, render, util


def model_conf(d_hidden, use_first_pool=True):
    """conf/default_mv.conf as a dict (model subtree), pretrained off (no network)."""
    mlp = dict(type="resnet", n_blocks=5, d_hidden=d_hidden, combine_layer=3, combine_type="average")
    return DictConf(dict(
        use_encoder=True, use_global_encoder=False, use_xyz=True, canon_xyz=False, use_code=True,
        code=dict(num_freqs=6, freq_factor=1.5, include_input=True),
        use_viewdirs=True, use_code_viewdirs=False,
        mlp_coarse=dict(mlp), mlp_fine=dict(mlp),
        encoder=dict(backbone="resnet34", pretrained=False, num_layers=4, use_first_pool=use_first_pool),
    ))


def build_reference(d_hidden, w_coarse, w_fine, n_coarse, n_fine, n_fine_depth, depth_std=0.01,
                    white_bkgd=True, eval_batch_size=50000, use_first_pool=True):
    """Reference PixelNeRFNet (+weights) and NeRFRenderer."""
    model, render, _ = import_reference()
    net = model.make_model(model_conf(d_hidden, use_first_pool))
    net.mlp_coarse.load_state_dict(w_coarse)
    if w_fine is not None:
        net.mlp_fine.load_state_dict(w_fine)
    else:
        net.mlp_fine = None
    net.eval()
    renderer = render.NeRFRenderer(n_coarse=n_coarse, n_fine=n_fine, n_fine_depth=n_fine_depth,
                                   depth_std=depth_std, eval_batch_size=eval_batch_size,
                                   white_bkgd=white_bkgd)
    renderer.eval()
    return net, renderer


def set_scene(net, latent, poses_c2w, focal, c, W, H):
    """Run the reference's own encode() bookkeeping (models.py:89-144) but with a given
    latent instead of the conv trunk's: the trunk is replaced by a stub for the call."""
    SB = poses_c2w.shape[0] if poses_c2w.dim() == 4 else 1
    NS = poses_c2w.shape[-3]
    images = torch.zeros(*(poses_c2w.shape[:-2]), 3, H, W)

    enc = net.encoder
    orig_forward = enc.forward

    def stub(x):
        enc.latent = latent
        enc.latent_scaling[0] = latent.shape[-1]
        enc.latent_scaling[1] = latent.shape[-2]
        enc.latent_scaling = enc.latent_scaling / (enc.latent_scaling - 1) * 2.0
        return latent

    enc.forward = stub
    try:
        net.encode(images, poses_c2w, focal, c=c)
    finally:
        enc.forward = orig_forward
    return SB, NS


def run_reference_render(net, renderer, rays, seed):
    """renderer(net, rays, want_weights=True) with the global RNG seeded; also captures the
    z samples handed to composite() (nerf.py:163) by wrapping the bound method."""
    captured = []
    orig = renderer.composite

    def spy(model, rays_, z_samp, coarse=True, sb=0):
        captured.append(z_samp.detach().clone())
        return orig(model, rays_, z_samp, coarse=coarse, sb=sb)

    renderer.composite = spy
    try:
        torch.manual_seed(seed)
        with torch.no_grad():
            out = renderer(net, rays, want_weights=True)
    finally:
        renderer.composite = orig
    return out, captured
