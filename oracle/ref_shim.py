"""TEST INFRASTRUCTURE -- not product code.

Loader for the *unmodified* reference (apchenstu/mvsnerf, mounted read-only at
/root/reference in the build container).  It exists for two jobs only:

  1. `tests/golden/make_golden.py` imports the reference through this shim to
     produce the committed golden vectors under tests/golden/.
  2. `tests/golden/make_golden_pins.py` records, the same way, what
     `tests/test_oracle_pins.py` checks the restatement in
     `oracle/mvsnerf_oracle.py` against.

Nothing here travels to the GPU box as a dependency: /root/reference does not
exist there and every caller must guard on `reference_available()`.

The reference cannot be imported as-is in this image (SURVEY.md F8): it imports
`inplace_abn`, `kornia`, `warmup_scheduler`, `configargparse`, none of which are
installed, calls `.cuda()` unconditionally (models.py:37) and `torch.load`s a
CUDA-saved checkpoint without map_location (models.py:624).  The stubs below
supply the *published semantics* of those third-party pieces:

  * inplace_abn.InPlaceABN  -- BatchNorm (train: biased batch statistics,
    eval: running statistics), eps 1e-5, momentum 0.1, affine weight used as
    |gamma|+eps, followed by leaky-ReLU(0.01); a train-mode forward also updates
    running_mean / running_var (unbiased variance) and counts itself in
    num_batches_tracked.  Un-pinned third-party package
    (not vendored, not in the reference's install line) => "parity unpinned"
    for this piece; all gamma in ckpts/mvsnerf-v0.tar are > 0.37 so the
    |gamma|+eps vs gamma variant moves RGB by ~3e-5 (SURVEY.md App. D).
  * kornia.create_meshgrid  -- (1,H,W,2) pixel grid, [...,0]=x, [...,1]=y.

F5 (SURVEY.md): `build_volume_costvar_img` allocates the 41-channel volume with
torch.empty and never writes the pad border of channels 0:3.  We pin that
border to ZERO by swapping torch.empty->torch.zeros while that method runs.
"""
from __future__ import annotations

import contextlib
import importlib
import os
import sys
import types
from types import SimpleNamespace

import torch
import torch.nn.functional as F

REFERENCE_ROOT = os.environ.get("MVSNERF_REFERENCE_ROOT", "/root/reference")
REFERENCE_CKPT = os.path.join(REFERENCE_ROOT, "ckpts", "mvsnerf-v0.tar")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "models.py"))


class _InPlaceABN(torch.nn.modules.batchnorm._BatchNorm):
    """Stand-in for inplace_abn.InPlaceABN (semantics in the module docstring)."""

    def __init__(self, num_features, eps=1e-5, momentum=0.1, affine=True,
                 activation="leaky_relu", activation_param=0.01):
        super().__init__(num_features, eps=eps, momentum=momentum, affine=affine)
        self.activation = activation
        self.activation_param = activation_param

    def _check_input_dim(self, input):  # one class serves 2-D and 3-D convs
        return

    def forward(self, x):
        # the published ABN counts train-mode forwards like nn.BatchNorm does; the shipped checkpoint's
        # num_batches_tracked (181165 = its training iterations) is the evidence that the real package did
        if self.training and self.track_running_stats and self.num_batches_tracked is not None:
            self.num_batches_tracked.add_(1)
        y = F.batch_norm(x, self.running_mean, self.running_var,
                         self.weight.abs() + self.eps, self.bias,
                         self.training, self.momentum, self.eps)
        return F.leaky_relu(y, self.activation_param)


def _create_meshgrid(height, width, normalized_coordinates=True, device=None, dtype=torch.float32):
    xs = torch.linspace(0, width - 1, width, device=device, dtype=dtype)
    ys = torch.linspace(0, height - 1, height, device=device, dtype=dtype)
    if normalized_coordinates:
        xs = (xs / (width - 1) - 0.5) * 2
        ys = (ys / (height - 1) - 0.5) * 2
    gy, gx = torch.meshgrid(ys, xs, indexing="ij")
    return torch.stack([gx, gy], dim=-1).unsqueeze(0)


def _install_stubs():
    if "inplace_abn" not in sys.modules:
        m = types.ModuleType("inplace_abn")
        m.InPlaceABN = _InPlaceABN
        sys.modules["inplace_abn"] = m
    if "kornia" not in sys.modules:
        k = types.ModuleType("kornia")
        ku = types.ModuleType("kornia.utils")
        k.create_meshgrid = _create_meshgrid
        ku.create_meshgrid = _create_meshgrid
        k.utils = ku
        sys.modules["kornia"] = k
        sys.modules["kornia.utils"] = ku
    if "warmup_scheduler" not in sys.modules:
        w = types.ModuleType("warmup_scheduler")
        w.GradualWarmupScheduler = type("GradualWarmupScheduler", (), {})
        sys.modules["warmup_scheduler"] = w
    if "configargparse" not in sys.modules:
        import argparse
        c = types.ModuleType("configargparse")

        class ArgumentParser(argparse.ArgumentParser):
            def add_argument(self, *a, **kw):
                kw.pop("is_config_file", None)
                return super().add_argument(*a, **kw)

        c.ArgumentParser = ArgumentParser
        sys.modules["configargparse"] = c


_REF = None


def load_reference():
    """Import the reference's models/renderer/utils/data.ray_utils; returns a namespace."""
    global _REF
    if _REF is not None:
        return _REF
    if not reference_available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    _install_stubs()
    if not torch.cuda.is_available():
        torch.Tensor.cuda = lambda self, *a, **k: self  # models.py:37
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # the reference's top-level module names are generic ("utils", "models", ...)
    for name in ("utils", "models", "renderer", "data", "data.ray_utils"):
        if name in sys.modules and not getattr(sys.modules[name], "__file__", "").startswith(REFERENCE_ROOT):
            raise RuntimeError(f"module name clash: {name} already imported from elsewhere")
    ref_utils = importlib.import_module("utils")
    ref_renderer = importlib.import_module("renderer")
    ref_models = importlib.import_module("models")
    ref_ray_utils = importlib.import_module("data.ray_utils")
    torch.autograd.set_detect_anomaly(False)  # models.py:2 turns it on globally
    _REF = SimpleNamespace(utils=ref_utils, renderer=ref_renderer, models=ref_models,
                           ray_utils=ref_ray_utils)
    return _REF


@contextlib.contextmanager
def _pinned_empty():
    """F5: make torch.empty return zeros while the cost volume is built."""
    real_empty = torch.empty
    torch.empty = lambda *a, **k: torch.zeros(*a, **k)
    try:
        yield
    finally:
        torch.empty = real_empty


@contextlib.contextmanager
def _cpu_torch_load(device="cpu"):
    real_load = torch.load

    def load(f, *a, **k):
        k.setdefault("map_location", device)
        k.setdefault("weights_only", False)
        return real_load(f, *a, **k)

    torch.load = load
    try:
        yield
    finally:
        torch.load = real_load


def reference_args(**overrides):
    """The attribute set the reference's call sites put on `args` (SURVEY.md App. C.7)."""
    a = dict(multires=10, i_embed=0, pts_dim=3, multires_views=4, dir_dim=3, netdepth=6,
             netwidth=128, feat_dim=20, net_type="v0", N_importance=0, netchunk=1024,
             ckpt=REFERENCE_CKPT, perturb=1.0, N_samples=128, use_viewdirs=True,
             white_bkgd=False, raw_noise_std=0.0, img_downscale=1.0, use_color_volume=False,
             chunk=5120, pad=24, imgScale_test=1.0)
    a.update(overrides)
    return SimpleNamespace(**a)


def build_reference(device="cpu", **arg_overrides):
    """create_nerf_mvs exactly as the notebooks do (renderer_video.ipynb DTU cell)."""
    ref = load_reference()
    args = reference_args(**arg_overrides)
    with _cpu_torch_load(device):
        kw_train, _, _, _ = ref.models.create_nerf_mvs(args, use_mvs=True, dir_embedder=False,
                                                       pts_embedder=True)
    ref.utils.filter_keys(kw_train)
    mvsnet = kw_train.pop("network_mvs")
    mvsnet.train()  # every shipped caller does this (SURVEY.md F2)

    real_build = mvsnet.build_volume_costvar_img

    def pinned_build(*a, **k):
        with _pinned_empty():
            return real_build(*a, **k)

    mvsnet.build_volume_costvar_img = pinned_build
    return SimpleNamespace(ref=ref, args=args, render_kwargs=kw_train, mvsnet=mvsnet)
