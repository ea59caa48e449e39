"""Import the UNMODIFIED reference model from a checkout of the original OnePose++ repository
(REFERENCE_ROOT below; the environment variable OPP_REFERENCE_ROOT points elsewhere) — TEST
INFRASTRUCTURE ONLY (used to pin oracle/oracle.py and to generate tests/golden/).

The reference needs three packages that are not in this image; each gets a tiny stand-in that
restates only what the hot path calls (SURVEY.md App. B):
  * timm.models.registry.register_model   — identity decorator (backbone/resnet.py:7,345,357)
  * kornia.utils.grid.create_meshgrid, kornia.geometry.subpix.dsnt.spatial_expectation2d
    (utils/fine_matching.py:7-8,86-87) — restated from kornia 0.4.1's published definitions
  * src.utils.profiler.PassThroughProfiler (pytorch_lightning dependency)
The original sources are not part of this repository: nothing under tests -m gpu, smoke() or
bench.py may import this module.
"""
import copy
import os
import sys
import types
from contextlib import contextmanager

import torch

# where the environment that builds and checks this project keeps the original checkout
REFERENCE_ROOT = os.environ.get("OPP_REFERENCE_ROOT") or "/root/reference"


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "models", "OnePosePlus"))


def _module(name):
    m = types.ModuleType(name)
    sys.modules[name] = m
    return m


def install():
    if "timm.models.registry" not in sys.modules:
        timm = _module("timm")
        timm.models = _module("timm.models")
        reg = _module("timm.models.registry")
        reg.register_model = lambda f: f
        timm.models.registry = reg
    if "kornia" not in sys.modules:
        kornia = _module("kornia")
        kornia.utils = _module("kornia.utils")
        grid = _module("kornia.utils.grid")

        def create_meshgrid(height, width, normalized_coordinates=True, device=None):
            xs = torch.linspace(0, width - 1, width, device=device)
            ys = torch.linspace(0, height - 1, height, device=device)
            if normalized_coordinates:
                xs = (xs / (width - 1) - 0.5) * 2
                ys = (ys / (height - 1) - 0.5) * 2
            base = torch.stack(torch.meshgrid(xs, ys, indexing="ij"), -1)  # [W, H, 2]
            return base.permute(1, 0, 2).unsqueeze(0)  # [1, H, W, 2], last = (x, y)

        grid.create_meshgrid = create_meshgrid
        kornia.utils.grid = grid
        kornia.geometry = _module("kornia.geometry")
        kornia.geometry.subpix = _module("kornia.geometry.subpix")
        dsnt = _module("kornia.geometry.subpix.dsnt")

        def spatial_expectation2d(inp, normalized_coordinates=True):
            b, n, h, w = inp.shape
            g = create_meshgrid(h, w, normalized_coordinates, inp.device).to(inp.dtype)
            px = g[..., 0].reshape(-1)
            py = g[..., 1].reshape(-1)
            flat = inp.reshape(b, n, -1)
            ex = (flat * px).sum(-1, keepdim=True)
            ey = (flat * py).sum(-1, keepdim=True)
            return torch.cat([ex, ey], -1)

        dsnt.spatial_expectation2d = spatial_expectation2d
        kornia.geometry.subpix.dsnt = dsnt
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import src  # noqa: F401  (reference package)
    import src.utils  # noqa: F401
    if "src.utils.profiler" not in sys.modules:
        prof = _module("src.utils.profiler")

        class PassThroughProfiler:
            @contextmanager
            def record_function(self, name):
                yield name

        prof.PassThroughProfiler = PassThroughProfiler


def build_reference_loftr(state_dict, config, enable_fine_matching=True):
    """Instantiate the reference LoFTR_for_OnePose_Plus (src/KeypointFreeSfM/loftr_for_sfm/loftr.py;
    its modules come from submodules/LoFTR/src) and load `state_dict` strictly.  `yacs` is absent
    from this image: a dict-with-attributes stand-in is enough for the two config modules."""
    install()
    if "yacs" not in sys.modules:
        yacs = _module("yacs")
        ycfg = _module("yacs.config")

        class CfgNode(dict):
            def __getattr__(self, k):
                try:
                    return self[k]
                except KeyError as e:
                    raise AttributeError(k) from e

            def __setattr__(self, k, v):
                self[k] = v

        ycfg.CfgNode = CfgNode
        yacs.config = ycfg
    lsrc = os.path.join(REFERENCE_ROOT, "submodules", "LoFTR", "src")
    if lsrc not in sys.path:
        sys.path.insert(0, lsrc)
    # the package __init__ files pull in ray / hydra: register bare package objects and import the
    # one module file (loftr.py) underneath them
    import importlib
    for name in ("src.KeypointFreeSfM", "src.KeypointFreeSfM.loftr_for_sfm", "src.KeypointFreeSfM.loftr_for_sfm.utils"):
        if name not in sys.modules:
            pkg = _module(name)
            pkg.__path__ = [os.path.join(REFERENCE_ROOT, *name.split("."))]
    LoFTR_for_OnePose_Plus = importlib.import_module("src.KeypointFreeSfM.loftr_for_sfm.loftr").LoFTR_for_OnePose_Plus
    model = LoFTR_for_OnePose_Plus(copy.deepcopy(config), enable_fine_matching=enable_fine_matching)
    model.load_state_dict(state_dict, strict=True)
    return model.eval()


def build_reference_model(state_dict, config):
    """Instantiate the reference OnePosePlus_model and load `state_dict` with strict=True — which
    also proves that our checkpoint layout is the reference's."""
    install()
    from src.models.OnePosePlus.OnePosePlusModel import OnePosePlus_model  # type: ignore

    model = OnePosePlus_model(copy.deepcopy(config))
    model.load_state_dict(state_dict, strict=True)
    return model.eval()
