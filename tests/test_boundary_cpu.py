"""Boundary proof (CPU): the reference's OWN code that constructs the matcher runs unchanged when
the two import lines of INTEGRATION.md §1 point at this package.  The first two tests execute the
original project's source files and run only where a checkout of it is readable
(oracle/ref_shims.REFERENCE_ROOT); the LoFTR layout test compares with the reference's
recorded state-dict layout (oracle/make_reference_runs.py).

The reference modules cannot be imported whole here (ray, pytorch_lightning, hydra ... are absent),
so the relevant definitions are taken from the reference source files with `ast` and executed in a
namespace where `OnePosePlus_model` is the drop-in class:
  * `build_model()`  — src/inference/inference_OnePosePlus.py:28-38 (strict=True load, .eval())
  * `PL_OnePosePlus.__init__` — src/lightning_model/OnePosePlus_lightning_model.py:20-49
    (matcher slot + full-checkpoint load with the `matcher.` prefix)
and the object is pickled as Ray does when it ships the model to its workers (:86-94)."""
import ast
import copy
import os
import pickle

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import oracle, ref_shims, workload
from oracle.make_reference_runs import sampled
from onepose_plus_plus_b200 import OnePosePlus_model
from tests import golden_io

needs_reference_sources = pytest.mark.skipif(
    not ref_shims.available(), reason="executes the original OnePose++ sources; no checkout at ref_shims.REFERENCE_ROOT")


def _extract(path, name):
    src = open(os.path.join(ref_shims.REFERENCE_ROOT, path)).read()
    for node in ast.parse(src).body:
        if isinstance(node, (ast.FunctionDef, ast.ClassDef)) and node.name == name:
            return ast.get_source_segment(src, node)
    raise KeyError(name)


def _pl_checkpoint(tmp_path):
    sd = workload.synthetic_state_dict(0)
    path = str(tmp_path / "pl.ckpt")
    torch.save({"state_dict": {"matcher." + k: v for k, v in sd.items()}}, path)   # PL checkpoint layout
    return sd, path


@needs_reference_sources
def test_reference_build_model_runs_on_the_drop_in(tmp_path):
    from loguru import logger
    sd, ckpt = _pl_checkpoint(tmp_path)
    ns = {"OnePosePlus_model": OnePosePlus_model, "torch": torch, "logger": logger}
    exec(_extract("src/inference/inference_OnePosePlus.py", "build_model"), ns)   # the reference's code, verbatim
    model = ns["build_model"](copy.deepcopy(oracle.DEFAULT_CONFIG), ckpt)
    assert isinstance(model, OnePosePlus_model) and not model.training
    got = model.state_dict()
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    # Ray serialises the module object for its workers (inference_OnePosePlus.py:86-94)
    clone = pickle.loads(pickle.dumps(model))
    assert not clone.training and all(torch.equal(clone.state_dict()[k], sd[k]) for k in sd)
    assert clone._plan is None and clone._ws == {}          # device caches never travel
    # the worker then does match_model.cuda(); match_model(data): without a GPU that must fail loudly
    with pytest.raises(RuntimeError, match="no CPU path"):
        clone(workload.random_workload(64, 64, 50))


@needs_reference_sources
def test_reference_lightning_module_builds_around_the_drop_in(tmp_path):
    from loguru import logger
    sd, ckpt = _pl_checkpoint(tmp_path)

    class LightningModule(nn.Module):                       # the two pl features __init__ uses
        def save_hyperparameters(self):
            pass

    class Loss(nn.Module):                                  # losses.py:7-16 holds no parameters
        def __init__(self, config):
            super().__init__()
            self.config = config

    pl = type("pl", (), {"LightningModule": LightningModule})
    ns = {"pl": pl, "OnePosePlus_model": OnePosePlus_model, "Loss": Loss, "torch": torch, "logger": logger}
    src = _extract("src/lightning_model/OnePosePlus_lightning_model.py", "PL_OnePosePlus")
    exec(src, ns)
    PL = ns["PL_OnePosePlus"]
    hparams = {"OnePosePlus": copy.deepcopy(oracle.DEFAULT_CONFIG), "loss": {},
               "trainer": {"n_val_pairs_to_plot": 4, "world_size": 2}, "pretrained_ckpt": ckpt}
    PL.hparams = property(lambda self: hparams)            # what save_hyperparameters() provides
    module = PL()
    assert isinstance(module.matcher, OnePosePlus_model) and module.n_vals_plot == 2
    got = module.matcher.state_dict()
    assert all(torch.equal(got[k], sd[k]) for k in sd)      # the strict full-checkpoint load went through
    # the hooks Lightning drives on the matcher
    module.eval()
    assert not module.matcher.training
    assert sum(p.numel() for p in module.parameters()) == 10_226_480


def test_loftr_drop_in_has_the_reference_layout():
    """LoFTR_for_OnePose_Plus (SURVEY §8 f3): same ctor, same state-dict keys / shapes as the reference
    class built from submodules/LoFTR/src/loftr (so a strict load works both ways), the same
    non-persistent pos-enc buffer (recorded values: sin / cos may differ in the last bit between
    machines)."""
    from oracle import loftr_oracle
    from onepose_plus_plus_b200 import LoFTR_for_OnePose_Plus
    z = golden_io.reference_run("loftr_layout")
    sd = workload.synthetic_loftr_state_dict(0)
    ours = LoFTR_for_OnePose_Plus(dict(loftr_oracle.DEFAULT_CONFIG), enable_fine_matching=True)
    os_ = ours.state_dict()
    keys = z["keys"].tolist()
    assert sorted(os_) == keys and sorted(sd) == keys
    for k, nd, shape in zip(keys, z["ndim"], z["shapes"]):
        assert tuple(os_[k].shape) == tuple(shape[:nd]), k
    ours.load_state_dict(sd, strict=True)
    pe = ours.pos_encoding.pe
    assert tuple(pe.shape) == tuple(z["pe_shape"]) and "pos_encoding.pe" not in os_
    assert np.allclose(z["pe"], sampled(pe, len(z["pe"])).numpy(), rtol=0, atol=1e-6)
    clone = pickle.loads(pickle.dumps(ours.eval()))
    assert all(torch.equal(clone.state_dict()[k], sd[k]) for k in sd)
    with pytest.raises(RuntimeError, match="no CPU path"):
        clone({"image0": torch.rand(1, 1, 64, 64), "image1": torch.rand(1, 1, 64, 64)})
