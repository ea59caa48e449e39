"""Rebuild the inputs stored in tests/golden/*.npz (see oracle/make_golden.py), and read the
reference's recorded results in tests/golden/reference_runs/ (see oracle/make_reference_runs.py)."""
import glob
import os

import numpy as np
import torch

from oracle.make_reference_runs import sampled

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def reference_run(name):
    return np.load(os.path.join(GOLDEN_DIR, "reference_runs", name + ".npz"))


def check_inputs(z, tensors, prefix="input_"):
    """The floating-point inputs rebuilt from their seeds are the ones the reference was run on.
    Planted descriptors come out of CPU convolutions whose rounding differs between machines, so
    the bound is relative to the tensor's scale: it catches a changed generator, not rounding."""
    for k, v in tensors.items():
        if v.is_floating_point():
            ref = z[prefix + k]
            err = np.abs(ref - sampled(v, len(ref)).numpy()).max()
            assert err <= 1e-4 * np.abs(ref).max(), \
                f"{k} differs from the input of the recorded reference run by {err:.3g}"


def check_conf(z, conf, atol, rtol=1e-5):
    """conf_matrix against the recorded one: every row and column maximum and a fixed sample."""
    conf = conf.detach()
    assert z["conf_rowmax"].shape == conf.shape[:2] and z["conf_colmax"].shape == (conf.shape[0], conf.shape[2])
    assert np.allclose(z["conf_rowmax"], conf.max(2).values.numpy(), rtol=rtol, atol=atol), "conf_matrix row maxima"
    assert np.allclose(z["conf_colmax"], conf.max(1).values.numpy(), rtol=rtol, atol=atol), "conf_matrix column maxima"
    ref = z["conf_sample"]
    assert np.allclose(ref, sampled(conf, len(ref)).numpy(), rtol=rtol, atol=atol), "conf_matrix sample"


def cases():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def load(case):
    z = np.load(os.path.join(GOLDEN_DIR, case + ".npz"))
    data = {
        "query_image": torch.from_numpy(z["image_u8"]).float() / 255,
        "keypoints3d": torch.from_numpy(z["keypoints3d"]),
        "descriptors3d_db": torch.from_numpy(z["descriptors3d_db_f16"]).float(),
        "descriptors3d_coarse_db": torch.from_numpy(z["descriptors3d_coarse_db_f16"]).float(),
    }
    if "query_image_scale" in z.files:
        data["query_image_scale"] = torch.from_numpy(z["query_image_scale"])
    return data, z
