"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported through
oracle/ref_shims.py from the checkout at ref_shims.REFERENCE_ROOT) on small planted workloads:

    python -m oracle.make_golden

Inputs are quantised so they can be stored exactly and compactly (image: uint8/255, descriptors:
fp16-representable, keypoints fp32); the weights are regenerated from their seed
(oracle.workload.synthetic_state_dict).  Outputs stored: everything the reference writes into
`data` that callers consume, plus sampled intermediate tensors captured with forward hooks so the
oracle is pinned stage by stage.
"""
import os
import sys

import numpy as np
import torch

from . import oracle, ref_shims, workload

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

SEED1 = int(os.environ.get("OPP_GOLDEN_SEED1", "11"))
CASES = {
    # name: (h, w, n_points, n_planted, batch, with_scale, distinct_banks, seed)
    "planted_128x160_n400": (128, 160, 400, 200, 1, True, False, SEED1),
    "planted_96x128_n300_b2": (96, 128, 300, 110, 2, False, True, 2),
}
WEIGHT_SEED = 0


def sample_idx(numel, k=256, seed=123):
    g = torch.Generator().manual_seed(seed + numel % 1000)
    return torch.randint(0, numel, (min(k, numel),), generator=g)


def build_inputs(sd, case):
    h, w, n, n_pl, batch, with_scale, distinct, seed = CASES[case]
    data, meta = workload.planted_workload(sd, h, w, n, n_pl, batch=batch, seed=seed,
                                           with_scale=with_scale)
    img8 = (data["query_image"] * 255).round().clamp(0, 255).to(torch.uint8)
    data["query_image"] = img8.float() / 255
    for k in ("descriptors3d_db", "descriptors3d_coarse_db"):
        data[k] = data[k].half().float()
    if distinct and batch > 1:
        # different clouds per batch element: exercises normalize_3d_keypoints' use of kpts[0]
        g = torch.Generator().manual_seed(seed + 77)
        data["keypoints3d"] = data["keypoints3d"].clone()
        data["keypoints3d"][1] = (torch.rand(n, 3, generator=g) - 0.5) * 1.7 + 0.1
    return data, img8


@torch.no_grad()
def main():
    assert ref_shims.available(), f"no checkout of the original OnePose++ at {ref_shims.REFERENCE_ROOT} (set OPP_REFERENCE_ROOT)"
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    sd = workload.synthetic_state_dict(WEIGHT_SEED)
    model = ref_shims.build_reference_model(sd, oracle.DEFAULT_CONFIG)
    for case in CASES:
        data, img8 = build_inputs(sd, case)
        captured = {}

        def hook(name):
            def fn(mod, inp, out):
                captured[name] = out
            return fn

        handles = [model.backbone.register_forward_hook(hook("backbone")),
                   model.loftr_coarse.register_forward_hook(hook("loftr_coarse")),
                   model.loftr_fine.register_forward_hook(hook("loftr_fine"))]
        for i, layer in enumerate(model.loftr_coarse.layers):
            handles.append(layer.register_forward_hook(hook(f"coarse_layer{i}")))
        d = {k: v.clone() for k, v in data.items()}
        model(d)
        for hnd in handles:
            hnd.remove()
        out = {
            "image_u8": img8.numpy(),
            "keypoints3d": data["keypoints3d"].numpy(),
            "descriptors3d_db_f16": data["descriptors3d_db"].half().numpy(),
            "descriptors3d_coarse_db_f16": data["descriptors3d_coarse_db"].half().numpy(),
        }
        if "query_image_scale" in data:
            out["query_image_scale"] = data["query_image_scale"].numpy()
        for k in ("b_ids", "i_ids", "j_ids", "m_bids", "mconf", "mkpts_3d_db", "mkpts_query_c",
                  "expec_f", "mkpts_query_f"):
            out[k] = d[k].numpy()
        conf = d["conf_matrix"]
        out["conf_rowmax"] = conf.max(2).values.numpy()
        out["conf_colmax"] = conf.max(1).values.numpy()
        idx = sample_idx(conf.numel(), 2048)
        out["conf_sample_idx"] = idx.numpy()
        out["conf_sample"] = conf.flatten()[idx].numpy()
        fc, ff = captured["backbone"]
        for name, t in (("feat_c", fc), ("feat_f", ff), ("tok3d_out", captured["loftr_coarse"][0]),
                        ("tok2d_out", captured["loftr_coarse"][1])):
            idx = sample_idx(t.numel(), 1024)
            out[name + "_idx"] = idx.numpy()
            out[name] = t.flatten()[idx].numpy()
            out[name + "_absmean"] = np.float32(t.abs().mean().item())
        if "loftr_fine" in captured:
            for name, t in (("fine3d_out", captured["loftr_fine"][0]), ("fine2d_out", captured["loftr_fine"][1])):
                idx = sample_idx(t.numel(), 1024)
                out[name + "_idx"] = idx.numpy()
                out[name] = t.flatten()[idx].numpy()
        # decision margins, recorded so tests can assert the fixture is well conditioned
        rowmax = conf.max(2).values
        out["min_thr_margin"] = np.float32((rowmax - 0.1).abs().min().item())
        top2r = conf.topk(2, dim=2).values
        top2c = conf.topk(2, dim=1).values
        b_, i_, j_ = d["b_ids"], d["i_ids"], d["j_ids"]
        out["min_row_margin"] = np.float32((top2r[b_, i_, 0] - top2r[b_, i_, 1]).min().item())
        out["min_col_margin"] = np.float32((top2c[b_, 0, j_] - top2c[b_, 1, j_]).min().item())
        path = os.path.join(GOLDEN_DIR, case + ".npz")
        np.savez_compressed(path, **out)
        print(f"{case}: M={len(d['b_ids'])} mconf[{d['mconf'].min().item():.3f},{d['mconf'].max().item():.3f}] "
              f"thr margin {out['min_thr_margin']:.4f} row {out['min_row_margin']:.4f} col {out['min_col_margin']:.4f}"
              f" -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


if __name__ == "__main__":
    sys.exit(main())
