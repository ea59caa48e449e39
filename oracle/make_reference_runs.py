"""Record the unmodified reference's results for the tests that compare the oracle with it, as
compact fixtures under tests/golden/reference_runs/ (one .npz per test case):

    python -m oracle.make_reference_runs       (original checkout: oracle/ref_shims.REFERENCE_ROOT)

The inputs are regenerated at test time from their seeds (oracle.workload), so a fixture stores a
sample of each input (the test checks that it still builds what the reference saw) and the
reference's outputs: match lists in full, large tensors (conf_matrix, gradients, the position
encoding) as row / column maxima plus a fixed sample of entries (spread_idx).
"""
import copy
import os
import sys

import numpy as np
import torch

from . import loftr_oracle, oracle, ref_shims, workload

OUT_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                       "reference_runs")

# test id -> (h, w, n_points, n_planted, batch, query mask, coarse attention); seed 5
ORACLE_CASES = {
    "small_b2": (96, 128, 300, 120, 2, False, "linear"),
    "baseline_512_n5000": (512, 512, 5000, 3000, 1, False, "linear"),
    "small_b2_query_mask": (96, 128, 300, 120, 2, True, "linear"),
    "small_b2_full_attention": (96, 128, 300, 120, 2, False, "full"),
}
# test id -> (h, w, batch, with_scale)
LOFTR_CASES = {"b2": (192, 256, 2, False), "b1_scaled": (256, 320, 1, True)}
# parameters whose gradients the training-path test compares
GRAD_PARAMS = ("backbone.conv1.weight", "backbone.layer2.0.bn1.weight", "backbone.layer1_outconv2.3.weight",
               "kpt_3d_pos_encoding.encoder.0.weight", "loftr_coarse.layers.0.q_proj.weight",
               "loftr_coarse.layers.5.mlp.2.weight", "loftr_coarse.layers.3.norm1.bias",
               "loftr_fine.layers.1.merge.weight")


def spread_idx(numel, k):
    """k flat indices spread over a tensor of numel entries (all of them when numel <= k); a fixed
    formula, so fixtures store only the sampled values."""
    if numel <= k:
        return torch.arange(numel)
    return torch.arange(k, dtype=torch.int64) * 2654435761 % numel


def sampled(t, k):
    return t.detach().flatten()[spread_idx(t.numel(), k)].float()


def put_sample(out, name, t, k=512):
    out[name] = sampled(t, k).numpy()


def put_conf(out, conf, name="conf"):
    out[name + "_rowmax"] = conf.max(2).values.numpy()
    out[name + "_colmax"] = conf.max(1).values.numpy()
    put_sample(out, name + "_sample", conf, 1024)


def put_inputs(out, data):
    for k, v in data.items():
        if v.is_floating_point():
            put_sample(out, "input_" + k, v, 64)


def put_matches(out, d, keys):
    for k in keys:
        v = d[k]
        out[k] = v.numpy().astype(np.int32) if v.dtype == torch.int64 else v.numpy()


def train_batch(sd, masked):
    """The training-path test's batch: planted workload + a seeded random ground-truth matrix."""
    data, _ = workload.planted_workload(sd, 96, 128, 300, 120, batch=2, seed=5)
    S = (96 // 8) * (128 // 8)
    g = torch.Generator().manual_seed(3)
    gt = torch.zeros(2, 300, S, dtype=torch.bool)
    gt[torch.randint(0, 2, (90,), generator=g), torch.randint(0, 300, (90,), generator=g),
       torch.randint(0, S, (90,), generator=g)] = True
    data["conf_matrix_gt"] = gt
    if masked:
        data["query_image_mask"] = workload.pad_mask(2, 12, 16)
    return data


def train_config():
    cfg = copy.deepcopy(oracle.DEFAULT_CONFIG)
    cfg["coarse_matching"]["train"]["train_pad_num_gt_min"] = 20      # < 0.3 * B * min(L, S) at this size
    return cfg


def train_loss(d):
    # (the std column is sqrt(clamp(var)): ill-conditioned near 0, left out of the gradient check)
    return (d["conf_matrix"] * d["conf_matrix_gt"]).sum() + d["expec_f"][:, :2].pow(2).sum()


def save(name, out):
    path = os.path.join(OUT_DIR, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def oracle_runs(sd):
    for name, case in ORACLE_CASES.items():
        h, w, n, npl, batch, masked, attention = case
        data, _ = workload.planted_workload(sd, h, w, n, npl, batch=batch, seed=5)
        if masked:
            data["query_image_mask"] = workload.pad_mask(batch, h // 8, w // 8)
        cfg = copy.deepcopy(oracle.DEFAULT_CONFIG)
        cfg["loftr_coarse"]["attention"] = attention
        ref = ref_shims.build_reference_model(sd, cfg)
        d = {k: v.clone() for k, v in data.items()}
        with torch.no_grad():
            ref(d)
        out = {"case": np.array(case[:6], dtype=np.int64), "attention": np.array(attention)}
        put_inputs(out, data)
        put_matches(out, d, ("b_ids", "i_ids", "j_ids", "m_bids", "mconf", "mkpts_3d_db", "mkpts_query_c",
                             "expec_f", "mkpts_query_f"))
        put_conf(out, d["conf_matrix"])
        save("oracle_" + name, out)


def loftr_runs():
    for name, case in LOFTR_CASES.items():
        h, w, batch, with_scale = case
        sd, data = workload.planted_loftr(h, w, batch=batch, with_scale=with_scale)
        ref = ref_shims.build_reference_loftr(sd, dict(loftr_oracle.DEFAULT_CONFIG))
        d = {k: v.clone() for k, v in data.items()}
        with torch.no_grad():
            ref(d)
        out = {"case": np.array(case, dtype=np.int64), "W": np.int64(d["W"])}
        put_inputs(out, data)
        # the planted checkpoint is derived from oracle forwards: pin the two derived tensors too
        for k in ("loftr_coarse.layers.7.norm2.bias", "backbone.layer1_outconv2.3.weight"):
            put_sample(out, "sd_" + k, sd[k], 64)
        put_matches(out, d, ("b_ids", "i_ids", "j_ids", "mkpts0_c", "mkpts1_c", "mconf", "expec_f",
                             "mkpts0_f", "mkpts1_f"))
        put_conf(out, d["conf_matrix"])
        save("loftr_" + name, out)


def loftr_layout():
    sd = workload.synthetic_loftr_state_dict(0)
    ref = ref_shims.build_reference_loftr(sd, dict(loftr_oracle.DEFAULT_CONFIG))
    rs = ref.state_dict()
    keys = sorted(rs)
    out = {"keys": np.array(keys), "ndim": np.array([rs[k].dim() for k in keys], dtype=np.int64),
           "shapes": np.array([list(rs[k].shape) + [0] * (4 - rs[k].dim()) for k in keys], dtype=np.int64),
           "pe_shape": np.array(ref.pos_encoding.pe.shape, dtype=np.int64)}
    put_sample(out, "pe", ref.pos_encoding.pe, 1024)
    save("loftr_layout", out)


def train_runs(sd):
    for masked in (False, True):
        ref = ref_shims.build_reference_model(sd, train_config()).train()
        data = train_batch(sd, masked)
        d = {k: v.clone() for k, v in data.items()}
        torch.manual_seed(11)
        ref(d)
        loss = train_loss(d)
        ref.zero_grad()
        loss.backward()
        d = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in d.items()}
        out = {"loss": np.float64(loss.item()), "W": np.int64(d["W"]), "q_hw_c": np.array(d["q_hw_c"]),
               "param_names": np.array(sorted(n for n, _ in ref.named_parameters()))}
        put_inputs(out, {k: v for k, v in data.items() if k != "conf_matrix_gt"})
        put_matches(out, d, ("b_ids", "i_ids", "j_ids", "gt_mask", "m_bids", "mconf", "mkpts_3d_db",
                             "mkpts_query_c", "expec_f", "mkpts_query_f"))
        put_conf(out, d["conf_matrix"])
        params = dict(ref.named_parameters())
        for k in GRAD_PARAMS:
            grad = params[k].grad
            put_sample(out, "grad_" + k, grad)
            out["grad_" + k + "_absmax"] = np.float32(grad.abs().max().item())
        out["running_mean"] = dict(ref.named_buffers())["backbone.layer1.0.bn1.running_mean"].numpy()
        save("train_" + ("masked" if masked else "plain"), out)


def main():
    assert ref_shims.available(), f"no checkout of the original OnePose++ at {ref_shims.REFERENCE_ROOT} (set OPP_REFERENCE_ROOT)"
    os.makedirs(OUT_DIR, exist_ok=True)
    sd = workload.synthetic_state_dict(0)
    oracle_runs(sd)
    loftr_runs()
    loftr_layout()
    train_runs(sd)


if __name__ == "__main__":
    sys.exit(main())
