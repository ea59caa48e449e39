"""CPU test of the training-mode forward (onepose_plus_plus_b200/train_path.py) against the
unmodified reference in .train() mode (its results recorded by oracle/make_reference_runs.py): same
outputs, same random ground-truth padding (identical RNG consumption), same gradients, same
BatchNorm running-statistic updates — i.e. PL_OnePosePlus.training_step
(OnePosePlus_lightning_model.py:54-60) sees the same thing from the drop-in as from the reference
class."""
import copy

import numpy as np
import pytest
import torch

from oracle import oracle, workload
from oracle.make_reference_runs import sampled
from onepose_plus_plus_b200 import OnePosePlus_model
from tests import golden_io


def _batch(sd, masked):
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


@pytest.mark.parametrize("masked", [False, True])
def test_training_forward_and_gradients_match_reference(masked):
    z = golden_io.reference_run("train_masked" if masked else "train_plain")
    sd = workload.synthetic_state_dict(0)
    cfg = copy.deepcopy(oracle.DEFAULT_CONFIG)
    cfg["coarse_matching"]["train"]["train_pad_num_gt_min"] = 20      # < 0.3 * B * min(L, S) at this size
    ours = OnePosePlus_model(copy.deepcopy(cfg))
    ours.load_state_dict(sd, strict=True)
    ours.train()
    data = _batch(sd, masked)
    golden_io.check_inputs(z, data)
    do = {k: v.clone() for k, v in data.items()}
    torch.manual_seed(11)
    ours(do)
    # (the std column is sqrt(clamp(var)): ill-conditioned near 0, left out of the gradient check)
    loss = (do["conf_matrix"] * do["conf_matrix_gt"]).sum() + do["expec_f"][:, :2].pow(2).sum()
    ours.zero_grad()
    loss.backward()
    lr, lo = float(z["loss"]), loss.item()
    do = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in do.items()}
    assert len(z["b_ids"]) > 50 and z["gt_mask"].any() and not z["gt_mask"].all()   # predictions + gt padding
    for k in ("b_ids", "i_ids", "j_ids", "gt_mask", "m_bids", "mkpts_3d_db", "mkpts_query_c"):
        assert np.array_equal(z[k], do[k].numpy()), k
    golden_io.check_conf(z, do["conf_matrix"], rtol=1e-3, atol=1e-5)
    for k in ("mconf", "mkpts_query_f"):
        assert np.allclose(z[k], do[k].numpy(), rtol=1e-3, atol=1e-5), k
    # the recorded run comes from another machine: the sharp fine softmax amplifies the CPU rounding of
    # the planted inputs and of the backbone (thread count alone moves it by 2e-5) beyond the 1e-5
    # that holds within one process
    assert np.allclose(z["expec_f"][:, :2], do["expec_f"][:, :2].numpy(), atol=1e-4)
    assert np.allclose(z["expec_f"][:, 2], do["expec_f"][:, 2].numpy(), atol=5e-3)
    assert do["W"] == 5 and tuple(do["q_hw_c"]) == (12, 16) and abs(lr - lo) <= 1e-4 * abs(lr)
    po = dict(ours.named_parameters())
    assert sorted(po) == z["param_names"].tolist()
    checked = 0
    for name in ("backbone.conv1.weight", "backbone.layer2.0.bn1.weight", "backbone.layer1_outconv2.3.weight",
                 "kpt_3d_pos_encoding.encoder.0.weight", "loftr_coarse.layers.0.q_proj.weight",
                 "loftr_coarse.layers.5.mlp.2.weight", "loftr_coarse.layers.3.norm1.bias",
                 "loftr_fine.layers.1.merge.weight"):
        gr, go = z["grad_" + name], po[name].grad
        assert go is not None, name
        gmax = float(z["grad_" + name + "_absmax"])    # of the whole reference gradient; gr is a fixed sample
        assert np.allclose(gr, sampled(go, len(gr)).numpy(), rtol=2e-4, atol=1e-6 + 2e-4 * gmax), name
        checked += 1
    assert checked == 8
    # BatchNorm ran on batch statistics and moved its running buffers identically
    bo = dict(ours.named_buffers())
    k = "backbone.layer1.0.bn1.running_mean"
    assert not torch.equal(bo[k], sd[k]) and np.allclose(z["running_mean"], bo[k].numpy(), atol=1e-6)
    assert int(bo["backbone.bn1.num_batches_tracked"]) == 1
    # back in eval mode the CUDA path is the only path (no silent fallback on CPU tensors)
    ours.eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        ours({k: v.clone() for k, v in data.items() if k != "conf_matrix_gt"})
