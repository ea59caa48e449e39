"""CPU tests: the oracle restatement against the committed golden fixtures generated from the
unmodified reference (oracle/make_golden.py: stored inputs; oracle/make_reference_runs.py: inputs
rebuilt from their seeds, the reference's results recorded under tests/golden/reference_runs/)."""
import numpy as np
import pytest
import torch

from oracle import oracle, workload
from tests import golden_io

WEIGHTS = {}


def weights(seed=0):
    if seed not in WEIGHTS:
        WEIGHTS[seed] = workload.synthetic_state_dict(seed)
    return WEIGHTS[seed]


def test_state_dict_layout():
    sd = weights()
    assert len(sd) == 195
    n_params = sum(v.numel() for k, v in sd.items()
                   if "running_" not in k and "num_batches_tracked" not in k)
    assert n_params == 10_226_480  # SURVEY.md App. C


def test_position_encoding_quirk():
    # position_encoding.py:25-28: (-ln(1e4) / d_model // 2) == -1.0 -> div_term = exp(-k), k even
    pe = oracle.position_encoding_sine(256, 8, 8)
    k = torch.arange(0, 128, 2).float()
    x = torch.arange(1, 9).float()
    assert torch.allclose(pe[0::4, 0, :], torch.sin(x[None] * torch.exp(-k)[:, None]), atol=1e-6)
    assert torch.allclose(pe[3::4, :, 0], torch.cos(x[None] * torch.exp(-k)[:, None]), atol=1e-6)


@pytest.mark.parametrize("case", golden_io.cases())
def test_oracle_matches_golden(case):
    data, z = golden_io.load(case)
    stages = {}
    oracle.forward(weights(), data, stages=stages)
    for k in ("b_ids", "i_ids", "j_ids", "m_bids"):
        assert np.array_equal(data[k].numpy(), z[k]), k
    for k, tol in (("mconf", 2e-4), ("mkpts_3d_db", 0), ("mkpts_query_c", 0), ("mkpts_query_f", 2e-3)):
        assert np.allclose(data[k].numpy(), z[k], rtol=0, atol=tol), k
    # expec_f: coordinates tight; the std column is sqrt(clamp(var)) and amplifies 1e-7 to 3e-4
    assert np.allclose(data["expec_f"].numpy()[:, :2], z["expec_f"][:, :2], atol=2e-4)
    assert np.allclose(data["expec_f"].numpy()[:, 2], z["expec_f"][:, 2], atol=5e-3)
    conf = data["conf_matrix"]
    assert np.allclose(conf.max(2).values.numpy(), z["conf_rowmax"], atol=2e-4)
    assert np.allclose(conf.flatten()[torch.from_numpy(z["conf_sample_idx"])].numpy(), z["conf_sample"], atol=2e-4)
    for name, t in (("feat_c", stages["feat_c"]), ("feat_f", stages["feat_f"]),
                    ("tok3d_out", stages["layers"][-1][0]), ("tok2d_out", stages["layers"][-1][1]),
                    ("fine3d_out", stages["fine3d"]), ("fine2d_out", stages["fine2d"])):
        got = t.flatten()[torch.from_numpy(z[name + "_idx"])].numpy()
        assert np.allclose(got, z[name], rtol=1e-3, atol=2e-4), name
    assert float(z["min_thr_margin"]) > 5e-3 and float(z["min_row_margin"]) > 0.05


def test_random_workload_has_no_matches():
    # BASELINE.json config 1 taken literally (random descriptors): no mutual match above thr, M = 0
    data = workload.random_workload(192, 192, 2000)
    oracle.forward(weights(), data)
    assert data["b_ids"].numel() == 0
    assert data["expec_f"].shape == (0, 3)
    assert data["mkpts_query_f"].shape == (0, 2)


@pytest.mark.parametrize("shape", [(96, 128, 300, 120, 2, False, "linear"), (512, 512, 5000, 3000, 1, False, "linear"),
                                   (96, 128, 300, 120, 2, True, "linear"), (96, 128, 300, 120, 2, False, "full")],
                         ids=["small_b2", "baseline_512_n5000", "small_b2_query_mask", "small_b2_full_attention"])
def test_oracle_matches_reference_live(shape, request):
    """The oracle against the results the unmodified reference computed on the same planted
    workload (recorded by oracle/make_reference_runs.py)."""
    import copy
    z = golden_io.reference_run("oracle_" + request.node.callspec.id)
    sd = weights()
    h, w, n, npl, batch, masked, attention = shape
    assert tuple(z["case"]) == shape[:6] and str(z["attention"]) == attention
    data, meta = workload.planted_workload(sd, h, w, n, npl, batch=batch, seed=5)
    if masked:   # img_pad flow (OnePosePlusModel.py:158): bottom / right of the coarse grid is padding
        data["query_image_mask"] = workload.pad_mask(batch, h // 8, w // 8)
    golden_io.check_inputs(z, data)
    cfg = copy.deepcopy(oracle.DEFAULT_CONFIG)
    cfg["loftr_coarse"]["attention"] = attention      # "full": FullAttention (linear_attention.py:64-95)
    d_or = {k: v.clone() for k, v in data.items()}
    oracle.forward(sd, d_or, cfg=cfg)
    golden_io.check_conf(z, d_or["conf_matrix"], atol=1e-4)
    if attention == "full":
        # same weights, different attention: the planted bank no longer matches, compare the raw matrix
        assert np.array_equal(z["b_ids"], d_or["b_ids"].numpy()) and np.array_equal(z["j_ids"], d_or["j_ids"].numpy())
        return
    assert len(z["b_ids"]) > 20
    for k in ("b_ids", "i_ids", "j_ids", "m_bids", "mkpts_3d_db", "mkpts_query_c"):
        assert np.array_equal(z[k], d_or[k].numpy()), k
    assert np.allclose(z["mkpts_query_f"], d_or["mkpts_query_f"].numpy(), atol=2e-3)
    assert np.allclose(z["expec_f"][:, :2], d_or["expec_f"][:, :2].numpy(), atol=2e-4)


def test_pnp_oracle_recovers_planted_poses():
    """oracle/pnp.py (cv2.solvePnPRansac as called by metric_utils.py:169-204, then LM on the inliers)
    on planted frames with 30 % outliers: the refined pose sits at the planted pose up to the noise."""
    import numpy as np
    from oracle import pnp
    b, p3, p2, K, gt = pnp.synthetic_frames(3, outlier_frac=0.3, noise_px=0.5, seed=3)
    for i in range(3):
        m = b == i
        pose, homo, inl, ok = pnp.ransac_pnp(K[i], p2[m], p3[m], pnp_reprojection_error=5)
        assert ok and homo.shape == (4, 4) and 0.6 * m.sum() < len(inl) < 0.8 * m.sum()
        ref = pnp.refined(K[i], p2[m], p3[m], pose, inl)
        assert np.abs(ref - gt[i]).max() < 5e-3 and np.abs(ref - pose).max() < 2e-3


@pytest.mark.parametrize("case", [(192, 256, 2, False), (256, 320, 1, True)], ids=["b2", "b1_scaled"])
def test_loftr_oracle_matches_reference_live(case, request):
    """oracle/loftr_oracle.py against the results of the unmodified LoFTR_for_OnePose_Plus
    (src/KeypointFreeSfM/loftr_for_sfm/loftr.py + submodules/LoFTR/src/loftr) on a planted pair
    (recorded by oracle/make_reference_runs.py)."""
    from oracle import loftr_oracle
    z = golden_io.reference_run("loftr_" + request.node.callspec.id)
    h, w, batch, with_scale = case
    assert tuple(z["case"]) == case
    sd, data = workload.planted_loftr(h, w, batch=batch, with_scale=with_scale)
    golden_io.check_inputs(z, data)
    golden_io.check_inputs(z, {k: sd[k] for k in ("loftr_coarse.layers.7.norm2.bias",
                                                  "backbone.layer1_outconv2.3.weight")}, prefix="sd_")
    cfg = dict(loftr_oracle.DEFAULT_CONFIG)
    d_or = loftr_oracle.forward(sd, {k: v.clone() for k, v in data.items()}, cfg)
    assert len(z["b_ids"]) > 100 * batch
    off = (z["i_ids"] - z["j_ids"])
    assert (off == 2 * (w // 8) + 3).mean() > 0.9      # the planted (16, 24) px shift
    for k in ("b_ids", "i_ids", "j_ids", "mkpts0_c", "mkpts1_c"):
        assert np.array_equal(z[k], d_or[k].numpy()), k
    golden_io.check_conf(z, d_or["conf_matrix"], atol=1e-4)
    assert np.allclose(z["mconf"], d_or["mconf"].numpy(), atol=1e-4)
    assert np.allclose(z["expec_f"][:, :2], d_or["expec_f"][:, :2].numpy(), atol=2e-4)
    assert np.allclose(z["mkpts1_f"], d_or["mkpts1_f"].numpy(), atol=2e-3) and np.array_equal(z["mkpts0_f"], d_or["mkpts0_f"].numpy())
    assert int(z["W"]) == 9
