"""GPU parity against the reference itself: the unmodified clean-pvnet CUDA extension compiled for
sm_100 by oracle/build_ref.py, recorded on these very cases by tests/golden/make_golden_parity.py
(tests/golden/reference_parity.npz; inputs are regenerated from their seeds and checked by sha256).

  kernel level : generate_hypothesis bit-equal, voting_for_hypothesis bytes equal, counts equal
  op level     : ransac_voting_layer_v3 / estimate_voting_distribution_with_mean under the same
                 torch.manual_seed (rng="torch" replays the reference's generator consumption):
                 keypoint L2 error < 1e-3 px (north-star bar), covariance rtol 2e-3.
"""
import os

import numpy as np
import pytest
import torch

from util import bits_equal, cuda, digest, field_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    """What the reference computed on each case, keyed as tests/golden/make_golden_parity.py names them."""
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_parity.npz"))


def _inputs(ref, key, cfg, **kw):
    from clean_pvnet_b200 import synth
    mask, vertex, kp = synth.make_inputs(cfg, device="cuda", **kw)
    assert digest(mask, vertex) == str(ref[key + "_inputs"]), f"{key}: inputs differ from those the reference ran on"
    return mask, vertex, kp


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("tn,vn,hn,seed", [(3000, 3, 128, 0), (4096, 9, 512, 1), (700, 1, 64, 2)])
def test_kernels_match_reference_extension(pvb, ref, tn, vn, hn, seed):
    key = f"kernels_{tn}_{vn}_{hn}_{seed}"
    direct, coords, idxs, _ = field_case(tn, vn, hn, seed)
    d, c, i = cuda(direct, coords, idxs)
    want_h = _t(ref[key + "_hyp"])
    got_h = pvb.ransac_voting.generate_hypothesis(d, c, i)
    assert bits_equal(got_h.cpu().numpy(), want_h.cpu().numpy())
    for thresh in (0.99, 0.999):
        want_counts = _t(ref[f"{key}_{thresh}_counts"])
        got_i = torch.zeros((hn, vn, tn), dtype=torch.uint8, device="cuda")
        pvb.ransac_voting.voting_for_hypothesis(d, c, want_h, got_i, thresh)
        assert torch.equal(got_i.sum(dim=2, dtype=torch.int32), want_counts)
        assert digest(got_i) == str(ref[f"{key}_{thresh}_inliers"])
        counts = pvb.ransac_voting.vote_count(d, c, want_h, thresh)
        assert torch.equal(counts, want_counts)


def test_vanishing_point_kernels_match_reference_extension(pvb, ref):
    direct, coords, idxs, _ = field_case(2000, 3, 128, 5)
    d, c, i = cuda(direct, coords, idxs)
    want_h = _t(ref["vp_hyp"])
    got_h = pvb.ransac_voting.generate_hypothesis_vanishing_point(d, c, i)
    assert bits_equal(got_h.cpu().numpy(), want_h.cpu().numpy())
    got_i = torch.zeros((128, 3, 2000), dtype=torch.uint8, device="cuda")
    pvb.ransac_voting.voting_for_hypothesis_vanishing_point(d, c, want_h, got_i, 0.999)
    assert torch.equal(got_i.sum(dim=2, dtype=torch.int32), _t(ref["vp_counts"]))
    assert digest(got_i) == str(ref["vp_inliers"])


@pytest.mark.parametrize("cfg,hn,max_num,seed", [("small", 64, 30000, 0), ("small", 128, 700, 1), ("tiny", 32, 30000, 2)])
def test_v3_matches_reference_under_same_seed(pvb, ref, cfg, hn, max_num, seed):
    key = f"v3_{cfg}_{hn}_{max_num}_{seed}"
    mask, vertex, _ = _inputs(ref, key, cfg, seed=100 + seed)
    want = _t(ref[key])
    torch.manual_seed(seed)
    got = pvb.ransac_voting_layer_v3(mask, vertex, hn, inlier_thresh=0.99, max_num=max_num, rng="torch")
    err = (got - want).norm(dim=-1).max().item()
    assert err < 1e-3, err


@pytest.mark.parametrize("layout", ["planar", "interleaved"])
def test_v3_full_size_matches_reference(pvb, ref, layout):
    """The FULL cfg-2 batch (B=16, 480x640, K=9, hn=512, thinning: fg ~ 92k > 30000), both vertex layouts, same seed.

    With ~22 000 inliers per keypoint the reference's fp32 normal equations (cuBLAS matmul + torch.sum,
    ransac_voting_gpu.py:189-193) carry their own rounding noise, largest on the ill-conditioned out-of-image keypoint;
    `<1e-3 px vs reference` is therefore only defined up to the reference's distance to itself.  That distance was measured
    with the reference: its own refit lines re-run on a PERMUTED pixel order (same inlier set, same formula, same fp32 ops).
    Pinned: ours within 1e-4 px of the exact (float64) value of the reference's formula on the reference's inlier set; the
    ours-vs-reference gap explained by the reference's distance to that value; and ours-vs-reference no larger than a small
    multiple of reference-vs-itself."""
    key = f"full_{layout}"
    mask, vertex, _ = _inputs(ref, key, "cfg2", seed=77, layout=layout)
    want, exact, ref_vs_itself = _t(ref[key + "_want"]), _t(ref[key + "_exact"]), _t(ref[key + "_ref_vs_itself"])
    torch.manual_seed(3)
    got = pvb.ransac_voting_layer_v3(mask, vertex, 512, inlier_thresh=0.99, rng="torch")
    ours_vs_exact = (got.double() - exact).norm(dim=-1)
    ref_vs_exact = (want.double() - exact).norm(dim=-1)
    ours_vs_ref = (got - want).norm(dim=-1)
    assert ours_vs_exact.max().item() < 1e-4, ours_vs_exact.max().item()
    assert (ours_vs_ref.double() <= ref_vs_exact + 2e-4).all(), (ours_vs_ref, ref_vs_exact)
    spread = max(ref_vs_itself.max().item(), ref_vs_exact.max().item())
    assert ours_vs_ref.max().item() <= max(1e-3, 3.0 * spread), (ours_vs_ref.max().item(), spread)


def test_distribution_matches_reference_under_same_seed(pvb, ref):
    mask, vertex, _ = _inputs(ref, "dist", "small", seed=200)
    mean, want = _t(ref["dist_mean"]), _t(ref["dist_cov"])
    torch.manual_seed(9)
    _, got = pvb.estimate_voting_distribution_with_mean(mask, vertex, mean, round_hyp_num=64, min_hyp_num=512,
                                                        rng="torch")
    assert torch.allclose(got, want, rtol=2e-3, atol=1e-3), (got - want).abs().max().item()


def test_distribution_with_thinning_matches_reference(pvb, ref):
    """fg > max_num: the reference thins, recomputes `foreground` (:219-223) and divides counts by it."""
    mask, vertex, _ = _inputs(ref, "dist_thinned", "small", seed=201)
    mean, want = _t(ref["dist_thinned_mean"]), _t(ref["dist_thinned_cov"])
    torch.manual_seed(10)
    _, got = pvb.estimate_voting_distribution_with_mean(mask, vertex, mean, round_hyp_num=64, min_hyp_num=256,
                                                        max_num=700, rng="torch")
    assert torch.allclose(got, want, rtol=2e-3, atol=1e-3), (got - want).abs().max().item()


def test_v1_layer_matches_reference(pvb, ref):
    """ransac_voting_layer (v1, torch.inverse instead of b_inv) -- imported by resnet18.py:5."""
    mask, vertex, _ = _inputs(ref, "v1", "small", seed=202)
    want = _t(ref["v1"])
    torch.manual_seed(4)
    got = pvb.ransac_voting_layer(mask, vertex, 64, inlier_thresh=0.99, rng="torch")
    assert (got - want).norm(dim=-1).max().item() < 1e-3


def test_production_call_pattern(pvb, ref):
    """decode_keypoint's two call patterns (resnet18.py:70-76) on the strided NCHW view with an argmax mask."""
    mask, vertex, _ = _inputs(ref, "production", "small", seed=203, layout="planar")
    seg = torch.stack([1.0 - mask.float(), mask.float()], dim=1)           # [B,2,H,W] logits
    amask = torch.argmax(seg, 1)                                           # int64, as resnet18.py:69
    want = _t(ref["production_max_num"])
    torch.manual_seed(6)
    got = pvb.ransac_voting_layer_v3(amask, vertex, 128, inlier_thresh=0.99, max_num=100, rng="torch")
    assert (got - want).norm(dim=-1).max().item() < 1e-3
    mean_w, var_w = _t(ref["production_mean"]), _t(ref["production_var"])
    torch.manual_seed(7)
    mean_g = pvb.ransac_voting_layer_v3(amask, vertex, 512, inlier_thresh=0.99, rng="torch")
    _, var_g = pvb.estimate_voting_distribution_with_mean(amask, vertex, mean_g, rng="torch")
    assert (mean_g - mean_w).norm(dim=-1).max().item() < 1e-3
    assert torch.allclose(var_g, var_w, rtol=5e-3, atol=2e-3), (var_g - var_w).abs().max().item()


def test_philox_mode_is_statistically_equivalent(pvb, ref):
    """Default (philox) sampling is a different random stream, not a different estimator."""
    mask, vertex, kp = _inputs(ref, "philox", "small", seed=300)
    want = _t(ref["philox"])
    got = pvb.ransac_voting_layer_v3(mask, vertex, 128, inlier_thresh=0.99, seed=0)
    # both land on the same inlier consensus: sub-pixel agreement on in-image keypoints
    assert (got - want)[:, :-1].norm(dim=-1).max().item() < 0.75
