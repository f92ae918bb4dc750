"""GPU: the other BASELINE.json configurations as parity / property cases (cfg-2 is the bench workload and is
covered in test_gpu_layer.py / test_gpu_reference_parity.py).  Full image size, keypoint count and hypothesis
count; batch reduced where only per-image behaviour is checked (images are independent).

Properties used (size-independent):
  * fused counts == the reference's byte-tensor formulation evaluated by the REFERENCE EXTENSION itself
    (oracle/_ref's voting_for_hypothesis, the unmodified .cu compiled by oracle/build_ref.py), recorded on these very
    cases by tests/golden/make_golden_parity.py (tests/golden/reference_counts.npz);
  * an image's result does not depend on batch composition (shard invariance);
  * noise-free fields recover the keypoints;
  * selected-pixel counts obey the thinning law (tn == nz when fg <= max_num, else ~ Binomial(nz, max_num/fg)).
"""
import os

import numpy as np
import pytest
import torch

from util import digest

pytestmark = pytest.mark.gpu
COUNTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_counts.npz")
CASES = ["cfg1", "cfg3", "cfg4"] + [f"cfg5_{K}_{hn}_{fill}" for K, hn, fill in
                                    [(4, 128, 0.01), (9, 2048, 0.80), (17, 512, 0.30), (4, 2048, 0.05)]]


def _inputs(cfg, **kw):
    from clean_pvnet_b200 import synth
    return synth.make_inputs(cfg, device="cuda", **kw)


def _reference_counts(key, mask, vertex):
    """[K, hn] hypothesis counts of the case's checked image, as the reference extension counted them."""
    g = np.load(COUNTS)
    assert digest(mask, vertex) == str(g[key + "_inputs"]), f"{key}: inputs differ from those the reference ran on"
    return torch.from_numpy(g[key]).cuda()


def test_reference_extension_is_the_checker_here():
    """Every count check below has the reference extension's counts to compare with."""
    g = np.load(COUNTS)
    for key in CASES:
        assert g[key].dtype == np.int32 and g[key].ndim == 2 and len(str(g[key + "_inputs"])) == 64, key


def test_cfg1_plumbing_case(pvb, oracle):
    """BASELINE.json configs[0]: single 128x128 mask, PURE RANDOM unit-vector field, K=1, 64 hypotheses.  No consensus
    exists; what is checked is that the CUDA path and the CPU oracle agree on every intermediate and on the result."""
    mask, vertex, _ = _inputs("cfg1", seed=1235)
    out, dbg = pvb.ransac_voting_layer_v3(mask, vertex, 64, inlier_thresh=0.99, seed=11, debug=True)
    want, odbg = oracle.ransac_voting_layer_v3(mask.cpu().numpy(), vertex.cpu().numpy(), 64, inlier_thresh=0.99, seed=11,
                                               debug=True)
    assert np.array_equal(dbg["tn"].cpu().numpy(), odbg["tn"])
    assert np.array_equal(dbg["hyp"].cpu().numpy().view(np.uint32), odbg["hyp"].view(np.uint32))
    assert np.array_equal(dbg["counts"].cpu().numpy(), odbg["counts"])
    assert np.abs(out.cpu().numpy() - want).max() < 1e-4
    assert torch.equal(dbg["counts"][0], _reference_counts("cfg1", mask, vertex))
    _, cov = pvb.estimate_voting_distribution_with_mean(mask, vertex, out, seed=12)
    _, wcov = oracle.estimate_voting_distribution_with_mean(mask.cpu().numpy(), vertex.cpu().numpy(), out.cpu().numpy(), seed=12)
    assert np.allclose(cov.cpu().numpy(), wcov, rtol=1e-5, atol=1e-6)


def test_cfg3_fragmented_masks_1024_hypotheses(pvb):
    """Occlusion-LINEMOD shape: 480x640, K=9, hn=1024, 5-15 % fragmented masks (two hypothesis slices)."""
    mask, vertex, _ = _inputs("cfg3", seed=1237, B=6)
    out, dbg = pvb.ransac_voting_layer_v3(mask, vertex, 1024, inlier_thresh=0.99, seed=31, debug=True)
    tn, nz = dbg["tn"].cpu().numpy(), dbg["nz"].cpu().numpy()
    fg = dbg["fgsum"].cpu().numpy()
    for b in range(6):
        if fg[b] <= 30000:
            assert tn[b] == nz[b]
        else:
            assert abs(tn[b] - 30000) < 6 * np.sqrt(30000)
    assert torch.isfinite(out).all()
    assert torch.equal(dbg["counts"][1], _reference_counts("cfg3", mask, vertex))
    one = pvb.ransac_voting_layer_v3(mask[4:5], vertex[4:5], 1024, inlier_thresh=0.99, seed=31, img_base=4)
    assert torch.equal(one[0], out[4])


def test_cfg4_tless_shape(pvb):
    """T-LESS shape: 720x540, K=17, hn=512 (per-GPU share of the 8-GPU batch is 16 images; 3 checked here)."""
    mask, vertex, kp = _inputs("cfg4", seed=1238, B=3, noise_deg=0.0, outlier_frac=0.0)
    out, dbg = pvb.ransac_voting_layer_v3(mask, vertex, 512, inlier_thresh=0.99, seed=41, debug=True)
    assert (out - kp).abs().max().item() < 2e-2          # noise-free: all 17 keypoints, incl. the out-of-image one
    assert torch.equal(dbg["counts"][2], _reference_counts("cfg4", mask, vertex))
    _, cov = pvb.estimate_voting_distribution_with_mean(mask, vertex, out, seed=42)
    assert cov.shape == (3, 17, 2, 2) and torch.isfinite(cov).all()
    assert (cov[..., 0, 0] >= 0).all() and (cov[..., 1, 1] >= 0).all()


@pytest.mark.parametrize("K,hn,fill", [(4, 128, 0.01), (9, 2048, 0.80), (17, 512, 0.30), (4, 2048, 0.05)])
def test_cfg5_stress_corners(pvb, oracle, K, hn, fill):
    """Stress sweep corners: 640x640, K in {4,9,17}, hn in {128,512,2048}, fill 1-80 %."""
    cfg = dict(B=2, H=640, W=640, K=K, hn=hn, fill=(fill, fill), kind="blob")
    mask, vertex, kp = _inputs(cfg, seed=1239)
    out, dbg = pvb.ransac_voting_layer_v3(mask, vertex, hn, inlier_thresh=0.99, seed=51, debug=True)
    assert torch.isfinite(out).all()
    assert torch.equal(dbg["counts"][0], _reference_counts(f"cfg5_{K}_{hn}_{fill}", mask, vertex))
    # operator-level parity with the oracle where the CPU finishes in seconds
    tn0 = int(dbg["tn"][0])
    if tn0 * K * hn < 3e8:
        want, odbg = oracle.ransac_voting_layer_v3(mask[:1].cpu().numpy(), vertex[:1].cpu().numpy(), hn,
                                                   inlier_thresh=0.99, seed=51, debug=True)
        assert np.array_equal(odbg["counts"][0], dbg["counts"][0].cpu().numpy())
        assert np.abs(want[0] - out[0].cpu().numpy()).max() < 1e-4
    # image order / batch composition do not matter when the global image index is kept
    solo = pvb.ransac_voting_layer_v3(mask[1:2], vertex[1:2], hn, inlier_thresh=0.99, seed=51, img_base=1)
    assert torch.equal(solo[0], out[1])


def test_large_batch_many_images(pvb):
    """B=64 at 480x640 (cfg-3 batch size): one launch, results equal to 4 separate 16-image launches."""
    mask, vertex, _ = _inputs("cfg2", seed=1241, B=64)
    full = pvb.ransac_voting_layer_v3(mask, vertex, 512, inlier_thresh=0.99, seed=61)
    parts = [pvb.ransac_voting_layer_v3(mask[i:i + 16], vertex[i:i + 16], 512, inlier_thresh=0.99, seed=61, img_base=i)
             for i in range(0, 64, 16)]
    assert torch.equal(full, torch.cat(parts))


def test_cfg5_maximum_batch(pvb):
    """Stress sweep batch size: B=256 at 640x640 in ONE launch set (K=4, hn=128 keep the dense input at 3.4 GB);
    fill varies 1-80 % per image; image 200 equals its stand-alone result."""
    cfg = dict(B=256, H=640, W=640, K=4, hn=128, fill=(0.01, 0.80), kind="blob")
    from clean_pvnet_b200 import synth
    mask, vertex, _ = synth.make_inputs(cfg, device="cuda", seed=1242)
    out, dbg = pvb.ransac_voting_layer_v3(mask, vertex, 128, inlier_thresh=0.99, seed=71, debug=True)
    assert out.shape == (256, 4, 2) and torch.isfinite(out).all()
    tn, nz, fg = dbg["tn"].cpu(), dbg["nz"].cpu(), dbg["fgsum"].cpu()
    assert (tn[fg <= 30000] == nz[fg <= 30000]).all()
    assert ((tn[fg > 30000] - 30000).abs() < 6 * 30000 ** 0.5).all()
    assert int((fg > 30000).sum()) > 50 and int((fg <= 30000).sum()) > 5
    solo = pvb.ransac_voting_layer_v3(mask[200:201], vertex[200:201], 128, inlier_thresh=0.99, seed=71, img_base=200)
    assert torch.equal(solo[0], out[200])
