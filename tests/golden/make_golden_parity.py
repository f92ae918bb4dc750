#!/usr/bin/env python
"""Records what the UNMODIFIED reference (oracle/_ref: clean-pvnet's CUDA extension + its Python operator, built by
oracle/build_ref.py) computes on the cases of tests/test_gpu_reference_parity.py and tests/test_gpu_configs.py, so that
those tests compare with the reference without needing it.  Needs a GPU and oracle/_ref:

    python tests/golden/make_golden_parity.py OUT_DIR     # -> OUT_DIR/reference_parity.npz, OUT_DIR/reference_counts.npz

Inputs are not stored (the full cfg-2 batch alone is 354 MB): the tests regenerate them from their seeds with
clean_pvnet_b200/synth.py, and `<case>_inputs` holds their sha256 so that changed inputs are told apart from changed
results.  Inlier byte tensors are stored as per-hypothesis counts plus a sha256 of the bytes, for the same reason.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from refload import load_reference  # noqa: E402
from util import cuda, digest, field_case  # noqa: E402

import clean_pvnet_b200 as pvb  # noqa: E402
from clean_pvnet_b200 import synth  # noqa: E402


def _inputs(g, key, cfg, **kw):
    mask, vertex, kp = synth.make_inputs(cfg, device="cuda", **kw)
    g[key + "_inputs"] = digest(mask, vertex)
    return mask, vertex, kp


def _np(t):
    return t.detach().cpu().numpy()


def _exact_refit(ext, dbg, thresh):
    """The reference's refit formula (ransac_voting_gpu.py:177-196) in float64 on the inlier set the
    reference extension itself produces for the winning hypotheses -- the value both implementations
    approximate (the reference in fp32 through cuBLAS matmul + torch.sum + LU)."""
    B, K = dbg["win"].shape[:2]
    out = torch.zeros((B, K, 2), dtype=torch.float64, device="cuda")
    for b in range(B):
        tn = int(dbg["tn"][b])
        direct = dbg["dirs"][b, :, :tn].permute(1, 0, 2).contiguous()
        coords = dbg["xy"][b, :tn].contiguous()
        inl = torch.zeros((1, K, tn), dtype=torch.uint8, device="cuda")
        ext.voting_for_hypothesis(direct, coords, dbg["win"][b][None].contiguous(), inl, thresh)
        w = inl[0].double()                                           # [K,tn]
        normal = torch.stack([direct[:, :, 1], -direct[:, :, 0]], dim=-1).double().permute(1, 0, 2) * w[:, :, None]
        bb = (normal * coords.double()[None]).sum(2)                  # [K,tn]
        ATA = normal.transpose(1, 2) @ normal
        ATb = (normal * bb[:, :, None]).sum(1)
        out[b] = torch.linalg.solve(ATA, ATb[:, :, None])[:, :, 0]
    return out


def _reference_refit_lines(ext, gpu, direct, coords, win, thresh):
    """ransac_voting_gpu.py:177-196 as the reference executes them (fp32 torch ops: matmul, sum, its own b_inv) on a given
    pixel ORDER -- the winner's inlier set does not depend on the order, the fp32 sums do."""
    tn, vn = direct.shape[0], direct.shape[1]
    normal = torch.zeros_like(direct)
    normal[:, :, 0] = direct[:, :, 1]
    normal[:, :, 1] = -direct[:, :, 0]
    inl = torch.zeros([1, vn, tn], dtype=torch.uint8, device=direct.device)
    ext.voting_for_hypothesis(direct, coords, win[None].contiguous(), inl, thresh)
    inl = torch.squeeze(inl.float(), 0)
    normal = normal.permute(1, 0, 2) * torch.unsqueeze(inl, 2)
    b = torch.sum(normal * torch.unsqueeze(coords, 0), 2)
    ATA = torch.matmul(normal.permute(0, 2, 1), normal)
    ATb = torch.sum(normal * torch.unsqueeze(b, 2), 1)
    return torch.matmul(gpu.b_inv(ATA), torch.unsqueeze(ATb, 2))[:, :, 0], inl.sum(1)


def parity(ext, gpu):
    """tests/test_gpu_reference_parity.py, case by case."""
    g = {}
    for tn, vn, hn, seed in [(3000, 3, 128, 0), (4096, 9, 512, 1), (700, 1, 64, 2)]:
        key = f"kernels_{tn}_{vn}_{hn}_{seed}"
        d, c, i = cuda(*field_case(tn, vn, hn, seed)[:3])
        hyp = ext.generate_hypothesis(d, c, i)
        g[key + "_hyp"] = _np(hyp)
        for thresh in (0.99, 0.999):
            inl = torch.zeros((hn, vn, tn), dtype=torch.uint8, device="cuda")
            ext.voting_for_hypothesis(d, c, hyp, inl, thresh)
            g[f"{key}_{thresh}_inliers"] = digest(inl)
            g[f"{key}_{thresh}_counts"] = _np(inl.sum(dim=2, dtype=torch.int32))
    d, c, i = cuda(*field_case(2000, 3, 128, 5)[:3])
    hyp = ext.generate_hypothesis_vanishing_point(d, c, i)
    inl = torch.zeros((128, 3, 2000), dtype=torch.uint8, device="cuda")
    ext.voting_for_hypothesis_vanishing_point(d, c, hyp, inl, 0.999)
    g["vp_hyp"], g["vp_inliers"], g["vp_counts"] = _np(hyp), digest(inl), _np(inl.sum(dim=2, dtype=torch.int32))

    for cfg, hn, max_num, seed in [("small", 64, 30000, 0), ("small", 128, 700, 1), ("tiny", 32, 30000, 2)]:
        key = f"v3_{cfg}_{hn}_{max_num}_{seed}"
        mask, vertex, _ = _inputs(g, key, cfg, seed=100 + seed)
        torch.manual_seed(seed)
        g[key] = _np(gpu.ransac_voting_layer_v3(mask, vertex, hn, inlier_thresh=0.99, max_num=max_num))

    for layout in ("planar", "interleaved"):
        key = f"full_{layout}"
        mask, vertex, _ = _inputs(g, key, "cfg2", seed=77, layout=layout)
        torch.manual_seed(3)
        want = gpu.ransac_voting_layer_v3(mask, vertex, 512, inlier_thresh=0.99)
        torch.manual_seed(3)
        _, dbg = pvb.ransac_voting_layer_v3(mask, vertex, 512, inlier_thresh=0.99, rng="torch", debug=True)
        exact = _exact_refit(ext, dbg, 0.99)
        # the reference against itself: identity order must reproduce its output, a permuted order shows its fp32 spread
        B = want.shape[0]
        same_order = torch.zeros_like(want)
        permuted = torch.zeros_like(want)
        gen = torch.Generator(device="cuda").manual_seed(5)
        for b in range(B):
            tn = int(dbg["tn"][b])
            direct = dbg["dirs"][b, :, :tn].permute(1, 0, 2).contiguous()
            coords = dbg["xy"][b, :tn].contiguous()
            same_order[b], n0 = _reference_refit_lines(ext, gpu, direct, coords, dbg["win"][b], 0.99)
            perm = torch.randperm(tn, generator=gen, device="cuda")
            permuted[b], n1 = _reference_refit_lines(ext, gpu, direct[perm].contiguous(), coords[perm].contiguous(),
                                                     dbg["win"][b], 0.99)
            assert torch.equal(n0, n1)                               # the inlier SET is order independent
        assert (same_order - want).norm(dim=-1).max().item() < 1e-4  # the helper is the reference's own computation
        g[key + "_want"], g[key + "_exact"] = _np(want), _np(exact)
        g[key + "_ref_vs_itself"] = _np((permuted - want).norm(dim=-1))

    for key, seed, tseed, kw in [("dist", 200, 9, dict(min_hyp_num=512)),
                                 ("dist_thinned", 201, 10, dict(min_hyp_num=256, max_num=700))]:
        mask, vertex, _ = _inputs(g, key, "small", seed=seed)
        mean = pvb.ransac_voting_layer_v3(mask, vertex, 64, inlier_thresh=0.99, seed=1)
        torch.manual_seed(tseed)
        _, cov = gpu.estimate_voting_distribution_with_mean(mask, vertex, mean.clone(), round_hyp_num=64, **kw)
        g[key + "_mean"], g[key + "_cov"] = _np(mean), _np(cov)

    mask, vertex, _ = _inputs(g, "v1", "small", seed=202)
    torch.manual_seed(4)
    g["v1"] = _np(gpu.ransac_voting_layer(mask, vertex, 64, inlier_thresh=0.99))

    mask, vertex, _ = _inputs(g, "production", "small", seed=203, layout="planar")
    amask = torch.argmax(torch.stack([1.0 - mask.float(), mask.float()], dim=1), 1)
    torch.manual_seed(6)
    g["production_max_num"] = _np(gpu.ransac_voting_layer_v3(amask, vertex, 128, inlier_thresh=0.99, max_num=100))
    torch.manual_seed(7)
    mean_w = gpu.ransac_voting_layer_v3(amask, vertex, 512, inlier_thresh=0.99)
    _, var_w = gpu.estimate_voting_distribution_with_mean(amask, vertex, mean_w)
    g["production_mean"], g["production_var"] = _np(mean_w), _np(var_w)

    mask, vertex, _ = _inputs(g, "philox", "small", seed=300)
    torch.manual_seed(0)
    g["philox"] = _np(gpu.ransac_voting_layer_v3(mask, vertex, 128, inlier_thresh=0.99))
    return g


def _counts_by_bytes(vote, dbg, b, thresh, kstep):
    """The reference's byte-tensor formulation (ransac_voting.cpp:41-55, then a sum) of image b's hypothesis counts."""
    tn = int(dbg["tn"][b])
    direct = dbg["dirs"][b, :, :tn].permute(1, 0, 2).contiguous()
    coords = dbg["xy"][b, :tn].contiguous()
    hyp = dbg["hyp"][b].permute(1, 0, 2).contiguous()
    hn, K = hyp.shape[0], hyp.shape[1]
    out = torch.empty((K, hn), dtype=torch.int32, device="cuda")
    for k0 in range(0, K, kstep):
        k1 = min(K, k0 + kstep)
        inl = torch.zeros((hn, k1 - k0, tn), dtype=torch.uint8, device="cuda")
        vote(direct[:, k0:k1].contiguous(), coords, hyp[:, k0:k1].contiguous(), inl, thresh)
        out[k0:k1] = inl.sum(dim=2, dtype=torch.int32).t()
    return out


def counts(ext):
    """tests/test_gpu_configs.py: the hypothesis counts of one image per case, counted by the reference extension."""
    g = {}
    cases = [("cfg1", "cfg1", dict(seed=1235), 64, 11, 0, 3),
             ("cfg3", "cfg3", dict(seed=1237, B=6), 1024, 31, 1, 3),
             ("cfg4", "cfg4", dict(seed=1238, B=3, noise_deg=0.0, outlier_frac=0.0), 512, 41, 2, 2)]
    for K, hn, fill in [(4, 128, 0.01), (9, 2048, 0.80), (17, 512, 0.30), (4, 2048, 0.05)]:
        cfg = dict(B=2, H=640, W=640, K=K, hn=hn, fill=(fill, fill), kind="blob")
        cases.append((f"cfg5_{K}_{hn}_{fill}", cfg, dict(seed=1239), hn, 51, 0, 1 if hn > 1024 else 3))
    for key, cfg, kw, hn, seed, b, kstep in cases:
        mask, vertex, _ = _inputs(g, key, cfg, **kw)
        _, dbg = pvb.ransac_voting_layer_v3(mask, vertex, hn, inlier_thresh=0.99, seed=seed, debug=True)
        g[key] = _np(_counts_by_bytes(ext.voting_for_hypothesis, dbg, b, 0.99, kstep))
    return g


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    ext, gpu = load_reference()
    np.savez_compressed(os.path.join(out_dir, "reference_parity.npz"), **parity(ext, gpu))
    np.savez_compressed(os.path.join(out_dir, "reference_counts.npz"), **counts(ext))
    print("golden vectors written to", out_dir, sorted(os.listdir(out_dir)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
