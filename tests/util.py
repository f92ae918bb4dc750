"""Shared helpers for the GPU parity tests."""
import hashlib

import numpy as np
import torch


def field_case(tn=2000, vn=3, hn=128, seed=0, noise_deg=3.0, outliers=0.2, extent=(640, 480)):
    """Reference-layout inputs: direct [tn,vn,2], coords [tn,2] (integer pixels), idxs [hn,vn,2]."""
    rng = np.random.default_rng(seed)
    W, H = extent
    coords = np.stack([rng.integers(0, W, tn), rng.integers(0, H, tn)], axis=1).astype(np.float32)
    kp = np.stack([rng.uniform(0.1 * W, 0.9 * W, vn), rng.uniform(0.1 * H, 0.9 * H, vn)], axis=1)
    kp[-1, 0] = 1.3 * W
    ang = np.arctan2(kp[None, :, 1] - coords[:, None, 1], kp[None, :, 0] - coords[:, None, 0])
    ang = ang + rng.normal(0, np.radians(noise_deg), size=ang.shape)
    out = rng.uniform(size=ang.shape) < outliers
    ang = np.where(out, rng.uniform(0, 2 * np.pi, size=ang.shape), ang)
    direct = np.stack([np.cos(ang), np.sin(ang)], axis=-1).astype(np.float32)
    idxs = rng.integers(0, tn, size=(hn, vn, 2)).astype(np.int32)
    idxs[0, :, 1] = idxs[0, :, 0]                       # t0 == t1 -> degenerate
    return direct, coords, idxs, kp.astype(np.float32)


def cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def digest(*tensors):
    """sha256 of the tensors' values in their logical (contiguous) order: pins inputs and byte-exact outputs that are
    too large to store in tests/golden/."""
    h = hashlib.sha256()
    for t in tensors:
        h.update(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes())
    return h.hexdigest()


def bits_equal(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    b = np.ascontiguousarray(b, dtype=np.float32).view(np.uint32)
    return np.array_equal(a, b)


def pnp_case(seed, pn=9, noise=1.0, pert=(0.05, 0.02)):
    """One synthetic uncertainty-PnP problem in the LINEMOD geometry (model points within +-10 cm, object 0.6-1.2 m away,
    LINEMOD intrinsics): (pts2d [pn,2], pts3d [pn,3], wgt2d [pn,3], K [3,3], init_rt [6], true_rt [6]), float64.
    Weights are inv(sqrtm(cov)) of random SPD covariances, i.e. what pvb_uncertainty_weights produces."""
    rng = np.random.default_rng(seed)
    pts3d = rng.uniform(-0.1, 0.1, (pn, 3))
    aa = rng.normal(size=3)
    aa *= rng.uniform(0.2, 2.5) / np.linalg.norm(aa)
    t = np.array([rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2), rng.uniform(0.6, 1.2)])
    K = np.array([[572.4114, 0, 325.2611], [0, 573.57043, 242.04899], [0, 0, 1.0]])
    theta = np.linalg.norm(aa)
    w = aa / theta
    Wx = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    R = np.eye(3) + np.sin(theta) * Wx + (1 - np.cos(theta)) * (Wx @ Wx)
    cam = pts3d @ R.T + t
    uv = np.stack([K[0, 0] * cam[:, 0] / cam[:, 2] + K[0, 2], K[1, 1] * cam[:, 1] / cam[:, 2] + K[1, 2]], 1)
    uv = uv + rng.normal(size=uv.shape) * noise
    wgt = np.empty((pn, 3))
    for i in range(pn):
        A = rng.normal(size=(2, 2))
        C = A @ A.T * rng.uniform(0.5, 4) + 0.1 * np.eye(2)
        lam, V = np.linalg.eigh(C)
        Wi = V @ np.diag(lam ** -0.5) @ V.T
        wgt[i] = [Wi[0, 0], Wi[0, 1], Wi[1, 1]]
    true_rt = np.concatenate([aa, t])
    init = true_rt + np.concatenate([rng.normal(size=3) * pert[0], rng.normal(size=3) * pert[1]])
    return uv, pts3d, wgt, K, init, true_rt
