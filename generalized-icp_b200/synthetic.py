"""Synthetic 3-D inputs of the shapes BASELINE.json names (SURVEY.md section 8d, configs 3-5):
planar-patch clouds (ours - the reference has no 3-D inputs).

:func:`patches3d_pair` is the host (numpy) generator, :func:`patches3d_batch_device` builds the
config-4 batch directly in HBM with torch (device plumbing only - no registration math lives here).
The seeded restatements of the reference demos' 2-D input recipes (configs 1-2) are test
infrastructure and live in ``tests/demo_inputs.py``.
"""
from __future__ import annotations

import numpy as np


# --------------------------------------------------------------------------
# configs 3-5: 3-D planar patches
# --------------------------------------------------------------------------
def _rand_rotation(rng, max_deg):
    axis = rng.normal(size=3)
    axis /= np.linalg.norm(axis)
    ang = np.deg2rad(rng.uniform(-max_deg, max_deg))
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def patches3d_pair(n=100_000, n_patches=64, cube=100.0, patch=30.0, sigma=0.02,
                   max_rot_deg=2.0, max_trans=0.5, seed=0, moved_patches=0, moved_offset=0.0):
    """Source and target drawn independently from the same random planar
    patches; the target surface is moved by a rigid motion about the cube
    centre.  Returned as float32 (N,3) arrays plus the 4x4 ground truth that
    maps source onto target.

    Structured outliers (a moved object): with ``moved_patches`` = m > 0 the
    target points of patches 0..m-1 are shifted by ``moved_offset`` along their
    patch's normal before the rigid motion, so those matches are wrong by a
    fixed distance that can lie inside the correspondence gate.  The defaults
    draw exactly the same clouds as before (no extra random numbers)."""
    rng = np.random.default_rng(seed)
    centres = rng.uniform(0.25 * cube, 0.75 * cube, size=(n_patches, 3))
    frames = np.stack([np.linalg.qr(rng.normal(size=(3, 3)))[0] for _ in range(n_patches)])

    def sample():
        which = rng.integers(0, n_patches, size=n)
        ab = rng.uniform(-patch / 2, patch / 2, size=(n, 2))
        p = centres[which] + ab[:, :1] * frames[which, :, 0] + ab[:, 1:] * frames[which, :, 1]
        return p + rng.normal(0, sigma, size=(n, 3)), which

    src, _ = sample()
    tgt, which_t = sample()
    if moved_patches:
        moved = which_t < moved_patches
        tgt[moved] += moved_offset * frames[which_t[moved], :, 2]
    R = _rand_rotation(rng, max_rot_deg)
    tdir = rng.normal(size=3)
    t = tdir / np.linalg.norm(tdir) * rng.uniform(0, max_trans)
    c = np.full(3, cube / 2)
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = c - R @ c + t
    tgt = tgt @ R.T + T[:3, 3]
    return src.astype(np.float32), tgt.astype(np.float32), T


CONFIG3 = dict(n=100_000, n_patches=64, cube=100.0, patch=30.0, sigma=0.02, max_rot_deg=2.0, max_trans=0.5)
CONFIG3_PARAMS = dict(k=20, max_distance_nearest_neighbors=6.0, max_distance_correspondence=4.0, tolerance=1e-6)
CONFIG4 = dict(n=32_768, n_patches=16, cube=40.0, patch=30.0, sigma=0.02, max_rot_deg=2.0, max_trans=0.5)
CONFIG4_PARAMS = dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=2.0, tolerance=1e-6)
CONFIG5 = dict(n=16_777_216, n_patches=1024, cube=400.0, patch=30.0, sigma=0.02, max_rot_deg=0.25, max_trans=0.5)
CONFIG5_PARAMS = dict(k=20, max_distance_nearest_neighbors=1.8, max_distance_correspondence=2.5, tolerance=1e-6)


def patches3d_batch_device(n_pairs, n=32_768, n_patches=16, cube=40.0, patch=30.0, sigma=0.02,
                           max_rot_deg=2.0, max_trans=0.5, seed=0, device="cuda", chunk=256, first_pair=0):
    """Config-4 batch generated in HBM: (src, tgt) float32 (n_pairs*n, 3), CSR
    offsets (n_pairs+1,) int64 (identical for both sides) and the ground-truth
    4x4 per pair.  Same distribution as :func:`patches3d_pair`; the random
    stream is torch's Philox generator seeded with ``seed`` (per-chunk), so a
    sample of pairs can be copied back for the CPU oracle.  ``first_pair``: the batch is pairs
    [first_pair, first_pair + n_pairs) of one job-wide sequence (a rank's share of a batch that is partitioned
    over GPUs); with ``first_pair`` a multiple of ``chunk`` every rank count reproduces the same job."""
    import torch

    g = torch.Generator(device=device)
    src = torch.empty((n_pairs * n, 3), dtype=torch.float32, device=device)
    tgt = torch.empty_like(src)
    Ts = torch.empty((n_pairs, 4, 4), dtype=torch.float64, device=device)
    for c0 in range(0, n_pairs, chunk):
        b = min(chunk, n_pairs - c0)
        g.manual_seed(seed * 1_000_003 + first_pair + c0)
        centres = torch.empty((b, n_patches, 3), device=device).uniform_(0.25 * cube, 0.75 * cube, generator=g)
        frames, _ = torch.linalg.qr(torch.randn((b, n_patches, 3, 3), device=device, generator=g))
        axis = torch.randn((b, 3), device=device, dtype=torch.float64, generator=g)
        axis = axis / axis.norm(dim=1, keepdim=True)
        ang = torch.deg2rad(torch.empty((b,), device=device, dtype=torch.float64).uniform_(-max_rot_deg, max_rot_deg, generator=g))
        K = torch.zeros((b, 3, 3), device=device, dtype=torch.float64)
        K[:, 0, 1], K[:, 0, 2], K[:, 1, 0] = -axis[:, 2], axis[:, 1], axis[:, 2]
        K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -axis[:, 0], -axis[:, 1], axis[:, 0]
        eye = torch.eye(3, device=device, dtype=torch.float64).expand(b, 3, 3)
        R = eye + torch.sin(ang)[:, None, None] * K + (1 - torch.cos(ang))[:, None, None] * (K @ K)
        tdir = torch.randn((b, 3), device=device, dtype=torch.float64, generator=g)
        t = tdir / tdir.norm(dim=1, keepdim=True) * torch.empty((b, 1), device=device, dtype=torch.float64).uniform_(0, max_trans, generator=g)
        cc = torch.full((3,), cube / 2, device=device, dtype=torch.float64)
        tt = cc - (R @ cc) + t
        Ts[c0:c0 + b] = torch.eye(4, device=device, dtype=torch.float64)
        Ts[c0:c0 + b, :3, :3] = R
        Ts[c0:c0 + b, :3, 3] = tt

        def sample():
            which = torch.randint(0, n_patches, (b, n), device=device, generator=g)
            ab = torch.empty((b, n, 2), device=device).uniform_(-patch / 2, patch / 2, generator=g)
            ctr = torch.gather(centres, 1, which[..., None].expand(b, n, 3))
            fr = torch.gather(frames.reshape(b, n_patches, 9), 1, which[..., None].expand(b, n, 9)).reshape(b, n, 3, 3)
            p = ctr + ab[..., :1] * fr[..., :, 0] + ab[..., 1:] * fr[..., :, 1]
            return p + sigma * torch.randn((b, n, 3), device=device, generator=g)

        s = sample()
        q = sample().double()
        q = q @ R.transpose(1, 2) + tt[:, None, :]
        src[c0 * n:(c0 + b) * n] = s.reshape(-1, 3)
        tgt[c0 * n:(c0 + b) * n] = q.float().reshape(-1, 3)
    off = torch.arange(0, n_pairs + 1, dtype=torch.int64, device=device) * n
    return src, tgt, off, Ts
