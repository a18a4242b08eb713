"""GPU: the device-side ray-pool construction (SURVEY 8(f)-3) against the REFERENCE's own functions:
  NerfRunner.make_frame_rays (nerf_runner.py:246-316) incl. compute_near_far_and_filter_rays (:39-65) and the cv2 mask dilation, through
  golden rows made by the reference's Python (tests/golden/make_golden_runner.py -> ref_gpu_frame_rays.npz),
  and the octree-cloud denoise of __init__ (:178-195, inline there: restated with the same scipy cKDTree call).
The occupancy trace inside make_frame_rays goes through the product's OctreeManager in both (kaolin is absent)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))


def _runner(denoise):
    import make_golden_runner as M
    return M.frame_rays_runner(denoise)


def test_make_frame_rays_matches_the_reference(golden_dir):
    import make_golden_runner as M
    g = np.load(os.path.join(golden_dir, 'ref_gpu_frame_rays.npz'))
    ours, seq = _runner(False)
    for fid in M.FRAME_RAYS_FRAMES:
        got = ours.make_frame_rays(fid).cpu().numpy().astype(np.float64)
        n = int(g[f'n_rows_{fid}'])
        assert got.shape == (n, 12) and n > 500, (got.shape, n)
        # fp32 on the device vs fp64 numpy; same rows in the same order: a seeded sample row by row, every row through the column sums
        np.testing.assert_allclose(got[M.frame_rays_sample(n)], g[f'rows_{fid}'], rtol=2e-5, atol=2e-5)
        tol = 2e-5 * (n + g[f'col_abs_sum_{fid}'])
        for have, want in ((got.sum(0), g[f'col_sum_{fid}']), (np.abs(got).sum(0), g[f'col_abs_sum_{fid}'])):
            assert (np.abs(have - want) <= tol).all(), (fid, have, want)


def test_octree_cloud_denoise_matches_ckdtree():
    from scipy.spatial import cKDTree
    ours, seq = _runner(False)
    sc = ours.cfg['sc_factor']
    rays = torch.cat([ours.make_frame_rays(i) for i in range(4)], 0)
    # push a tenth of the depths off the surface so that the filter has something to remove
    g = torch.Generator(device='cpu').manual_seed(1)
    off = torch.rand(len(rays), generator=g).to(rays.device) < 0.1
    rays[off, 6] += 0.05 * sc
    got = ours._denoise_rays(rays.clone()).cpu().numpy()
    # the reference's lines (nerf_runner.py:178-195) on the same rows
    r = rays.cpu().numpy().astype(np.float64)
    mask = (r[:, 7] > 0) & (r[:, 6] <= ours.cfg['far'] * sc)
    pts = r[mask][:, 0:3] * r[mask][:, 6:7]
    fid = r[mask][:, 8].astype(int)
    P = np.asarray(ours.poses)
    pts_w = (P[fid] @ np.concatenate([pts, np.ones((len(pts), 1))], 1)[..., None])[:, :3, 0]
    d, _ = cKDTree(ours.build_octree_pts).query(pts_w, k=1)
    bad = d > 0.02 * sc
    margin = np.abs(d - 0.02 * sc) < 1e-5                                         # fp32-vs-fp64 ties
    keep = np.ones(len(r), bool)
    keep[np.arange(len(r))[mask][bad]] = False
    want = r[keep]
    assert bad.sum() > 50 and abs(len(got) - len(want)) <= int(margin.sum())
    if len(got) == len(want):
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)
