"""Golden vectors of the reference's own NerfRunner methods that the runner tests compare against, so that those tests need
neither the reference's sources nor its compiled extensions:

    python tests/golden/make_golden_runner.py [OUT_DIR]        (default: tests/golden; needs a B200 and oracle/_ref)

  ref_py_truncation.npz      NerfRunner.get_truncation (nerf_runner.py:663-676) on a stand-in self, every decay type
                             -> tests/test_host_logic.py
  ref_gpu_frame_rays.npz     NerfRunner.make_frame_rays (nerf_runner.py:246-316) of frames 0 and 2 of a seeded synthetic
                             sequence: row count, per-column sums and a seeded sample of the rows -> tests/test_gpu_raypool.py
  ref_gpu_training_500.npz   500 x the reference's train_loop on its own extensions (oracle/ref_train_loop.py), started from the
                             product's initial parameters: the loss of every step, and the SDF and normals of the trained field at a
                             seeded sample of probe points -> tests/test_gpu_reference_training.py

The scenes are rebuilt by the tests from the same seeds (bundlesdf_b200.synthetic), so only the reference's results are stored."""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)

TRUNC_CFG = dict(trunc_start=0.03, trunc=0.01, n_step=500, sc_factor=3.7)
TRUNC_STEPS = list(range(0, 40)) + [123, 124, 125, 126, 250, 499, 500, 501]
FRAME_RAYS_FRAMES = (0, 2)
FRAME_RAYS_SAMPLE = 256
TRAINING_PROBES = 3000


def frame_rays_runner(denoise):
    """The scene and runner of tests/test_gpu_raypool.py."""
    from bundlesdf_b200 import synthetic as syn
    from bundlesdf_b200.nerf_runner import NerfRunner
    seq = syn.make_sequence(4, H=120, W=160, device='cuda', seed=5, pose_noise=True)
    cfg = syn.default_cfg(N_rand=128, N_samples=32, N_samples_around_depth=32, num_levels=4, finest_res=128, log2_hashmap_size=12,
                          sc_factor=seq['sc_factor'], translation=seq['translation'].tolist(), denoise_depth_use_octree_cloud=denoise)
    r = NerfRunner(cfg, seq['images'], seq['depths'], seq['masks'], None, seq['poses'], seq['K'], build_octree_pcd=syn.PointCloud(seq['pcd_normalized']))
    return r, seq


def frame_rays_sample(n_rows):
    """Row indices of the stored sample of a frame's [n_rows, 12] rays."""
    return np.sort(np.random.default_rng(0).choice(n_rows, size=min(n_rows, FRAME_RAYS_SAMPLE), replace=False))


def training_runner(n_step=500):
    """The scene and runner of tests/test_gpu_reference_training.py."""
    from bundlesdf_b200 import synthetic as syn
    from bundlesdf_b200.nerf_runner import NerfRunner, set_seed
    set_seed(0)
    seq = syn.make_sequence(6, H=120, W=160, device='cuda', seed=3, pose_noise=True)
    cfg = syn.default_cfg(N_rand=512, N_samples=64, N_samples_around_depth=64, num_levels=16, finest_res=256, log2_hashmap_size=14, amp=True,
                          sc_factor=seq['sc_factor'], translation=seq['translation'].tolist(), n_step=n_step, defer_table_update=True)
    return NerfRunner(cfg, seq['images'], seq['depths'], seq['masks'], None, seq['poses'], seq['K'], build_octree_pcd=syn.PointCloud(seq['pcd_normalized']))


def probe_points(r, step=0.04):
    """Lattice points of the normalised cube that fall into occupied cells (what extract_mesh sweeps, nerf_runner.py:1351-1380)."""
    ax = np.arange(-1 + 0.5 * step, 1, step, dtype=np.float32)
    g = torch.tensor(np.stack(np.meshgrid(ax, ax, ax, indexing='ij'), -1).reshape(-1, 3)).cuda()
    return g[r.octree_m.get_center_ids(g) >= 0]


def truncation(nr):
    out = {'steps': np.array(TRUNC_STEPS, np.int64)}
    for decay in ('', 'linear', 'exp'):
        cfg = dict(TRUNC_CFG, trunc_decay_type=decay)
        out['trunc_' + (decay or 'const')] = np.array([nr.NerfRunner.get_truncation(types.SimpleNamespace(cfg=cfg, global_step=g))
                                                       for g in TRUNC_STEPS], np.float64)
    return out


def frame_rays(nr):
    ours, _ = frame_rays_runner(False)
    fake = types.SimpleNamespace(masks=ours.masks, images=ours.images, depths=ours.depths, poses=np.asarray(ours.poses), K=ours.K, H=ours.H, W=ours.W,
                                 cfg=ours.cfg, occ_masks=None, normal_maps=None, octree_m=ours.octree_m)
    out = {}
    for fid in FRAME_RAYS_FRAMES:
        want = np.asarray(nr.NerfRunner.make_frame_rays(fake, fid), np.float64)
        out[f'n_rows_{fid}'] = np.int64(want.shape[0])
        out[f'col_sum_{fid}'] = want.sum(0)
        out[f'col_abs_sum_{fid}'] = np.abs(want).sum(0)
        out[f'rows_{fid}'] = want[frame_rays_sample(want.shape[0])]
    return out


def training(n_step=500):
    from bundlesdf_b200.nerf_runner import set_seed
    from oracle import ref_train_loop as RT
    r = training_runner(n_step)
    ref = RT.build_reference_runner(r)                    # the reference's own create_nerf / create_optimizer / GradScaler(65536)
    with torch.no_grad():                                 # same starting point as the product's runner: its initial parameters
        ref.models['embed_fn'].embeddings.copy_(r.table)
        ref.models['model'].load_state_dict(r.models['model'].state_dict())
    losses = []
    real_scale = ref.amp_scaler.scale

    def scale(loss):                                      # the loss of every step, captured at the GradScaler
        losses.append(loss.detach().float())
        return real_scale(loss)
    ref.amp_scaler.scale = scale
    set_seed(1)
    ref.data_loader = RT.reference_modules()[1].DataLoader(rays=ref.rays, batch_size=r.cfg['N_rand'])
    for _ in range(n_step):
        batch = next(ref.data_loader)
        ref.data_loader.batch_ray_ids = ref.data_loader.batch_ray_ids.to(batch.device)      # torch >= 2 indexing rule, see oracle/ref_train_loop.py
        ref.train_loop(batch)
        ref.global_step += 1
    pts = probe_points(r)
    sel = np.sort(np.random.default_rng(0).choice(len(pts), size=min(len(pts), TRAINING_PROBES), replace=False))
    pts = pts[torch.from_numpy(sel).to(pts.device)]
    sn = ref.run_network_density(pts.clone(), get_normals=True)[0].detach()
    sdf = sn[:, 0].cpu().numpy()
    print(f'training: {len(sel)} probes, {(np.abs(sdf) < 0.9).sum()} with |sdf| < 0.9; loss {float(losses[0]):.5f} -> {float(losses[-1]):.5f}')
    return {'losses': torch.stack(losses).cpu().numpy(), 'probe_points': pts.cpu().numpy(), 'sdf_normals': sn.float().cpu().numpy()}


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out_dir, exist_ok=True)
    from oracle import ref_train_loop as RT
    torch.cuda.set_device(0)
    _, nr, _ = RT.reference_modules()
    for name, fn in (('ref_py_truncation', lambda: truncation(nr)), ('ref_gpu_frame_rays', lambda: frame_rays(nr)),
                     ('ref_gpu_training_500', training)):
        cap = fn()
        path = os.path.join(out_dir, name + '.npz')
        np.savez_compressed(path, **cap)
        print(path, os.path.getsize(path), {k: getattr(v, 'shape', v) for k, v in cap.items()})


if __name__ == '__main__':
    main()
