"""GPU: a whole training run (the reference's n_step = 500) of the drop-in NerfRunner against the reference's OWN NerfRunner.train_loop
(nerf_runner.py:679-852, run verbatim on top of its own CUDA extensions, oracle/ref_train_loop.py) on the same data from the same initial
parameters, as recorded by tests/golden/make_golden_runner.py (ref_gpu_training_500.npz). The two draw different sample noise
(torch.rand there, in-kernel Philox here), so the runs are compared as what they are — two realisations of the same stochastic
optimisation: the loss level they reach, the SDF field and the surface normals they learn.

Tolerances (stated, not tuned per run): final loss within 20 %; SDF fields correlate > 0.9 and agree in sign on > 90 % of the probes inside
the truncation band; normals of the two fields within the band have a mean cosine > 0.8."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))


def test_500_steps_track_the_references_own_training(golden_dir):
    import make_golden_runner as M
    from bundlesdf_b200.nerf_runner import set_seed
    gold = np.load(os.path.join(golden_dir, 'ref_gpu_training_500.npz'))
    n_step = 500
    r = M.training_runner(n_step)
    cfg = r.cfg
    # the reference's run (tests/golden/make_golden_runner.py) started from this runner's initial parameters: 500 x train_loop, the loss of
    # every step captured at the GradScaler
    ref_losses = gold['losses']
    assert ref_losses.shape == (n_step,)

    # ---- ours: the same number of steps through train_steps (10-step graph blocks), loss read after every block
    set_seed(1)
    r.data_loader = type(r.data_loader)(r.rays, cfg['N_rand'])
    ours_losses = []
    r.train_steps(11)                                     # steps 0..10: the graph blocks of train_steps start at step 1 (mod 10), after the lr schedule's host action
    ours_losses.append(r._step_buf['losses'][0].clone())
    for _ in range((n_step - 11) // 10):                  # steps 11..20, ..., 481..490: one CUDA graph each
        r.train_steps(10)
        ours_losses.append(r._step_buf['losses'][0].clone())
    assert any(k[0] == 'blk' and k[2] == 10 for k in r._graph), list(r._graph)
    r.train_steps(n_step - r.global_step)
    assert r.global_step == n_step
    ours_losses = torch.stack(ours_losses).cpu().numpy()  # the loss of steps 10, 20, ..., 490
    r.synchronize_parameters()                            # the last step's table update + bookkeeping are still pending
    r.check_device_flags()
    assert r.adam_step_count.item() + int(r._adam_step_buf[5].item()) == n_step          # updates + skipped (inf) steps

    ref_at = ref_losses[10::10]
    first_o, first_r = ours_losses[0], ref_at[0]
    last_o, last_r = ours_losses[-10:].mean(), ref_at[-10:].mean()
    print(f'loss at step 10: ours {first_o:.5f} ref {first_r:.5f}; mean of the last 100 steps (sampled every 10): ours {last_o:.5f} ref {last_r:.5f}')
    assert last_r < 0.5 * ref_losses[0] and last_o < 0.5 * ref_losses[0]
    assert abs(last_o - last_r) <= 0.2 * last_r, (last_o, last_r)

    # ---- the fields, at the probe points the reference's field was evaluated at (a seeded sample of M.probe_points)
    pts = torch.from_numpy(gold['probe_points']).cuda()
    so = r.run_network_density(pts, get_normals=True)[0]
    sr = gold['sdf_normals']
    sdf_o, sdf_r = so[:, 0].cpu().numpy(), sr[:, 0]
    band = (np.abs(sdf_r) < 0.9) | (np.abs(sdf_o) < 0.9)
    assert band.sum() > 200, band.sum()
    corr = np.corrcoef(sdf_o[band], sdf_r[band])[0, 1]
    sign = (np.sign(sdf_o[band]) == np.sign(sdf_r[band])).mean()
    near = (np.abs(sdf_r) < 0.5) & (np.abs(sdf_o) < 0.5)
    no, nr = so[:, 1:].cpu().numpy()[near], sr[:, 1:][near]
    cos = (no * nr).sum(-1) / np.maximum(np.linalg.norm(no, axis=-1) * np.linalg.norm(nr, axis=-1), 1e-12)
    print(f'probes {len(pts)}, in band {band.sum()}: sdf correlation {corr:.4f}, sign agreement {sign:.4f}; normals on {near.sum()} probes: mean cosine {cos.mean():.4f}')
    assert corr > 0.9 and sign > 0.9, (corr, sign)
    assert cos.mean() > 0.8, cos.mean()
