"""CPU tests of the host-side logic and of the C-ABI surface (no GPU compute)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import nof_oracle as O

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from bundlesdf_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(REPO, 'include', 'nof.h')).read()
    declared = set(re.findall(r'\b(nof_[a-z0-9_]+)\s*\(', hdr))
    assert declared, 'no declarations parsed from include/nof.h'
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/nof.h but not exported by libnof_sm100.so'
    assert set(_lib.EXPORTS) == declared
    assert lib.nof_version() == 100


def test_ctypes_struct_layouts_match_the_header():
    """sizeof(NofStep)/NofMarchCfg/NofAdamSeg as the C compiler sees them (compiled on the fly with gcc)."""
    import subprocess, tempfile
    from bundlesdf_b200 import _lib
    src = '#include <stdio.h>\n#include "nof.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n", sizeof(NofStep), sizeof(NofMarchCfg), sizeof(NofAdamSeg),' \
          ' __builtin_offsetof(NofStep, workspace), __builtin_offsetof(NofStep, loss_scale));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, 't.c'), 'w').write(src)
        subprocess.check_call(['gcc', '-I', os.path.join(REPO, 'include'), os.path.join(d, 't.c'), '-o', os.path.join(d, 't')])
        out = subprocess.check_output([os.path.join(d, 't')]).decode().split()
    assert int(out[0]) == ctypes.sizeof(_lib.NofStep)
    assert int(out[1]) == ctypes.sizeof(_lib.NofMarchCfg)
    assert int(out[2]) == ctypes.sizeof(_lib.NofAdamSeg)
    assert int(out[3]) == _lib.NofStep.workspace.offset
    assert int(out[4]) == _lib.NofStep.loss_scale.offset


def test_argument_validation_without_gpu():
    from bundlesdf_b200 import _lib
    lib = _lib.load()
    assert lib.nof_grid_encode_forward(None, None, None, None, 1, 3, 2, 16, 0.5, 16, 0, None, 0, 0, 0, None) == -1
    assert b'null pointer' in lib.nof_last_error()
    assert lib.nof_adam_step(None, 0, 0.9, 0.999, 1e-15, None, None, None, None, None) == -1
    with pytest.raises(_lib.NofError):
        _lib.ptr(torch.zeros(3))            # CPU tensor: the product path has no CPU fallback


def test_mlp_param_layout():
    from bundlesdf_b200 import ops
    count, offs = ops.mlp_param_layout(32, 9)
    assert offs == [0, 2048, 2112, 3136, 3152, 4688, 4752, 8848, 8912, 9104]
    assert count == 9108 and count % 4 == 0


def test_product_never_imports_the_oracle():
    bad = []
    for root, _, files in os.walk(os.path.join(REPO, 'bundlesdf_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.cpp', '.h')):
                txt = open(os.path.join(root, f), errors='ignore').read()
                if re.search(r'^\s*(from|import)\s+oracle\b', txt, re.M) or 'nof_oracle' in txt or 'oracle/' in txt:
                    bad.append(os.path.join(root, f))
    assert not bad, f'product files referencing oracle/: {bad}'


def test_pack_occupancy_bit_order():
    from bundlesdf_b200 import ops
    occ = np.zeros((4, 4, 4), bool)
    occ[0, 0, 0] = occ[0, 0, 3] = occ[1, 2, 3] = occ[3, 3, 3] = True
    words = ops.pack_occupancy(occ).numpy().view(np.uint32)
    for cid in range(64):
        ix, iy, iz = cid // 16, (cid // 4) % 4, cid % 4
        assert bool((words[cid >> 5] >> (cid & 31)) & 1) == bool(occ[ix, iy, iz])


def test_occupancy_build_matches_oracle():
    from bundlesdf_b200 import synthetic as syn
    from bundlesdf_b200.occupancy import OctreeManager, build_occupancy_points
    seq = syn.make_sequence(3, H=60, W=80, seed=1)
    cfg = syn.default_cfg(sc_factor=seq['sc_factor'])
    want, level = O.build_occupancy(seq['pcd_normalized'], cfg)
    centers, max_level, lvl = build_occupancy_points(torch.tensor(seq['pcd_normalized']).float(), cfg)
    assert lvl == level
    # OctreeManager packs bits through ops (CPU ok) — ray tracing itself needs the GPU
    om = OctreeManager(centers, max_level, level=lvl, device=torch.device('cpu'))
    np.testing.assert_array_equal(om.occ.numpy(), want)
    om2 = OctreeManager(octree=om.octree, device=torch.device('cpu'))
    np.testing.assert_array_equal(om2.occ.numpy(), want)


def test_dataloader_order_matches_reference(golden_dir):
    from bundlesdf_b200.nerf_runner import DataLoader, set_seed
    g = np.load(os.path.join(golden_dir, 'ref_py_misc.npz'))
    set_seed(0)
    dl = DataLoader(rays=torch.arange(23).float().reshape(-1, 1), batch_size=5)
    got = [dl.next_ids().numpy().copy() for _ in range(9)]
    np.testing.assert_array_equal(np.stack(got), g['dl_order'].astype(np.int64))


def test_model_state_dict_keys_match_reference(golden_dir):
    from bundlesdf_b200.nerf_helpers import NeRFSmall
    g = np.load(os.path.join(golden_dir, 'ref_py_mlp_L16.npz'))
    m = NeRFSmall(num_layers=2, hidden_dim=64, geo_feat_dim=15, num_layers_color=3, hidden_dim_color=64, input_ch=32, input_ch_views=9)
    ref_keys = sorted(k[2:] for k in g.files if k.startswith('p_'))
    assert sorted(m.state_dict().keys()) == ref_keys
    # same init stream as the reference for the same seed (make_golden_cpu.py used torch.manual_seed(7))
    torch.manual_seed(7)
    m = NeRFSmall(num_layers=2, hidden_dim=64, geo_feat_dim=15, num_layers_color=3, hidden_dim_color=64, input_ch=32, input_ch_views=9)
    for k, v in m.state_dict().items():
        np.testing.assert_array_equal(v.numpy(), g['p_' + k])
    x = torch.from_numpy(g['x'])
    np.testing.assert_allclose(m(x).detach().numpy(), g['y'], rtol=1e-5, atol=1e-6)


def test_camera_rays_match_reference(golden_dir):
    from bundlesdf_b200.nerf_helpers import get_camera_rays_np
    g = np.load(os.path.join(golden_dir, 'ref_py_misc.npz'))
    np.testing.assert_array_equal(get_camera_rays_np(8, 10, g['K']), g['dirs'])


def test_nerf_runner_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    from bundlesdf_b200 import synthetic as syn
    from bundlesdf_b200._lib import NofError
    from bundlesdf_b200.nerf_runner import NerfRunner
    with pytest.raises(NofError):
        NerfRunner(syn.default_cfg(), None, None, None, None, None, np.eye(3), build_octree_pcd=syn.PointCloud(np.zeros((1, 3))))


def test_ray_walk_as_merge_of_axis_crossings_is_bit_identical():
    """Design check for a warp-parallel ray march (DESIGN.md §8-3): the voxel walk restated as the merge of three closed-form
    per-axis crossing lists gives exactly the sequential walk's intervals, including axis-aligned rays, rays with zero components,
    origins inside the grid and origins on cell planes."""
    rng = np.random.default_rng(0)
    for n in (8, 16, 32):
        occ = rng.random((n, n, n)) < 0.3
        N = 300
        o = (rng.random((N, 3)) * 3 - 1.5).astype(np.float32)
        tgt = (rng.random((N, 3)) * 1.6 - 0.8).astype(np.float32)
        d = tgt - o
        d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
        d[:30] = np.eye(3, dtype=np.float32)[rng.integers(0, 3, 30)] * rng.choice([-1, 1], (30, 1)).astype(np.float32)
        d[30:60, rng.integers(0, 3)] = 0
        nn = np.linalg.norm(d[30:60], axis=1, keepdims=True)
        d[30:60] = (d[30:60] / np.where(nn == 0, 1, nn)).astype(np.float32)
        o[60:150] = (rng.random((90, 3)) * 1.8 - 0.9).astype(np.float32)
        o[150:180] = np.round(o[150:180] * n / 2) / (n / 2)
        a = O.ray_trace_intervals(occ, o, d)
        b = O.ray_trace_intervals_merge(occ, o, d, i_max=a.shape[1])
        np.testing.assert_array_equal(a, b)
        assert (a[:, 0, 0] != 0).sum() > N // 2


def test_reference_shims_reimport_once_the_extensions_are_there(tmp_path):
    """tests/golden/ref_shims.import_reference: the CPU-side golden generators import the reference WITHOUT its CUDA extensions (its
    `from mycuda import common` then fails silently); a later import WITH them (oracle/ref_train_loop.py on a GPU) has to
    produce fresh modules that see the extensions, or the reference's train_loop dies on `common`. The modules here are stand-ins with
    the reference's import chain (Utils.py:28-31 imports `common` under try/except; nerf_helpers and nerf_runner star-import Utils)."""
    import sys
    import types
    (tmp_path / 'Utils.py').write_text('try:\n    from mycuda import common\nexcept Exception:\n    pass\n')
    (tmp_path / 'nerf_helpers.py').write_text('from Utils import *\n')
    (tmp_path / 'nerf_runner.py').write_text('from nerf_helpers import *\nfrom Utils import *\n')
    ref_dir = str(tmp_path)
    sys.path.insert(0, os.path.join(REPO, 'tests', 'golden'))
    import ref_shims
    saved = {k: sys.modules.get(k) for k in ('Utils', 'nerf_helpers', 'nerf_runner', 'mycuda', 'mycuda.common', 'gridencoder')}
    for k in ('Utils', 'nerf_helpers', 'nerf_runner'):
        sys.modules.pop(k, None)
    try:
        _, nr_plain, _ = ref_shims.import_reference(ref_dir)
        assert not hasattr(nr_plain, 'common')
        fake_c, fake_g = types.ModuleType('common_fake'), types.ModuleType('gridencoder_fake')
        _, nr_ext, _ = ref_shims.import_reference(ref_dir, mycuda_common=fake_c, mycuda_gridencoder=fake_g)
        assert nr_ext is not nr_plain and nr_ext.common is fake_c
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        sys.path.remove(ref_dir)


def test_device_cursor_protocol_walks_the_same_batches_as_the_per_step_loader():
    """DataLoader.reserve / consumed (what NerfRunner.train_steps drives: k batches read at a device cursor by one CUDA graph) against
    next_ids() (the reference's per-step protocol, nerf_runner.py:90-107): same permutation, same batch boundaries, same reshuffle points —
    including the reference's rule that the last batch of an epoch is dropped when `pos + batch_size < len(ids)` fails."""
    from bundlesdf_b200.nerf_runner import DataLoader, set_seed
    rays = torch.arange(1003 * 12, dtype=torch.float32).reshape(1003, 12)        # 1003 rays, batches of 100: 10 per epoch, 3 rays dropped
    set_seed(5)
    a = DataLoader(rays, 100)
    ids_a = []
    for _ in range(37):
        a.next_ids()
        ids_a.append(a.batch_ray_ids.clone())
    set_seed(5)
    b = DataLoader(rays, 100)
    ids_b, want = [], [4, 4, 10, 1, 7, 10, 1]                # block lengths a caller may ask for, crossing epoch boundaries
    done = 0
    while done < 37:
        k = b.reserve(min(want[len(ids_b) % len(want)], 37 - done))
        assert k >= 1
        assert int(b.cursor_dev.item()) == b.pos
        for j in range(k):                                   # what the k prologues of the graph read at the device cursor
            cur = int(b.cursor_dev.item())
            ids_b.append(b.ids_dev[cur: cur + 100].clone())
            b.cursor_dev += 100                              # nof_step_prologue advances the cursor when its last block retires
        b.consumed(k)
        assert torch.equal(b.batch_ray_ids, ids_b[-1])
        done += k
    assert len(ids_b) >= 37
    for x, y in zip(ids_a, ids_b[:37]):
        assert torch.equal(x, y)
    assert a.pos == b.pos


@pytest.mark.parametrize('decay', ['', 'linear', 'exp'])
def test_truncation_schedule_matches_the_references_own_method(golden_dir, decay):
    """get_truncation (nerf_runner.py:663-676): the product's host formula (which also fills the device table of the annealed schedule) and the
    oracle's, against the reference's own NerfRunner.get_truncation called on a stand-in self — every step of a 500-step run, bit for bit."""
    import types
    from bundlesdf_b200.nerf_runner import NerfRunner
    from oracle import nof_oracle as O
    gold = np.load(os.path.join(golden_dir, 'ref_py_truncation.npz'))   # tests/golden/make_golden_runner.py
    cfg = dict(trunc_decay_type=decay, trunc_start=0.03, trunc=0.01, n_step=500, sc_factor=3.7)
    steps, wants = gold['steps'], gold['trunc_' + (decay or 'const')]
    assert list(steps) == list(range(0, 40)) + [123, 124, 125, 126, 250, 499, 500, 501]
    for g, want in zip(steps.tolist(), wants.tolist()):
        me = types.SimpleNamespace(cfg=cfg, global_step=g)
        assert NerfRunner.get_truncation(me) == want
        assert NerfRunner.get_truncation(me, step=g) == want
        assert O.get_truncation(cfg, g) == want
