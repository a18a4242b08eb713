"""GPU: nof_ray_march (bundlesdf_b200/csrc/nof_sampling.cu) against the sequential numpy oracle at every occupancy level the kernel
accepts (0-6), on the rays where a voxel walk goes wrong, with several rays per warp, and on its in-kernel Philox jitter.

The inputs are built here, not from a synthetic scene: every ray has its own frame row in `tf`, so its origin is exactly that
frame's translation. Where the world direction must be exact (axis-parallel rays, zero components, exact ties between axes) the
rotation is a signed permutation; elsewhere it is random. The references are the SEQUENTIAL walk O.ray_trace_intervals (not the
merge restatement, which is the kernel's own design) and O.sample_along_rays, fed the kernel's fp32 origins and directions
(O.rays_world_np); intervals and samples are compared bit for bit, and the error flag exactly.

Oracle cost: the walk takes ~3 * 2^level Python steps per ray and the sample walk ~S * (intervals) steps, so the ray counts
shrink with the level and the large sample counts run at level 3."""
import ctypes as C

import numpy as np
import pytest
import torch

from bundlesdf_b200 import synthetic as syn
from oracle import nof_oracle as O

pytestmark = pytest.mark.gpu

f32 = np.float32
NEAR, FAR, TRUNC, NEG_TRUNC = f32(0.25), f32(6.0), f32(0.05), 1.0
RUNNER_SEED = 0x5DEECE66D                          # NerfRunner._forward_backward's sampler seed
OCC_KINDS = ['p05', 'p30', 'p90', 'shell', 'empty', 'full']
FAMILIES = ['camera', 'inside', 'planes', 'ties', 'axis', 'zero', 'face', 'miss', 'away']


def _sm_count():
    from bundlesdf_b200 import _lib
    sm = C.c_int(0)
    _lib.check(_lib.load().nof_device_info(C.byref(sm), None), 'nof_device_info')
    return sm.value


# ------------------------------------------------------------------------------------------------------------------- inputs
def _occupancy(kind, level, seed=0):
    """[n,n,n] bool, n = 2^level: Bernoulli at 5 / 30 / 90 %, the cells an ellipsoid's surface passes through (a hollow,
    object-like shell at every level), all empty or all full."""
    n = 1 << level
    if kind == 'empty':
        return np.zeros((n, n, n), bool)
    if kind == 'full':
        return np.ones((n, n, n), bool)
    if kind.startswith('p'):
        return np.random.default_rng(seed + 100 * level).random((n, n, n)) < int(kind[1:]) / 100
    assert kind == 'shell'
    g = np.linspace(-1.0, 1.0, 2 * n + 1)                      # cell corners and centres
    x, y, z = np.meshgrid(g, g, g, indexing='ij')
    f = np.sqrt(((x - 0.05) / 0.6) ** 2 + ((y + 0.1) / 0.5) ** 2 + (z / 0.75) ** 2) - 1.0
    lo = np.full((n, n, n), np.inf)
    hi = np.full((n, n, n), -np.inf)
    for dx in range(3):
        for dy in range(3):
            for dz in range(3):
                s = f[dx:dx + 2 * n:2, dy:dy + 2 * n:2, dz:dz + 2 * n:2]
                lo, hi = np.minimum(lo, s), np.maximum(hi, s)
    return (lo <= 0) & (hi >= 0)


def _rotations(rng, k):
    q = rng.normal(size=(k, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
                     np.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], -1),
                     np.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1)], 1).astype(f32)


def _signed_perms(rng, k):
    P = np.zeros((k, 3, 3), f32)
    for i in range(k):
        P[i, np.arange(3), rng.permutation(3)] = rng.choice([-1.0, 1.0], 3)
    return P


def _family(name, k, level, occ, rng):
    """k rays of one family: (camera-frame directions [k,3], rotations [k,3,3], origins [k,3]), float32. Generic families pick the
    world ray (o, w) and a random rotation R, and give the camera direction R^T w; exact families use signed permutations, so the
    kernel's world direction is exactly R c / |c| with its zero components and equal magnitudes intact."""
    n = 1 << level
    cell = 2.0 / n
    lattice = lambda v: np.round((v + 1.0) / cell) * cell - 1.0      # nearest cell plane (exact in fp32)
    unit = lambda v: v / np.linalg.norm(v, axis=-1, keepdims=True)
    inner = lambda: rng.uniform(-0.8, 0.8, (k, 3))
    if name in ('camera', 'inside', 'planes', 'miss', 'away'):
        R = _rotations(rng, k)
        if name == 'camera':                                   # from 2-4 units away towards a point of the box
            w = unit(rng.normal(size=(k, 3)))
            o = inner() - w * rng.uniform(2.0, 4.0, (k, 1))
        elif name == 'inside':                                 # origins inside the grid; half of them at the centre of an occupied cell
            w = unit(rng.normal(size=(k, 3)))
            o = rng.uniform(-0.97, 0.97, (k, 3))
            cells = np.argwhere(occ)
            if len(cells):
                pick = cells[rng.integers(0, len(cells), k // 2)]
                o[:k // 2] = (pick + 0.5) * cell - 1.0
        elif name == 'planes':                                 # one or two coordinates on a cell plane, or a lattice point; inside and outside
            w = unit(rng.normal(size=(k, 3)))
            o = np.where(rng.random((k, 1)) < 0.5, rng.uniform(-1.0, 1.0, (k, 3)), inner() - w * rng.uniform(1.5, 3.0, (k, 1)))
            snap = rng.random((k, 3)) < np.array([[0.5, 0.5, 0.5]])
            snap[::3] = True
            o = np.where(snap, lattice(o), o)
        elif name == 'miss':                                   # passes beside the box: stays beyond |x| > 1.2 on the offset axis
            o = rng.uniform(-1.0, 1.0, (k, 3))
            a = rng.integers(0, 3, k)
            sgn = rng.choice([-1.0, 1.0], k)
            o[np.arange(k), a] = sgn * rng.uniform(1.2, 2.0, k)
            w = unit(rng.normal(size=(k, 3)))
            w[np.arange(k), a] = sgn * np.abs(w[np.arange(k), a])    # moving away from the box along that axis
            o = o - w * 3.0
            o[np.arange(k), a] = sgn * rng.uniform(1.2, 2.0, k)
        else:                                                  # 'away': outside, pointing away from a point of the box
            w = unit(rng.normal(size=(k, 3)))
            o = inner() + w * rng.uniform(2.0, 4.0, (k, 1))
        cam = np.einsum('kji,kj->ki', R.astype(np.float64), w)
        return cam.astype(f32), R, o.astype(f32)
    R = _signed_perms(rng, k)
    if name == 'ties':                                         # equal |components|: every crossing of those axes is an exact tie
        dirs = np.array([[1, 1, 0], [1, 0, -1], [1, 1, 1], [-1, 1, -1], [1, 1, -2], [-2, 1, 1]], np.float64)
        cam = dirs[np.arange(k) % len(dirs)]
        w = np.einsum('kij,kj->ki', R.astype(np.float64), cam)
        p = rng.integers(0, n + 1, (k, 3)) * cell - 1.0          # a lattice point of the box, or m half-cell steps back along the
        m = rng.integers(0, 4 * n + 1, (k, 1))                  # ray from it (outside for large m): x - p is a multiple of cell / 2
        o = p - m * cell * w / np.abs(w).max(1, keepdims=True)
        return cam.astype(f32), R, o.astype(f32)
    if name == 'axis':                                         # +-e_a in the world, both signs; half on cell edges, half entering from outside
        cam = np.tile(np.array([[0.0, 0.0, -1.0]]), (k, 1))
        w = np.einsum('kij,kj->ki', R.astype(np.float64), cam)
        o = rng.uniform(-1.0, 1.0, (k, 3))
        o[::2] = lattice(o[::2])
        a = np.abs(w).argmax(1)
        out = rng.random(k) < 0.5
        o[out, a[out]] = -np.sign(w[out, a[out]]) * rng.uniform(1.1, 3.0, out.sum())
        return cam.astype(f32), R, o.astype(f32)
    # 'zero' / 'face': one zero world component (ray parallel to a pair of faces); 'face' puts it in a box face or an inner cell plane
    xy = rng.uniform(0.2, 0.8, k) * rng.choice([-1.0, 1.0], k)
    cam = np.zeros((k, 3))
    cam[:, 2] = -1.0
    cam[np.arange(k), rng.integers(0, 2, k)] = xy
    w = unit(np.einsum('kij,kj->ki', R.astype(np.float64), cam))
    o = inner() - w * rng.uniform(0.0, 3.0, (k, 1))
    if name == 'face':
        a = np.argmin(np.abs(w), 1)
        o[np.arange(k), a] = np.where(np.arange(k) % 3 == 2, lattice(o[np.arange(k), a]), rng.choice([-1.0, 1.0], k))
    return cam.astype(f32), R, o.astype(f32)


def _rays(N, level, occ, seed, families=FAMILIES):
    """N rays cycling through the families, with the depth column cycling through valid / invalid (BAD_DEPTH) / exactly near_sc /
    exactly far_sc. Returns (batch [N,12], tf [N,12]) float32; ray r reads frame r."""
    rng = np.random.default_rng(seed)
    k = -(-N // len(families))
    parts = [_family(f, k, level, occ, rng) for f in families]
    cam = np.stack([p[0] for p in parts], 1).reshape(-1, 3)[:N]             # interleaved: ray r is family r % len(families)
    R = np.stack([p[1] for p in parts], 1).reshape(-1, 3, 3)[:N]
    o = np.stack([p[2] for p in parts], 1).reshape(-1, 3)[:N]
    tf = np.concatenate([R, o[:, :, None]], 2).reshape(N, 12).astype(f32)
    batch = np.zeros((N, 12), f32)
    batch[:, 0:3] = cam
    batch[:, 3:6] = 0.5
    batch[:, 7] = 1.0
    batch[:, 8] = np.arange(N)
    batch[:, 10], batch[:, 11] = NEAR, FAR
    # depth: a point of the ray's passage through the box (z = travel * |u_z|) for the valid rays, so that clipping bites
    u, oo, dw = O.rays_world_np(batch, tf)
    with np.errstate(divide='ignore', invalid='ignore'):
        ta, tb = (-1.0 - oo) / dw, (1.0 - oo) / dw
    t0 = np.nan_to_num(np.minimum(ta, tb), nan=-np.inf).max(1).clip(0.0)
    t1 = np.nan_to_num(np.maximum(ta, tb), nan=np.inf).min(1)
    hit = t1 > t0
    t = np.where(hit, t0 + (np.minimum(t1, 10.0) - t0) * rng.random(N), 2.0)
    depth = np.clip(np.abs(u[:, 2]) * t, NEAR, FAR)
    col = np.arange(N) % 4
    batch[:, 6] = np.select([col == 0, col == 1, col == 2], [depth, syn.BAD_DEPTH, NEAR], FAR).astype(f32)
    return batch, tf


# ------------------------------------------------------------------------------------------------------------------- kernel / oracle
def _march(batch, tf, occ, level, S_occ, S_d, I_max=None, t_rand=None, perturb=True, z_vals=None, trunc=TRUNC, **kw):
    from bundlesdf_b200 import ops
    err = torch.zeros(1, dtype=torch.int32, device='cuda')
    tr = None if t_rand is None else torch.from_numpy(np.ascontiguousarray(t_rand, f32)).cuda()
    z, inter = ops.ray_march(torch.from_numpy(batch).cuda(), torch.from_numpy(tf).cuda(), ops.pack_occupancy(occ).cuda(), level,
                             S_occ, S_d, float(trunc), float(NEAR), float(FAR), NEG_TRUNC, t_rand=tr, perturb=perturb, I_max=I_max,
                             z_vals=z_vals, want_intervals=True, err_flag=err, **kw)
    torch.cuda.synchronize()
    return z.cpu().numpy(), inter.cpu().numpy(), int(err.item())


def _oracle(batch, tf, occ, level, S_occ, S_d, I_max=None, t_rand=None):
    """(intervals [N,I_max,2], z_vals [N,S], expected error flag, untruncated interval counts [N])."""
    I_max = 3 * (1 << level) if I_max is None else I_max
    u, o, dw = O.rays_world_np(batch, tf)
    io = O.ray_trace_intervals(occ, o, dw, i_max=I_max)
    counts = (O.ray_trace_intervals(occ, o, dw)[:, :, 0] != 0).sum(1)         # packed intervals never start at 0 (stop rule)
    cfg = dict(sc_factor=1.0, N_samples=S_occ, N_samples_around_depth=S_d, near=NEAR, far=FAR, neg_trunc_ratio=NEG_TRUNC)
    zv, walk_err = O.sample_along_rays(io, u, batch[:, 6], cfg, TRUNC, t_rand)
    return io, zv, int(walk_err or bool((counts > I_max).any())), counts


def _check(batch, tf, occ, level, S_occ, S_d, I_max=None, t_rand=None, **kw):
    z, inter, err = _march(batch, tf, occ, level, S_occ, S_d, I_max=I_max, t_rand=t_rand, perturb=t_rand is not None, **kw)
    io, zv, want_err, counts = _oracle(batch, tf, occ, level, S_occ, S_d, I_max=I_max, t_rand=t_rand)
    bad = np.nonzero((inter != io).any(axis=(1, 2)))[0]
    assert len(bad) == 0, f'{len(bad)} of {len(batch)} rays with wrong intervals, first {bad[:8]}'
    bad = np.nonzero((z != zv).any(axis=1))[0]
    assert len(bad) == 0, f'{len(bad)} of {len(batch)} rays with wrong z_vals, first {bad[:8]}'
    assert err == want_err
    return z, io, counts


# ------------------------------------------------------------------------------------------------------------------- tests
N_PER_LEVEL = {0: 360, 1: 360, 2: 360, 3: 360, 4: 360, 5: 270, 6: 180}


@pytest.mark.parametrize('kind', OCC_KINDS)
@pytest.mark.parametrize('level', range(7))
def test_ray_march_matches_sequential_walk(level, kind):
    """Every level 0-6 (level 6: all MAX_EV = 6 event slots per lane, and more than 48 KB of dynamic shared memory), every
    occupancy kind, all ray families and depth kinds in one batch, I_max = 3 * 2^level (never exceeded: err_flag only from the walk)."""
    occ = _occupancy(kind, level)
    N = N_PER_LEVEL[level]
    batch, tf = _rays(N, level, occ, seed=level * 10 + OCC_KINDS.index(kind))
    t_rand = np.random.default_rng(level).random((N, 24), dtype=np.float32)
    z, io, counts = _check(batch, tf, occ, level, 16, 8, t_rand=t_rand)
    assert counts.max() <= 3 * (1 << level)
    if kind == 'full' and level > 0:
        assert (io[:, 0, 0] > 0).sum() >= N // 4          # the batch is not vacuous: many rays do collect intervals
        assert counts.max() >= 2 * (1 << level) - 1       # ... some of them across most of the grid


@pytest.mark.parametrize('level', [4, 6])
def test_ray_families_are_what_they_claim(level):
    """Guards the generator: the exact families have the zero components and ties they are meant to have, in the kernel's fp32."""
    occ = _occupancy('shell', level)
    batch, tf = _rays(90, level, occ, seed=1)
    u, o, dw = O.rays_world_np(batch, tf)
    fam = np.array([FAMILIES[i % len(FAMILIES)] for i in range(90)])
    a = np.abs(dw)
    assert ((a[fam == 'axis'] == 1.0).sum(1) == 1).all() and ((a[fam == 'axis'] == 0.0).sum(1) == 2).all()
    assert ((a[fam == 'zero'] == 0.0).sum(1) == 1).all()
    for row in a[fam == 'ties']:
        nz = row[row > 0]
        assert len(np.unique(nz)) < len(nz), row             # two equal magnitudes: exact ties between those axes
    face = fam == 'face'
    za = np.argmin(a[face], 1)
    ov = o[face][np.arange(face.sum()), za]
    assert (np.abs(ov) == 1.0).sum() >= face.sum() // 2 and (a[face][np.arange(face.sum()), za] == 0).all()
    inside = fam == 'inside'
    assert (np.abs(o[inside]) < 1).all()


SAMPLE_CASES = [
    # S_occ, S_d, z_vals view offset by one float (scalar stores)
    (1, 0, False),          # make_frame_rays' probe: one sample, no depth samples
    (3, 5, False),
    (3, 5, True),           # S % 4 == 0 but a misaligned row base: vec_ok false
    (5, 6, False),          # S % 4 != 0
    (64, 64, False),
    (128, 64, False),
]


@pytest.mark.parametrize('S_occ,S_d,shifted', SAMPLE_CASES)
def test_sample_counts_and_store_paths(S_occ, S_d, shifted):
    level = 3
    occ = _occupancy('shell', level)
    N = 90 if S_occ + S_d <= 16 else 45
    batch, tf = _rays(N, level, occ, seed=7)
    S = S_occ + S_d
    t_rand = np.random.default_rng(S).random((N, S), dtype=np.float32)
    buf = torch.full((N * S + 2,), float('nan'), device='cuda')
    z_view = buf[1:N * S + 1].view(N, S) if shifted else buf[:N * S].view(N, S)
    z, _, _ = _check(batch, tf, occ, level, S_occ, S_d, t_rand=t_rand, z_vals=z_view)
    tail = buf.cpu().numpy()
    assert np.isnan(tail[-1]) and (not shifted or np.isnan(tail[0])), 'a store outside the z_vals view'
    _check(batch, tf, occ, level, S_occ, S_d, t_rand=None)                      # no-perturb path


@pytest.mark.parametrize('level,kind,I_max', [(4, 'p90', 4), (5, 'full', 7), (6, 'p30', 1), (3, 'full', 9)])
def test_interval_overflow_truncates_and_flags(level, kind, I_max):
    """A ray that pierces more than I_max kept cells: the list is the first I_max intervals (as the oracle truncates) and err_flag is
    raised; the same rays with I_max = 3 * 2^level raise nothing."""
    occ = _occupancy(kind, level)
    N = 45 if level == 6 else 90
    batch, tf = _rays(N, level, occ, seed=3, families=['camera', 'planes', 'ties'])
    t_rand = np.random.default_rng(1).random((N, 24), dtype=np.float32)
    _, _, counts = _check(batch, tf, occ, level, 16, 8, I_max=I_max, t_rand=t_rand)
    assert (counts > I_max).any()
    _, _, err = _march(batch, tf, occ, level, 16, 8, t_rand=t_rand)
    assert err == _oracle(batch, tf, occ, level, 16, 8, t_rand=t_rand)[2] == 0


@pytest.mark.parametrize('level,kind', [(4, 'p30'), (5, 'shell')])
def test_several_rays_per_warp(level, kind):
    """More rays than 8 warps x 4 CTAs per SM: warps take a second ray, which must start from clean keep bits and counts."""
    sms = _sm_count()
    N = 32 * sms + 32 * sms // 4
    occ = _occupancy(kind, level)
    batch, tf = _rays(N, level, occ, seed=11)
    t_rand = np.random.default_rng(2).random((N, 8), dtype=np.float32)
    _, io, _ = _check(batch, tf, occ, level, 4, 4, t_rand=t_rand)
    assert (io[32 * sms:, 0, 0] > 0).sum() > 100          # second rays of their warps that do carry intervals


def test_device_truncation_scalar_matches_the_launch_constant():
    level = 4
    occ = _occupancy('shell', level)
    batch, tf = _rays(90, level, occ, seed=5)
    t_rand = np.random.default_rng(4).random((90, 24), dtype=np.float32)
    want, _, _ = _check(batch, tf, occ, level, 16, 8, t_rand=t_rand)
    tp = torch.tensor([float(TRUNC)], device='cuda')
    got, _, _ = _march(batch, tf, occ, level, 16, 8, t_rand=t_rand, trunc=0.5, trunc_ptr=tp)
    np.testing.assert_array_equal(got, want)
    other, _, _ = _march(batch, tf, occ, level, 16, 8, t_rand=t_rand, trunc=0.5)
    assert (other != want).any()                          # the truncation does reach the samples of this batch


PHILOX_CASES = [
    # seed, launch offset, device tick, S_occ, S_d, N ('sweep': more rays than one pass of the grid)
    (RUNNER_SEED, 0, 1, 16, 8, 180),
    (0x89ABCDEF_01234567, 0x00000003_FFFFFFFE, 5, 16, 8, 180),      # nonzero high words; offset + tick carries into the high word
    (RUNNER_SEED, 2, 3, 5, 6, 180),                                   # S % 4 != 0
    (RUNNER_SEED, 0, 7, 4, 4, 'sweep'),
]


@pytest.mark.parametrize('seed,offset,tick,S_occ,S_d,N', PHILOX_CASES)
def test_in_kernel_jitter_is_the_documented_philox_stream(seed, offset, tick, S_occ, S_d, N):
    """t_rand = NULL: the kernel's jitter equals O.march_uniforms(N, S, seed, offset + *offset_ptr), injected or given to the oracle."""
    level = 3
    if N == 'sweep':
        N = 32 * _sm_count() + 96
    occ = _occupancy('shell', level)
    batch, tf = _rays(N, level, occ, seed=9)
    S = S_occ + S_d
    ticks = torch.tensor([tick], dtype=torch.int64, device='cuda')
    got, _, err = _march(batch, tf, occ, level, S_occ, S_d, t_rand=None, perturb=True, seed=seed, offset=offset, offset_ptr=ticks)
    U = O.march_uniforms(N, S, seed, offset + tick)
    inj, _, _ = _march(batch, tf, occ, level, S_occ, S_d, t_rand=U)
    np.testing.assert_array_equal(got, inj)
    z, _, _ = _check(batch, tf, occ, level, S_occ, S_d, t_rand=U)
    np.testing.assert_array_equal(got, z)
    assert int(ticks.item()) == tick                      # the march reads the tick, it never advances it
    plain, _, _ = _march(batch, tf, occ, level, S_occ, S_d, t_rand=None, perturb=False)
    assert (got != plain).mean() > 0.3                    # the jitter is there


def test_runner_step_draws_jitter_at_the_tick_its_prologue_advanced():
    """NerfRunner._forward_backward without t_rand: nof_step_prologue bumps march_tick when its last CTA retires, before the ray march of
    the same step reads it (nof_pose.cu, completion ticket), so step k of a fresh runner samples with offset k (1-based)."""
    from bundlesdf_b200 import ops
    from bundlesdf_b200.nerf_runner import NerfRunner
    seq = syn.make_sequence(3, H=120, W=160, device='cuda', seed=3)
    cfg = syn.default_cfg(N_rand=256, N_samples=64, N_samples_around_depth=64, num_levels=16, finest_res=256, log2_hashmap_size=14,
                          sc_factor=seq['sc_factor'], translation=seq['translation'].tolist(), n_step=20)
    r = NerfRunner(cfg, seq['images'], seq['depths'], seq['masks'], None, seq['poses'], seq['K'], build_octree_pcd=syn.PointCloud(seq['pcd_normalized']))
    assert r.cfg['perturb']
    batch = next(r.data_loader).contiguous()
    N, S = batch.shape[0], 128
    sc = r.cfg['sc_factor']

    def march_with(tf, tick):
        U = torch.from_numpy(O.march_uniforms(N, S, RUNNER_SEED, tick)).cuda()
        return ops.ray_march(batch, tf, r.octree_m.occ_bits, r.octree_m.level, 64, 64, r.get_truncation(), r.cfg['near'] * sc,
                             r.cfg['far'] * sc, r.cfg['neg_trunc_ratio'], t_rand=U, perturb=True)

    seen = []
    for _ in range(2):
        tick0 = int(r.march_tick.item())
        b = r._forward_backward(batch)
        torch.cuda.synchronize()
        z, tf = b['z_vals'].clone(), b['tf'].clone()
        assert int(r.march_tick.item()) == tick0 + 1
        assert torch.equal(z, march_with(tf, tick0 + 1))
        assert not torch.equal(z, march_with(tf, tick0))
        seen.append(z)
    assert (seen[0] != seen[1]).float().mean() > 0.3      # the second step draws new jitter


def test_interval_walk_folds_rays_past_the_grid_y_limit():
    """sampleRaysUniformOccupiedVoxels launches once per 65535 rays: the rays of the second launch read their own samples."""
    from bundlesdf_b200.mycuda import common
    N, I, S = 70001, 4, 2
    rng = np.random.default_rng(0)
    k = rng.integers(0, I + 1, N)
    lens = rng.uniform(0.01, 0.2, (N, I)).astype(f32)
    gaps = rng.uniform(0.0, 0.1, (N, I)).astype(f32)
    a = (rng.uniform(0.1, 1.0, (N, 1)) + np.cumsum(gaps + lens, 1) - lens).astype(f32)
    b = (a + lens).astype(f32)
    io = np.where((np.arange(I)[None] < k[:, None])[..., None], np.stack([a, b], -1), f32(0)).astype(f32)
    total = np.zeros(N, f32)
    for j in range(I):
        total = (total + (io[:, j, 1] - io[:, j, 0]).astype(f32)).astype(f32)
    zs = (total[:, None] * rng.random((N, S), dtype=np.float32)).astype(f32)
    z = torch.zeros(N, S, device='cuda')
    common.sampleRaysUniformOccupiedVoxels(torch.from_numpy(io).cuda(), torch.from_numpy(zs).cuda(), z)
    want, err = O.interval_walk(io, zs)
    assert not err
    got = z.cpu().numpy()
    np.testing.assert_array_equal(got, want)
    assert (got[65535:] != 0).any(axis=1).sum() > 0.5 * (N - 65535)
