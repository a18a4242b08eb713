#!/usr/bin/env python
"""bench.py — Neural-Object-Field train-step throughput (BASELINE.json metric: NeRF train rays/s, steps/s, % HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2|C1|C3|C5] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] "C2" — milk-jug-shaped synthetic sequence, 200 frames 640x480,
2048 rays x 128 samples (64 occupied-voxel + 64 around-depth), hash grid L=16 T=2^19 finest 256, MLP = the reference
NeRFSmall (SDF 2x64, colour 3x64), AMP on, pose refinement on. A step = one NerfRunner.train_loop (gather batch from the
ray pool -> pose correction -> ray march -> fused forward/loss/backward -> pose backward -> Adam).
  value : rays/s with the ray pool resident in HBM: K = --steps timed steps (NerfRunner.train_steps: one CUDA graph per 10 steps,
          batch cursor on the device), CUDA-event timed between barrier + synchronize; the max over ranks.
  e2e   : same metric through the public API from HOST buffers, K more timed steps: every step copies its batch from pinned host
          memory (what the reference does after add_new_frames, nerf_runner.py:431: rays live on the CPU) and reads the loss back.
  --dump-outputs DIR : after the K timed steps of `value`, what a caller of train_steps has from the last of them, as DIR/<name>.npy
          (float32): the step's loss terms and the trained parameters, the hash table as a fixed seeded sample of its rows. The
          workload and the number of steps before the dump depend on the arguments only, so two builds can be compared output for output.
  roofline : the fused step kernel alone, algorithmic bytes P*64*L*C + N*60 (SURVEY.md 8d) / its mean launch time (`achieved`, `frac`);
          the whole step incl. the 34 B/param Adam stream (`achieved_step`, `frac_step`); `traffic` = ncu dram bytes of this config.
  cpu_baseline : the oracle port (oracle/nof_oracle.py, torch fp32 on all host cores) at the workload's full batch (fewer steps).
  reference_cuda : the reference's own train_loop + its own CUDA extensions (oracle/_ref) on the same GPU (rank 0, N=1 only).
  config4 : under torchrun, additionally BASELINE.json configs[3] = C3 x N sequences.
Multi-GPU (torchrun): one independent sequence per rank, NCCL only for barrier + gather of the timings ("weak" scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

CONFIGS = {
    # name: frames, N_rand, S_occ, S_depth, L, finest, log2T, optimize_poses, pose_noise, frame_stride
    'C1': dict(frames=1, N=1024, S_occ=32, S_d=32, L=4, finest=128, log2T=22, pose=0, noise=False, stride=1),
    'C2': dict(frames=200, N=2048, S_occ=64, S_d=64, L=16, finest=256, log2T=19, pose=1, noise=False, stride=1),
    'C3': dict(frames=20, N=4096, S_occ=64, S_d=64, L=16, finest=256, log2T=19, pose=1, noise=True, stride=50),
    'C5': dict(frames=300, N=8192, S_occ=128, S_d=64, L=16, finest=512, log2T=22, pose=1, noise=False, stride=1, eik=0.1),
}
WORKLOAD = {
    'C1': 'C1: single 640x480 synthetic RGBD frame, 1024 rays x 64 samples, hash L=4, MLP 2x64/3x64',
    'C2': 'C2: milk-jug synthetic sequence, 200 frames 640x480, 2048 rays x 128 samples, hash L=16 T=2^19, MLP 2x64/3x64, 1xB200',
    'C3': 'C3: HO3D-shaped synthetic, 640x480, 1000-frame orbit, 20-frame memory pool, 4096 rays x 128 samples, pose refinement on',
    'C5': 'C5: global-refine mode, 300 frames, 8192 rays x 192 samples, hash L=16 T=2^22, eikonal on (weight 0.1)',
}


DEFER_TABLE = os.environ.get('NOF_DEFER_TABLE', '1') != '0'   # overlap the table's Adam pass with the next step's ray march


def make_cfg(c):
    from bundlesdf_b200 import synthetic as syn
    return syn.default_cfg(N_rand=c['N'], N_samples=c['S_occ'], N_samples_around_depth=c['S_d'], num_levels=c['L'], finest_res=c['finest'],
                           log2_hashmap_size=c['log2T'], optimize_poses=c['pose'], amp=True, n_step=2000, denoise_depth_use_octree_cloud=True,
                           defer_table_update=DEFER_TABLE, eikonal_weight=c.get('eik', 0.0))


def algorithmic_bytes(c):
    """SURVEY.md §8(d): 64*L*C B/point with pose refinement (48*L*C without; + 16*L*C for the eikonal term's re-gather) + 60 B/ray."""
    P = c['N'] * (c['S_occ'] + c['S_d'])
    per_pt = ((64 if c['pose'] else 48) + (16 if c.get('eik', 0) > 0 else 0)) * c['L'] * 2
    return P * per_pt + c['N'] * 60


def optimizer_bytes(n_params):
    """SURVEY.md §8(d): dense Adam 28 B/param + 4 B/param gradient clear (the fp16 shadow refresh, 2 B/param, is ours and not counted)."""
    return 32 * int(n_params)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line) through NVML (the library
    behind nvidia-smi) every 25 ms — rarely enough that a query (50 us .. 2 ms of host time) does not land in every step (polling
    every 2 ms inside a 6 ms region once halved the 8-GPU headline); a region shorter than 25 ms gets one sample. Falls back to
    spawning `nvidia-smi --query-gpu=clocks.sm,...` when pynvml is not importable."""

    REASONS = ((0x8, 'hw_slowdown'), (0x40, 'hw_thermal_slowdown'), (0x20, 'sw_thermal_slowdown'), (0x4, 'sw_power_cap'))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt, self.error, self.source = index, [], threading.Event(), None, None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:                                            # honour CUDA_VISIBLE_DEVICES remapping: look the device up by UUID
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._nvml, self._h, self.source = pynvml, h, 'nvml'
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception as e:
            self.error = repr(e)[:200]

    def _sample_nvml(self):
        nv, h = self._nvml, self._h
        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        try:
            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        self.rows.append((sm, self.sm_max, mask))

    def _sample_smi(self):
        r = subprocess.run(['nvidia-smi', f'--id={self.index}', '--query-gpu=clocks.sm,clocks.max.sm,clocks_throttle_reasons.active',
                            '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
        f = [x.strip() for x in r.stdout.strip().split(',')]
        if r.returncode == 0 and len(f) >= 2 and f[0].replace('.', '').isdigit():
            mask = int(f[2], 16) if len(f) > 2 and f[2].lower().startswith('0x') else 0
            self.rows.append((float(f[0]), float(f[1]), mask))
        else:
            self.error = (r.stdout.strip() or r.stderr.strip())[:200]

    def run(self):
        self.source = self.source or 'nvidia-smi'
        while not self._stop_evt.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception as e:
                self.error = repr(e)[:200]
            self._stop_evt.wait(0.025 if self._nvml is not None else 0.2)

    def summary(self):
        self._stop_evt.set()
        self.join(timeout=6)
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable'], 'error': self.error}
        sm = sorted(r[0] for r in self.rows)
        mask = 0
        for r in self.rows:
            mask |= r[2]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': self.rows[0][1], 'reasons': [n for bit, n in self.REASONS if mask & bit],
                'samples': len(self.rows), 'source': self.source}


def build_runner(c, seed, device, eager=False):
    from bundlesdf_b200 import synthetic as syn
    from bundlesdf_b200.nerf_runner import NerfRunner
    total = c['frames'] * c['stride'] if c['stride'] > 1 else None
    seq = syn.make_sequence(c['frames'], H=480, W=640, device=device, seed=seed, pose_noise=c['noise'], frame_stride=c['stride'], total_frames=total)
    cfg = make_cfg(c)
    cfg['sc_factor'] = seq['sc_factor']
    cfg['translation'] = seq['translation'].tolist()
    cfg['use_cuda_graph'] = not eager
    runner = NerfRunner(cfg, seq['images'], seq['depths'], seq['masks'], None, seq['poses'], seq['K'], build_octree_pcd=syn.PointCloud(seq['pcd_normalized']))
    return runner, seq


def rank_seed(base_seed, rank):
    """Sequence seed of a rank: independent sequences, one per GPU (SURVEY.md §8e)."""
    return int(base_seed) + int(rank)


def aggregate_throughput(units_local, seconds_local, world, device='cpu'):
    """Whole-job throughput = units processed by ALL ranks / MAX over ranks of the elapsed time. No data-path collective:
    one all_reduce(MAX) of a scalar and one all_reduce(SUM) of the unit counts."""
    if world == 1:
        return units_local / seconds_local, seconds_local
    import torch.distributed as dist
    t = torch.tensor([seconds_local], dtype=torch.float64, device=device)
    u = torch.tensor([float(units_local)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(u, op=dist.ReduceOp.SUM)
    return float(u.item()) / float(t.item()), float(t.item())


def time_steps(fn, n):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(n):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / 1e3


_CPU_SCENE = {}


def _cpu_scene(c, seed):
    from oracle import nof_oracle as O
    from bundlesdf_b200 import synthetic as syn
    n_frames = min(c['frames'], 8)
    seq = syn.make_sequence(n_frames, H=480, W=640, device='cpu', seed=seed, pose_noise=c['noise'])
    cfg = make_cfg(c)
    cfg['sc_factor'] = seq['sc_factor']
    rng = np.random.default_rng(seed)
    K = seq['K']
    rows = []
    for f in range(n_frames):
        vs, us = np.nonzero(seq['masks'][f, ..., 0])
        sel = rng.choice(len(vs), size=min(len(vs), 4096), replace=False)
        vs, us = vs[sel], us[sel]
        r = np.zeros((len(vs), 12), np.float32)
        r[:, 0] = (us - K[0, 2]) / K[0, 0]; r[:, 1] = -(vs - K[1, 2]) / K[1, 1]; r[:, 2] = -1
        r[:, 3:6] = seq['images'][f, vs, us]; r[:, 6] = seq['depths'][f, vs, us, 0]; r[:, 7] = 1; r[:, 8] = f; r[:, 10] = 0.5; r[:, 11] = 8.0
        rows.append(r)
    pool = torch.from_numpy(np.concatenate(rows, 0))
    occ, level = O.build_occupancy(seq['pcd_normalized'], cfg)
    return seq, cfg, pool, occ, level, n_frames


_CPU_THREADS = None


def pick_cpu_threads(c):
    """All host cores unless fewer are faster: the step is a chain of small torch ops whose OpenMP fork/join cost grows with the
    thread count (128 threads on the GPU box are ~60x slower than 16 for this workload). One probe step per candidate."""
    global _CPU_THREADS
    if _CPU_THREADS is None:
        n = os.cpu_count() or 1
        best, best_t = n, None
        # more than 32 threads only ever lost on this workload (128 threads: 70 s per 256-ray step on the B200 host), so the
        # probe stays within {8, 16, 32} to keep the default bench run short
        for cand in sorted({min(n, 64), min(n, 32), min(n, 16), min(n, 8)}, reverse=True):
            t, _ = cpu_baseline_run(c, 1, 0, 256, threads=cand)
            if best_t is None or t < best_t:
                best, best_t = cand, t
        _CPU_THREADS = best
    return _CPU_THREADS


def cpu_baseline_run(c, steps, warmup, sample_rays, seed=0, threads=None):
    """The oracle port timed on the host cores: full train step (sampling, encode, MLP, losses, backward, Adam) on
    `sample_rays` rays of the workload per step."""
    from oracle import nof_oracle as O
    from bundlesdf_b200 import synthetic as syn
    torch.set_num_threads(threads or pick_cpu_threads(c))
    key = (c['frames'], c['noise'], seed)
    if key not in _CPU_SCENE:
        _CPU_SCENE[key] = _cpu_scene(c, seed)
    seq, cfg, pool, occ, level, n_frames = _CPU_SCENE[key]
    rng = np.random.default_rng(seed)
    offsets, pls = O.grid_offsets(c['L'], 16, c['finest'], c['log2T'])
    g = torch.Generator().manual_seed(seed)
    P = {'embeddings': ((torch.rand(int(offsets[-1]), 2, generator=g) * 2 - 1) * 1e-4).requires_grad_(True), 'offsets': offsets,
         'S': float(np.log2(pls)), 'H': 16}
    for k, v in O.init_mlp(c['L'] * 2, 9, seed=seed).items():
        P[k] = v.requires_grad_(True)
    P['pose_data'] = torch.zeros(n_frames, 6, requires_grad=True) if c['pose'] else None
    P['feature_data'] = None
    leaves = [v for v in P.values() if torch.is_tensor(v) and v.requires_grad]
    state = [(torch.zeros_like(p), torch.zeros_like(p)) for p in leaves]
    c2w = torch.from_numpy(seq['poses']).float()
    S = c['S_occ'] + c['S_d']
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        ids = torch.from_numpy(rng.choice(len(pool), size=sample_rays, replace=False))
        batch = pool[ids]
        t_rand = rng.random((sample_rays, S), dtype=np.float32)
        out = O.forward_step(P, batch, c2w, occ, cfg, t_rand_occ=t_rand[:, :c['S_occ']], t_rand_depth=t_rand[:, c['S_occ']:])
        for p in leaves:
            p.grad = None
        out['loss'].backward()
        with torch.no_grad():
            for p, (m, v) in zip(leaves, state):
                O.adam_update(p, p.grad, m, v, it + 1, 0.01)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return float(np.sum(times)), sample_rays * len(times)


def timed_blocks(run_block, reps, world, dev):
    """REPS repetitions of one K-step block, each bracketed by barrier + synchronize on both sides and timed with CUDA events on
    the launching stream; per block the MAX over ranks. Returns the list of block times in seconds (same on every rank)."""
    out = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
        ev0.record()
        run_block()
        ev1.record()
        torch.cuda.synchronize()
        out.append(ev0.elapsed_time(ev1) / 1e3)
    return max_over_ranks(out, world, dev)


def max_over_ranks(times, world, dev='cpu'):
    """Per timed block the MAX over ranks of the elapsed time (one all_reduce of a small vector; no data-path collective)."""
    t = torch.tensor(list(times), dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def whole_job_value(units_per_rank_per_block, block_times, world):
    """Whole-job throughput under weak scaling: every rank processes the same number of units per block; the job's block time is
    the median over repetitions of the max-over-ranks time."""
    return world * units_per_rank_per_block / float(np.median(block_times))


def cpu_sample_rays(c, requested):
    """Rays per step of the CPU arm: the workload's full batch unless one step would take far more than ~20 s of host time
    (C5: Adam over 59 M parameters + 1.6 M points per step), then a bounded sample — the TRUE count is what gets printed."""
    if requested:
        return int(requested)
    t_probe, _ = cpu_baseline_run(c, 1, 0, 256)
    per_ray = t_probe / 256.0                               # pessimistic: the dense Adam pass is amortised over 256 rays only
    return int(min(c['N'], max(256, 20.0 / max(per_ray, 1e-6))))


def measure_config(args, c, name, rank, world, local_rank, dev, with_kernel=True):
    """Device-resident value + e2e (+ the fused kernel's roofline) of one workload on this rank's GPU."""
    import torch.distributed as dist
    from bundlesdf_b200 import ops as nof_ops
    t_setup = time.perf_counter()
    runner, seq = build_runner(c, seed=rank_seed(0, rank), device=dev, eager=args.eager)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup
    N, K = c['N'], args.steps
    n_params = sum(int(sg['param'].numel()) for sg in runner.adam_segs.values())

    def align():                                            # on to a step index = 1 (mod 10): K timed steps are whole graph replays
        while runner.global_step % 10 != 1:
            runner.train_steps(1)

    # ---- warm-up: >= W steps, then the same K steps as the timed region once, which captures its graphs outside of it
    runner.train_steps(max(args.warmup, 3))
    align()
    runner.train_steps(K)
    align()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if args.profile_range:                      # ncu --profile-from-start off: capture only the steady-state steps
        torch.cuda.cudart().cudaProfilerStart()
    blocks = timed_blocks(lambda: runner.train_steps(K), 1, world, dev)
    if args.profile_range:
        torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(runner, args.dump_outputs)
    t_med = float(np.median(blocks))
    value = whole_job_value(N * K, blocks, world)           # every rank processes N*K rays per block (weak scaling)

    # ---- e2e: host-resident ray pool (pinned), per-step H2D of the batch and D2H of the loss
    # Double-buffered like any input pipeline: while the GPU runs step k the host gathers batch k+1 into a pinned stage and a copy
    # stream uploads it; the loss of step k is copied back asynchronously and READ by the host one step later. Every step still
    # does its own H2D (N*48 B) and D2H (32 B) inside the timed region, through NerfRunner.train_loop.
    pool_host = runner.rays.cpu().pin_memory()
    stages = [torch.empty(N, 12).pin_memory() for _ in range(2)]
    pool_np, stages_np = pool_host.numpy(), [t.numpy() for t in stages]
    dev_bufs = [torch.empty(N, 12, device=dev) for _ in range(2)]
    loss_host = [torch.zeros(8).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ev_copy = [torch.cuda.Event() for _ in range(2)]
    ev_used = [torch.cuda.Event() for _ in range(2)]
    ev_loss = [torch.cuda.Event() for _ in range(2)]
    state = {'k': 0, 'loss_sum': 0.0}
    for e in ev_used:
        e.record()

    def prefetch(slot):
        runner.data_loader.next_ids()                   # advances the epoch permutation; batch_ray_ids is its CPU slice
        ev_copy[slot].synchronize()                     # the previous upload from this pinned stage has finished
        np.take(pool_np, runner.data_loader.batch_ray_ids.numpy(), axis=0, out=stages_np[slot])     # one host thread (an OpenMP fork per step costs more than the gather)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_used[slot])       # the step that read dev_bufs[slot] two steps ago is done with it
            dev_bufs[slot].copy_(stages[slot], non_blocking=True)
            ev_copy[slot].record(copy_stream)

    def step_e2e():
        k = state['k']
        cur = k % 2
        if k == 0:
            prefetch(0)
        prefetch(1 - cur)                               # host gather + H2D of the NEXT batch overlap the GPU work in flight
        torch.cuda.current_stream().wait_event(ev_copy[cur])
        b = runner.train_loop(dev_bufs[cur])
        ev_used[cur].record()
        loss_host[cur].copy_(b['losses'], non_blocking=True)
        ev_loss[cur].record()
        if k > 0:                                       # the caller reads every step's loss (one step late)
            ev_loss[1 - cur].synchronize()
            state['loss_sum'] += float(loss_host[1 - cur][0])
        runner.global_step += 1
        state['k'] = k + 1

    def e2e_block():
        for _ in range(K):
            step_e2e()

    for _ in range(5):
        step_e2e()
    e2e_blocks = timed_blocks(e2e_block, 1, world, dev)
    t_e2e = float(np.median(e2e_blocks))
    e2e_value = world * N * K / t_e2e

    res = {'value': value, 'ms_per_step': 1e3 * t_med / K, 'steps_per_s': K / t_med, 'clocks': clocks,
           'timing': {'timed_steps': K, 'block_ms': 1e3 * t_med,
                      'rule': 'max-over-ranks CUDA-event time of the K timed steps (barrier + synchronize on both sides)'},
           'e2e': {'value': e2e_value, 'unit': 'rays/s', 'h2d_bytes_per_step': N * 12 * 4, 'd2h_bytes_per_step': 32, 'steps': K,
                   'ms_per_step': 1e3 * t_e2e / K},
           'ray_pool': int(runner.rays.shape[0]), 'setup_s': round(t_setup, 1), 'n_params': n_params}
    launches_per_step = (7 if DEFER_TABLE else 6) + (1 if c.get('eik', 0) > 0 else 0)   # prologue, ray march, operand pack, fused step, pose backward, Adam (1 | 2: small segments + table, bookkeeping on the last block of either) [+ eikonal count pass]
    res['gpu_launches'] = launches_per_step * K
    if not with_kernel:
        return res

    # ---- roofline of the dominant kernel (fused step), timed alone on its launch stream
    runner.synchronize_parameters()
    batch = next(runner.data_loader)
    runner._forward_backward(batch)
    sb = runner._step_buf['sb']
    for _ in range(3):
        sb.launch()
    n_k = 50
    t_k = time_steps(sb.launch, n_k) / n_k
    for sg in runner.adam_segs.values():                # the extra launches accumulated garbage gradients: clear them
        sg['grad'].zero_()
    runner.amp_scaler.found_inf.zero_()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    abytes = algorithmic_bytes(c)
    achieved = abytes / t_k / 1e9
    traffic, kname = None, 'fused step kernel'
    try:
        tr = json.load(open(os.path.join(REPO, 'profiles', 'step_kernel_traffic.json'))).get(name)
        if isinstance(tr, dict):
            traffic, kname = tr.get('dram_bytes_per_launch'), tr.get('kernel', kname)
        else:
            traffic = tr
    except Exception:
        pass
    step_bytes = abytes + optimizer_bytes(n_params)
    res['roofline'] = {'bound': 'hbm', 'kernel': kname + ' (fused forward+loss+backward) incl. its operand-pack launch', 'achieved': achieved, 'peak': peak,
                       'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'algorithmic_bytes_per_launch': abytes, 'kernel_ms': t_k * 1e3,
                       'achieved_step': step_bytes / (t_med / K) / 1e9, 'frac_step': step_bytes / (t_med / K) / 1e9 / peak, 'step_bytes': step_bytes,
                       'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured)' if peaks else 'fallback 6650 GB/s (of fallback)',
                       'note': 'algorithmic bytes assume no cache credit (SURVEY.md 8d); `traffic` is the ncu dram__bytes of one launch of this config (profiles/); '
                               'a table that fits L2 makes traffic << algorithmic bytes and the kernel issue/latency-bound, not HBM-bound (DESIGN.md)'}
    return res


DUMP_TABLE_ROWS = 1 << 18     # hash-table rows in the dump (all of them when the table is smaller)


def dump_outputs(runner, out_dir):
    """What a caller of train_steps has after its last step, as float32 .npy files (2 MB + the MLP and per-frame parameters)."""
    runner.synchronize_parameters()                         # the last step's deferred table update
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    table = runner.table
    rows = np.sort(np.random.default_rng(0).choice(table.shape[0], size=min(table.shape[0], DUMP_TABLE_ROWS), replace=False))
    out = {'losses': runner._step_buf['losses'], 'mlp_params': runner.mlp_flat,
           'hash_table_sample': table[torch.from_numpy(rows).to(table.device)]}
    for key, name in (('pose_array', 'pose_params'), ('feature_array', 'frame_features')):
        if runner.models[key] is not None:
            out[name] = runner.models[key].data.data
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20, help='timed steps of each measurement (value, e2e)')
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='C2', choices=list(CONFIGS))
    ap.add_argument('--cpu-rays', type=int, default=0, help='rays per step of the CPU baseline (0: the full batch unless a step would exceed ~20 s)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-config4', action='store_true', help='N > 1 only: skip the extra BASELINE configs[3] measurement (C3 x N)')
    ap.add_argument('--profile-range', action='store_true', help='bracket the timed steps with cudaProfilerStart/Stop (for ncu)')
    ap.add_argument('--eager', action='store_true', help='disable CUDA-graph replay of the step (launch the kernels one by one)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be >= 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs dumps the timed path of --impl ours')
    c = CONFIGS[args.config]
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    S = c['S_occ'] + c['S_d']

    def config_of(cc, nm):
        return {'workload': WORKLOAD[nm], 'rays_per_step': cc['N'], 'samples_per_ray': cc['S_occ'] + cc['S_d'], 'hash_levels': cc['L'],
                'log2_hashmap_size': cc['log2T'], 'finest_res': cc['finest'], 'frames': cc['frames'], 'amp': True, 'optimize_poses': bool(cc['pose']),
                'eikonal_weight': cc.get('eik', 0.0),
                'defer_table_update': DEFER_TABLE, 'graph_block_steps': 10,
                'parallelism': f'{world} independent sequence(s), one per GPU',
                'l2_policy': 'inputs larger than L2 are not claimed: the fp16 table (17.4 MB at C2/C3) is L2-resident by design; every step draws a '
                             'fresh random batch from a >100 MB ray pool and the Adam pass streams ~300 MB per step, so no two timed steps reuse inputs'}
    config = config_of(c, args.config)

    if args.impl == 'reference':
        # The reference has no CPU implementation of this path (its grid encoder and samplers are CUDA-only, kaolin is absent):
        # the reference arm is the oracle port on the host cores. Each step is the workload's FULL batch when K such steps fit the
        # time budget, else a bounded sample of it; the line prints the true per-step ray count either way.
        if rank != 0:
            return
        warm = max(1, min(args.warmup, 1))
        steps = max(1, args.steps)
        budget_s = 170.0
        t_probe, _ = cpu_baseline_run(c, 1, 0, 256)
        per_ray = t_probe / 256.0
        rays = int(min(c['N'], max(32, budget_s / (steps + warm) / max(per_ray, 1e-6))))
        if args.cpu_rays:
            rays = args.cpu_rays
        t, n_rays = cpu_baseline_run(c, steps, warm, rays)
        v = n_rays / t
        cores = pick_cpu_threads(c)
        config['rays_per_step'] = rays
        config['workload_rays_per_step'] = c['N']
        line = {'impl': 'reference', 'metric': 'nerf_train_rays_per_s', 'value': v, 'unit': 'rays/s', 'n_gpus': args.gpus, 'steps': steps,
                'warmup': warm, 'ms_per_step': 1e3 * t / steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic', 'config': config,
                'cpu_baseline': {'value': v, 'unit': 'rays/s', 'cores': cores, 'kind': 'port',
                                 'sample': f'{steps} full train steps (sample, encode, MLP, losses, backward, Adam) of {rays} rays x {S} samples each '
                                           f'(workload batch: {c["N"]} rays), torch fp32, {cores} of {os.cpu_count()} host threads (fastest of a probe)'},
                'e2e': {'value': v, 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
        print(json.dumps(line))
        return

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    m = measure_config(args, c, args.config, rank, world, local_rank, dev)
    line = {'metric': 'nerf_train_rays_per_s', 'value': m['value'], 'unit': 'rays/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': m['ms_per_step'], 'steps_per_s': m['steps_per_s'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f16 (fp32 accumulate, fp32 master weights)', 'data': 'synthetic', 'config': config, 'clocks': m['clocks'], 'timing': m['timing'],
            'e2e': m['e2e'], 'gpu_launches': m['gpu_launches'], 'roofline': m['roofline'], 'ray_pool': m['ray_pool'], 'setup_s': m['setup_s']}
    if world > 1 and args.config == 'C2' and not args.no_config4:
        # BASELINE.json configs[3]: the HO3D-shaped config (C3), one independent sequence per GPU. The headline stays C2 x N so that the
        # driver's 1 -> 8 efficiency compares like with like; this is the same measurement on the workload BASELINE names for 8 GPUs.
        m4 = measure_config(args, CONFIGS['C3'], 'C3', rank, world, local_rank, dev, with_kernel=False)
        line['config4'] = {'config': config_of(CONFIGS['C3'], 'C3'), 'value': m4['value'], 'unit': 'rays/s', 'ms_per_step': m4['ms_per_step'],
                           'timing': m4['timing'], 'e2e': m4['e2e'], 'clocks': m4['clocks']}
    if rank == 0 and not args.no_cpu_baseline:
        rays = cpu_sample_rays(c, args.cpu_rays)
        tc, nr = cpu_baseline_run(c, 2, 1, rays)
        cores = pick_cpu_threads(c)
        line['cpu_baseline'] = {'value': nr / tc, 'unit': 'rays/s', 'cores': cores, 'kind': 'port', 'rays_per_step': rays,
                                'sample': f'2 full train steps of {rays} rays x {S} samples (workload batch: {c["N"]} rays; oracle port, torch fp32, '
                                          f'{cores} of {os.cpu_count()} host threads, fastest of a probe) after 1 warm-up'}
        ref_cuda = reference_cuda_column(c, args.config)
        if ref_cuda is not None:
            line['reference_cuda'] = ref_cuda
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def reference_cuda_column(c, name):
    """SURVEY.md 8(d) second comparison column: the reference's OWN train_loop (nerf_runner.py:679-852) on its own compiled CUDA
    extensions (oracle/_ref) on this B200. Test infrastructure timed in the cpu_baseline leg only; None when oracle/_ref is absent."""
    import contextlib
    try:
        sys.path.insert(0, os.path.join(REPO, 'oracle'))
        with contextlib.redirect_stdout(sys.stderr):      # the reference prints while it builds its models; stdout carries ONE JSON line
            import ref_train_loop
            return ref_train_loop.time_reference(c, name)
    except Exception as e:      # the checker is optional
        return {'unavailable': repr(e)[:300]}


if __name__ == '__main__':
    main()
