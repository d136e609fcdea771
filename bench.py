#!/usr/bin/env python
"""Benchmark of the per-ray rendering hot path (BASELINE.json metric: rays/s, fwd+bwd, NeRF-Synthetic-lego shape).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2|C3|C4] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline (`value`, `e2e`, `roofline`): config C2 = nerf-blender HashGrid L16/F2/T2^19 + FullyFused-64 fields, 8192 rays per GPU.
One "step" = one pass of the hot path over one batch of synthetic rays: lattice-mask march (+ row allocation) + persistent per-ray forward
(hash gather, both MLPs, compositing, early termination) + fused masked smooth-L1 loss + per-ray backward + the field backward as a
tensor-core network half and a high-occupancy table scatter (+ the gradient mean over the ranks when N > 1: one-launch NVLink exchange,
pipelined with the scatter's level groups), replayed as ONE CUDA graph.  The optimizer is outside the path (SURVEY.md 8f).
`ms_per_step` / `value` use the MEDIAN of the K per-step CUDA-event times (SURVEY 8d), max over ranks; the mean is reported beside it.

At N = 1 the same JSON line also carries
  * `extra.C3` / `extra.C4`: BASELINE.json configs 3 (neus-blender with mask, 8192 rays) and 4 (neus-dtu with learned background,
    4096 rays) measured the same way (own `roofline`, `e2e`, kernel times); `--config C3|C4` makes one of them the headline instead;
  * `cpu_baseline`: BASELINE.json config 1 -- the reference's own pure-torch fields (VanillaFrequency + VanillaMLP, 4096 rays) inside
    the CPU oracle's marching / compositing, fwd+bwd on the host cores; `cpu_baseline_secondary`: the fp32 CPU port of C2 itself.
`--impl reference` times the CPU port of the headline config on the host cores at the SAME rays per step it reports.
`--dump-outputs DIR` (GPU headline only, rank 0) writes what the last timed step handed its caller to DIR/<name>.npy: `loss`, the
per-ray float outputs, `num_samples` and `grad.<parameter name>` for every trainable parameter.  Inputs are seeded, so two builds run with
the same arguments can be compared array by array.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_RAYS = 8192            # per GPU (max_train_num_rays, configs/nerf-blender.yaml:24)
POOL = 8                 # distinct ray batches cycled through
CPU_SAMPLE_RAYS = 1024   # rays per step of the CPU arms (bounded sample of the same workload)
CPU_RAY_BUDGET = 8192 * 30   # rays the reference arm traces in total (steps + warm-up): full 8192-ray steps up to 30 of them (~2 min)
CPU_MAX_THREADS = 16     # the torch-CPU oracle stops scaling (and then collapses) beyond ~16 threads; `cores` reports what was used


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


# --------------------------------------------------------------------------------------------------
# CPU arms: the oracle port of the same workload (the reference's own stack -- tiny-cuda-nn + nerfacc --
# is CUDA-only and not installable offline, DESIGN.md)
# --------------------------------------------------------------------------------------------------
def cpu_workload(n_rays, seed):
    from oracle import models as om
    from nsr_b200 import configs, synthetic, ops
    cfg = configs.nerf_blender()
    grid = ops.GridSpec(cfg['geometry']['xyz_encoding_config'])
    mlp = ops.MlpSpec(32, 16, cfg['geometry']['mlp_network_config'])
    cmlp = ops.MlpSpec(32, 3, cfg['texture']['mlp_network_config'])
    g = torch.Generator().manual_seed(7)
    dflat = torch.cat([mlp.init_params(g), (torch.rand(grid.n_params, generator=g) * 2 - 1) * 0.1])
    synthetic.shape_density(dflat, grid, mlp.n_params)
    cflat = cmlp.init_params(g)
    dflat.requires_grad_(True)
    cflat.requires_grad_(True)
    P = om.NerfParams(cfg['geometry']['xyz_encoding_config'], dflat, cflat)
    P.one_gather = True   # one indexing op over all corners: no table-sized autograd temporaries per corner (oracle/hashgrid.py)
    binary = synthetic.occupancy()
    step = np.float32(synthetic.render_step_size())
    tg = torch.Generator().manual_seed(seed)

    def run(i):
        rays = synthetic.sample_rays(n_rays, seed=seed * 1000 + i)
        jit = np.random.default_rng(seed * 1000 + i + 1).random(n_rays).astype(np.float32)
        target = torch.rand(n_rays, 3, generator=tg)
        bg = torch.rand(3, generator=tg)
        dflat.grad = cflat.grad = None
        out = om.nerf_render(P, rays, binary, 1.5, step, bg, jitter=jit, emulate_fp16=False)
        loss = om.smooth_l1_masked(out['comp_rgb'], target, out['rays_valid'])
        loss.backward()
        return int(out['num_samples']), out['num_marched']
    return run


def time_cpu(steps, warmup, n_rays=CPU_SAMPLE_RAYS):
    torch.set_num_threads(min(os.cpu_count(), CPU_MAX_THREADS))
    run = cpu_workload(n_rays, seed=3)
    for i in range(warmup):
        run(i)
    t0 = time.perf_counter()
    kept = marched = 0
    for i in range(steps):
        k, m = run(warmup + i)
        kept += k
        marched += m
    dt = time.perf_counter() - t0
    return {'rays_per_s': n_rays * steps / dt, 'ms_per_step': dt / steps * 1e3, 'kept': kept / steps, 'marched': marched / steps,
            'cores': torch.get_num_threads(), 'n_rays': n_rays}


WORKLOAD = {
    'C2': f'nerf-blender lego shape, HashGrid L16 F2 T2^19 + FullyFused-64 fields, {N_RAYS} rays/GPU (C2)',
    'C3': 'neus-blender lego shape with mask, HashGrid L16 F2 T2^19 + fp32 SDF MLP + FullyFused-64 colour, cos anneal, 8192 rays/GPU (C3)',
    'C4': 'neus-dtu shape with learned background (NeRF++ contraction), VanillaMLP colour / background networks, 4096 rays/GPU (C4)',
}


def time_cpu_c1(steps, warmup, n_rays=4096):
    """BASELINE.json config 1: nerf-blender with the reference's pure-torch fields (VanillaFrequency n=10/4 + VanillaMLP,
    models/network_utils.py:14-37,95-139 -- the oracle classes are pinned bit-for-bit to the reference's by tests/test_oracle_golden.py),
    4096 rays, inside the CPU oracle's marching / visibility / compositing, fwd + bwd, fp32."""
    from oracle import models as om
    from nsr_b200 import synthetic
    torch.set_num_threads(min(os.cpu_count(), CPU_MAX_THREADS))
    fields = om.VanillaNerfFields(10, 4, 16, seed=0)
    with torch.no_grad():
        fields.geo.layers[-1].bias[0] = 4.0   # densities ~ exp(3): the visibility filter and early termination matter (as in the C1 GPU test)
    binary = synthetic.occupancy()
    step = np.float32(synthetic.render_step_size())
    tg = torch.Generator().manual_seed(5)
    kept = marched = 0
    t0 = None
    for i in range(warmup + steps):
        if i == warmup:
            t0 = time.perf_counter()
            kept = marched = 0
        rays = synthetic.sample_rays(n_rays, seed=7000 + i)
        jit = np.random.default_rng(8000 + i).random(n_rays).astype(np.float32)
        target, bg = torch.rand(n_rays, 3, generator=tg), torch.rand(3, generator=tg)
        for p in fields.parameters():
            p.grad = None
        out = om.vanilla_nerf_render(fields, rays, binary, 1.5, step, bg, jitter=jit)
        om.smooth_l1_masked(out['comp_rgb'], target, out['rays_valid']).backward()
        kept += int(out['num_samples'])
        marched += int(out['num_marched'])
    dt = time.perf_counter() - t0
    return {'rays_per_s': n_rays * steps / dt, 'ms_per_step': dt / steps * 1e3, 'kept': kept / steps, 'marched': marched / steps,
            'cores': torch.get_num_threads(), 'n_rays': n_rays}


def reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.config != 'C2':
        print(json.dumps({'impl': 'reference', 'unavailable': f'the CPU port is timed for the headline config C2 only (asked for {args.config})'}), flush=True)
        return
    # every step = one full batch of the reported workload (8192 rays): ~4 s per step on 16 host threads, so the driver's
    # --steps 20 --warmup 5 ends in ~2 min.  Only when steps + warmup would push the run past CPU_RAY_BUDGET rays is the batch cut
    # down, and then the workload string says so.
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    n_rays = N_RAYS if N_RAYS * (steps + warmup) <= CPU_RAY_BUDGET else max(64, CPU_RAY_BUDGET // (steps + warmup))
    r = time_cpu(steps, warmup, n_rays=n_rays)
    workload = WORKLOAD['C2'] if n_rays == N_RAYS else WORKLOAD['C2'].replace(f'{N_RAYS} rays/GPU', f'{n_rays} rays/step (bounded sample of the {N_RAYS}-ray batch)')
    line = {
        'impl': 'reference', 'metric': 'rays/sec fwd+bwd (NeRF-Synthetic lego shape)', 'value': r['rays_per_s'], 'unit': 'rays/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload, 'rays_per_step': n_rays,
                   'note': 'the reference stack (tiny-cuda-nn + nerfacc 0.3.3) is CUDA-only and not installable offline; this arm times '
                           'the fp32 CPU oracle port of the same path on the host cores (kind: port)'},
        'cpu_baseline': {'value': r['rays_per_s'], 'unit': 'rays/s', 'cores': r['cores'], 'kind': 'port',
                         'sample': f"{r['n_rays']} rays/step of the C2 workload (marched {r['marched']:.0f}, kept {r['kept']:.0f} samples/step), "
                                   f"fwd+bwd, torch CPU fp32, {r['cores']} threads"},
        'e2e': {'value': r['rays_per_s'], 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = f'/tmp/nsr_clocks_{os.getpid()}.csv'

    def start(self):
        try:
            self.f = open(self.path, 'w')
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in open(self.path):
            c = [x.strip() for x in ln.split(',')]
            if len(c) < 8 or not c[0].isdigit() or int(c[0]) != self.idx:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for nme, v in zip(names, c[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(nme)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


def build_model(device, seed=0):
    from nsr_b200 import models, configs, synthetic
    cfg = configs.nerf_blender()
    torch.manual_seed(seed)
    model = models.make('nerf', cfg).to(device)
    if model._fused is None:
        raise RuntimeError('bench: the fused CUDA path was not selected')
    net = model.geometry.encoding_with_network
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        p = net.params.detach().cpu().clone()
        p[net.mlp.n_params:] = (torch.rand(net.grid.n_params, generator=g) * 2 - 1) * 0.1
        synthetic.shape_density(p, net.grid, net.mlp.n_params)
        net.params.copy_(p.to(device))
    model.occupancy_grid.set_binary(torch.from_numpy(synthetic.occupancy()))
    model.train()
    return model


DUMP_MAX_ELEMS = 1 << 22   # larger arrays are dumped as a fixed seeded sample of this many entries: a whole dump stays well under 64 MB


def snapshot_outputs(loss, out, named_params, n_rays):
    """device copies of what one step returns to its caller: the loss, the per-ray float outputs (the capacity-length per-sample buffers
    are undefined past num_samples and laid out in allocation order, so they are left out), the kept-sample count, every gradient"""
    snap = {'loss': loss, 'num_samples': out['num_samples_dev'] if 'num_samples_dev' in out else out['num_samples']}
    snap.update({k: v for k, v in out.items() if torch.is_tensor(v) and v.is_floating_point() and v.dim() >= 1 and v.shape[0] == n_rays})
    snap.update({f'grad.{name}': p.grad for name, p in named_params if p.requires_grad and p.grad is not None})
    return {k: v.detach().clone() for k, v in snap.items()}


def write_outputs(dirname, snap):
    os.makedirs(dirname, exist_ok=True)
    for name, v in snap.items():
        if v.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(v.numel(), DUMP_MAX_ELEMS, replace=False))
            v = v.reshape(-1)[torch.from_numpy(idx).to(v.device)]
        v = v.float() if v.is_floating_point() and v.dtype != torch.float64 else v.double()
        np.save(os.path.join(dirname, f'{name}.npy'), v.cpu().numpy())


def masked_smooth_l1(comp_rgb, target, valid):
    """systems/nerf.py:97 without the host sync of boolean indexing: mean over valid rays x 3 channels."""
    m = valid.float()
    per = F.smooth_l1_loss(comp_rgb, target, reduction='none') * m
    return per.sum() / (m.sum() * 3.0).clamp(min=1.0)


def neus_config(name, dev, steps, warmup, flush, peak, peak_src, dump=None):
    """BASELINE.json config 3 (neus-blender with mask, 8192 rays; static-shape step = one CUDA graph) or config 4 (neus-dtu with learned
    background, 4096 rays; eager: the background pass has host-sized outputs) on one GPU: fwd + the reference's loss terms
    (systems/neus.py:98-121 as nsr_b200.losses.neus_losses) + bwd.  Returns a sub-line: rays/s (median of per-step CUDA events, L2
    flushed before every step), e2e (pinned host rays / targets / masks in, loss scalar out), per-kernel times and the roofline of the
    dominant kernel.  Synthetic scene as SURVEY 8d: sphere-init SDF, occupancy = shell around the surface (+ a 15 % random background
    grid for C4), seeded rays, cos_anneal_ratio 0.25.  ``dump``: a dict that receives snapshot_outputs() of the last timed step."""
    from nsr_b200 import models, configs, synthetic
    from nsr_b200.lib import lib
    from nsr_b200.losses import neus_losses
    from nsr_b200.graph import GraphedStep
    cfg_fn, n = (configs.neus_blender, 8192) if name == 'C3' else (configs.neus_dtu, 4096)
    cfg = cfg_fn()
    torch.manual_seed(0)
    m = models.make('neus', cfg).to(dev)
    r = cfg['radius']
    g = (np.arange(128) + 0.5) / 128 * 2 * r - r
    X, Y, Z = np.meshgrid(g, g, g, indexing='ij')
    d = np.sqrt(X ** 2 + Y ** 2 + Z ** 2)
    m.occupancy_grid.set_binary(torch.from_numpy((d > 0.336 * r) & (d < 0.464 * r + 0.1)))   # shell around the sphere-init surface
    if cfg['learned_background']:
        m.occupancy_grid_bg.set_binary(torch.from_numpy(np.random.default_rng(0).random((256, 256, 256)) < 0.15))
    m.train()
    m.update_step(0, 5001)   # cos_anneal_ratio = 0.25 (neus-blender: cos_anneal_end 20000); not a multiple of 16: no grid refresh
    pool = 4
    rays_np = []
    for i in range(pool):
        rr = synthetic.sample_rays(n, seed=500 + i)
        if r != 1.5:
            rr[:, :3] *= r / 1.5 * 0.6
        rays_np.append(rr)
    tg = torch.Generator().manual_seed(17)
    tgt = [torch.rand(n, 3, generator=tg) for _ in range(pool)]
    msk = [(torch.rand(n, generator=tg) > 0.5).float() for _ in range(pool)]
    rays_pin, tgt_pin, msk_pin = [torch.from_numpy(x).pin_memory() for x in rays_np], [t.pin_memory() for t in tgt], [t.pin_memory() for t in msk]
    rays_dev, tgt_dev, msk_dev = [x.to(dev) for x in rays_pin], [x.to(dev) for x in tgt_pin], [x.to(dev) for x in msk_pin]
    lam = dict(lambda_rgb_mse=10., lambda_eikonal=0.1, lambda_mask=0.1)
    params = [p for p in m.parameters() if p.requires_grad]
    graphed = name == 'C3'
    if graphed:
        gs = GraphedStep(m, lambda out, b: neus_losses(out, b['rgb'], b['fg_mask'], **lam)[0], n, batch_spec={'rgb': (3,), 'fg_mask': ()},
                         device=dev, warmup=3)

        def step(rays, target, mask):
            return gs(rays, rgb=target, fg_mask=mask, background_color=torch.rand(3, device=dev))
    else:
        def step(rays, target, mask):
            m.background_color = torch.rand(3, device=dev)
            out = m(rays.to(dev, non_blocking=True))
            loss, _ = neus_losses(out, target.to(dev, non_blocking=True), mask.to(dev, non_blocking=True), **lam)
            for p in params:
                p.grad = None
            loss.backward()
            step.last = out
            return loss
    for i in range(warmup):
        step(rays_dev[i % pool], tgt_dev[i % pool], msk_dev[i % pool])
    torch.cuda.synchronize()
    lib.launches = 0
    evs = []
    for i in range(steps):
        j = i % pool
        flush.fill_(float(i))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step(rays_dev[j], tgt_dev[j], msk_dev[j])
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    launches = lib.launches
    if dump is not None:
        dump.update(snapshot_outputs(loss, gs.out if graphed else step.last, m.named_parameters(), n))
    per = [a.elapsed_time(b) for a, b in evs]
    host = []
    for i in range(steps):
        j = i % pool
        flush.fill_(float(i))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _ = step(rays_pin[j], tgt_pin[j], msk_pin[j]).item()
        host.append((time.perf_counter() - t0) * 1e3)
    ms, ms_e2e = statistics.median(per), statistics.median(host)
    # sample counts (one read-back)
    if graphed:
        k_fg, k_bg, m_bg = float(gs.out['num_samples_dev']), 0.0, 0.0
        overflow = bool(gs.out['overflow'])
    else:
        o = step.last
        k_fg, k_bg, overflow = float(o['num_samples'].sum()), float(o['num_samples_bg'].sum()), False
        m_bg = k_bg   # marched background samples are not reported separately by the eager API: count the kept ones
    # per-kernel durations: eager API, CUDA events around every C-ABI call
    if graphed:
        m.randomized = True

        def eager(rays, target, mask):
            m.background_color = torch.rand(3, device=dev)
            out = m(rays)
            loss, _ = neus_losses(out, target, mask, **lam)
            for p in params:
                p.grad = None
            loss.backward()
    else:
        eager = step
    for i in range(2):
        eager(rays_dev[i], tgt_dev[i], msk_dev[i])
    lib.profile = {}
    nprof = 5
    for i in range(nprof):
        flush.fill_(1.0)
        eager(rays_dev[i % pool], tgt_dev[i % pool], msk_dev[i % pool])
    torch.cuda.synchronize()
    kern = {kn: sum(a.elapsed_time(b) for a, b in v) / nprof for kn, v in lib.profile.items()}
    lib.profile = None
    # algorithmic bytes (SURVEY 8d): NeuS sample = 512 B gather (fwd) + 512 B re-gather + 512 B scatter + 512 B second-order scatter (bwd);
    # background NeRF sample = 512 B gather + 512 B scatter (+ 512 B per marched sample for the visibility pre-pass)
    alg = {'nsr_neus_field_fwd': 512.0 * k_fg, 'nsr_neus_field_bwd': 1536.0 * k_fg}
    dom = max((kn for kn in alg if kn in kern), key=lambda kn: kern[kn], default=None)
    step_bytes = 2048.0 * k_fg + 1024.0 * k_bg + 512.0 * m_bg
    roofline = None
    if dom is not None:
        ach = alg[dom] / (kern[dom] * 1e-3) / 1e9
        roofline = {'bound': 'hbm', 'kernel': dom, 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': None,
                    'peak_source': peak_src, 'algorithmic_bytes_per_launch': alg[dom], 'kernel_ms': kern[dom],
                    'per_kernel': {kn: {'algorithmic_bytes': alg[kn], 'ms': kern[kn], 'frac': alg[kn] / (kern[kn] * 1e-3) / 1e9 / peak}
                                   for kn in alg if kn in kern},
                    'whole_step': {'algorithmic_bytes': step_bytes, 'achieved': step_bytes / (ms * 1e-3) / 1e9, 'frac': step_bytes / (ms * 1e-3) / 1e9 / peak}}
    sub = {'metric': 'rays/sec fwd+bwd', 'value': n / (ms * 1e-3), 'unit': 'rays/s', 'ms_per_step': ms, 'steps': steps, 'warmup': warmup,
           'dtype': 'f32 SDF field + f16 colour networks' if name == 'C3' else 'f32 SDF field + f16-operand VanillaMLP kernels',
           'config': {'workload': WORKLOAD[name], 'rays_per_gpu': n, 'fg_samples_per_step': k_fg, 'bg_samples_per_step': k_bg,
                      'samples_per_s': (k_fg + k_bg) / (ms * 1e-3), 'l2': 'flushed (256 MB write) before every timed step',
                      'step': ('static-shape forward + fused losses + backward as ONE CUDA graph (nsr_b200.graph.GraphedStep)' if graphed
                               else 'eager public API (NeuSModel.forward + nsr_b200.losses.neus_losses + backward); exact-size outputs, host-sized background pass'),
                      'capacity_overflow': overflow},
           'e2e': {'value': n / (ms_e2e * 1e-3), 'unit': 'rays/s', 'h2d_bytes_per_step': n * (6 + 3 + 1) * 4, 'd2h_bytes_per_step': 4},
           'gpu_launches': launches, 'roofline': roofline, 'kernels_ms': {kn: round(v, 5) for kn, v in kern.items()}}
    if graphed:
        del gs
    del m
    torch.cuda.empty_cache()
    return sub


def neus_arm(args):
    """--config C3 | C4 as the headline (single GPU)."""
    if int(os.environ.get('WORLD_SIZE', '1')) != 1 or args.gpus != 1:
        raise SystemExit('bench.py --config C3|C4 runs on one GPU')
    torch.cuda.set_device(0)
    dev = torch.device('cuda', 0)
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    peak, peak_src = peaks()
    sampler = ClockSampler(0)
    sampler.start()
    dump = {} if args.dump_outputs else None
    sub = neus_config(args.config, dev, args.steps, max(3, args.warmup), flush, peak, peak_src, dump=dump)
    clocks = sampler.stop()
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    line = dict(sub)
    line.update({'n_gpus': 1, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'data': 'synthetic', 'clocks': clocks})
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


def gpu_arm(args):
    import torch.distributed as dist
    from nsr_b200 import synthetic
    from nsr_b200.lib import lib
    from nsr_b200.parallel import make_grad_sync
    from nsr_b200.graph import GraphedStep
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world == 1 and args.gpus > 1:
        raise SystemExit('bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    # stdout carries exactly ONE JSON line: anything libraries print there meanwhile (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    model = build_model(dev)
    params = [p for p in model.parameters() if p.requires_grad]
    # inputs: POOL batches of rays / targets, different per rank (the reference seeds all ranks alike, SURVEY 2.1 quirk)
    rays_np = [synthetic.sample_rays(N_RAYS, seed=1000 * rank + i) for i in range(POOL)]
    tg = torch.Generator().manual_seed(99 + rank)
    tgt_np = [torch.rand(N_RAYS, 3, generator=tg) for _ in range(POOL)]
    rays_dev = [torch.from_numpy(r).to(dev) for r in rays_np]
    tgt_dev = [t.to(dev) for t in tgt_np]
    rays_pin = [torch.from_numpy(r).pin_memory() for r in rays_np]
    tgt_pin = [t.pin_memory() for t in tgt_np]
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)  # > 126 MB L2

    from nsr_b200.losses import nerf_rgb_loss

    def loss_fn(out, batch):
        # systems/nerf.py:68-97 (background blend + masked smooth-L1) as the fused CUDA op of the package
        return nerf_rgb_loss(out['acc_rgb'], out['opacity'], model.background_color, batch['rgb'])[0]

    # the public fast path: whole step (march .. backward) as one CUDA graph, no host sync inside
    # N > 1: the NCCL all-reduce (mean) of the parameter gradients is captured into the same graph, right behind the backward
    comm = os.environ.get('NSR_GRAD_COMM_DTYPE', 'fp32')  # 'bf16': opt-in wire compression of the table gradient
    # exchange: our own reduce-scatter + all-gather kernel over NVLink peer memory (csrc/p2p.cu); NCCL if symmetric memory / P2P is
    # unavailable, if NSR_GRAD_SYNC=nccl, or for the bf16 wire format
    sync, sync_desc = (None, None)
    if world > 1:
        sync, sync_desc = make_grad_sync(params, world, comm_dtype=(torch.bfloat16 if comm == 'bf16' else None),
                                         prefer_p2p=os.environ.get('NSR_GRAD_SYNC', 'p2p') != 'nccl')
    post_backward = sync.all_reduce_mean if sync is not None else None
    if sync is not None and hasattr(sync, 'bind_direct'):
        # the backward accumulates straight into the peer-mapped exchange buffer (no copy-in); NSR_P2P_OVERLAP=1 (default): the table gradient
        # is scattered level group by level group and each finished group is exchanged beside the next group's scatter
        if os.environ.get('NSR_P2P_OVERLAP', '1') == '1' and sync.one_launch and model._fused.bwd_kernel == 'tiles_split':
            sync.bind_pipelined(model._fused)
            post_backward = sync.finish
            sync_desc += ', zero-copy gradients, exchange pipelined with the table scatter in 3 level groups (one launch per group)'
        else:
            sync.bind_direct(model._fused)
            sync_desc += ', zero-copy gradients' + (', one launch' if sync.one_launch else ', barrier + reduce + barrier')
    # inside the graph only what the fused loss reads is materialised (comp_rgb / rays_valid come out of nsr_nerf_loss_fwd itself)
    model._fused.lean_static_outputs = True
    gstep = GraphedStep(model, loss_fn, N_RAYS, batch_spec={'rgb': (3,)}, device=dev, warmup=3,
                        post_backward=post_backward)

    model._fused.lean_static_outputs = False   # (captured already; the eager API below returns the full dict)

    def step(rays, target, do_sync=True):
        bg = torch.rand(3, device=dev)                      # systems/nerf.py:71 (random background per step)
        return gstep(rays, rgb=target, background_color=bg)

    def eager_step(rays, target):
        """the same step through the eager public API (NeRFModel.forward), exact-size outputs, ~40 launches from Python"""
        model.background_color = torch.rand(3, device=dev)
        out = model(rays)
        loss = masked_smooth_l1(out['comp_rgb'], target, out['rays_valid'])
        for p in params:
            p.grad = None
        loss.backward()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(nsteps, e2e, fn=step):
        """per-step times in ms (list); L2 flushed (untimed) before every step.  e2e: host-clock per step including the
        H2D copies of that step's inputs and the D2H read of its loss."""
        evs, host_t = [], []
        for i in range(nsteps):
            j = i % POOL
            flush.fill_(float(i))
            if e2e:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                loss = fn(rays_pin[j], tgt_pin[j])
                _ = loss.item()
                host_t.append((time.perf_counter() - t0) * 1e3)
            else:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn(rays_dev[j], tgt_dev[j])
                e1.record()
                evs.append((e0, e1))
        torch.cuda.synchronize()
        return host_t if e2e else [a.elapsed_time(b) for a, b in evs]

    for i in range(max(3, args.warmup)):
        step(rays_dev[i % POOL], tgt_dev[i % POOL])
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- timed region: exactly K steps, inputs resident in HBM
    lib.launches = 0
    barrier()
    per_step = timed(args.steps, e2e=False)
    barrier()
    launches = lib.launches
    dump = snapshot_outputs(gstep.loss, gstep.out, model.named_parameters(), N_RAYS) if args.dump_outputs and rank == 0 else None
    # ---- end-to-end: pinned host buffers in, loss out, same K steps
    barrier()
    per_step_e2e = timed(args.steps, e2e=True)
    barrier()
    # median of the K per-step times (SURVEY 8d) x K: `ms` / `ms_e2e` stay "time of the K steps" so that everything below is unchanged
    ms_mean, ms_e2e_mean = sum(per_step) / args.steps, sum(per_step_e2e) / args.steps
    ms, ms_e2e = statistics.median(per_step) * args.steps, statistics.median(per_step_e2e) * args.steps
    clocks = None
    # keep the GPUs under the same load until the clock sampler has seen it (short timed regions); every rank replays
    # the same number of steps because the captured graph contains the collective
    n_soak = int(max(0.0, 1.5 - (ms + ms_e2e) / 1e3) / max(ms / args.steps * 1e-3, 1e-4)) if world == 1 else int(1.5 / max(ms / args.steps * 1e-3, 1e-4))
    if world > 1:
        t = torch.tensor([n_soak], device=dev)
        dist.broadcast(t, 0)
        n_soak = int(t.item())
    for _ in range(n_soak):
        step(rays_dev[0], tgt_dev[0])
    torch.cuda.synchronize()
    if rank == 0:
        clocks = sampler.stop()
    # ---- sample counts of the workload (one replay per pool batch, read back)
    kept = marched = 0.0
    for j in range(POOL):
        step(rays_dev[j], tgt_dev[j])
        mm, kk = gstep.counts()
        marched += mm / POOL
        kept += kk / POOL
    if world > 1:
        if hasattr(sync, 'check'):
            sync.check()
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
        cnt = torch.tensor([kept, marched], device=dev, dtype=torch.float64)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        kept, marched = cnt.tolist()
        dist.barrier()
        torch.cuda.synchronize()
        if rank != 0:
            # hard exit: tearing down an NCCL communicator that is referenced by a live CUDA graph can block forever
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)

    # ---- rank 0: eager-API timing and per-kernel durations (CUDA events around every C-ABI call; same workload)
    model._fused.exchange_hook = model._fused.level_groups = model._fused.direct_grads = None   # single-rank eager steps from here on: no exchange
    nprof = min(args.steps, 20)
    for i in range(3):
        eager_step(rays_dev[i % POOL], tgt_dev[i % POOL])
    ms_eager = statistics.median(timed(nprof, e2e=False, fn=eager_step))
    lib.profile = {}
    for i in range(nprof):
        flush.fill_(1.0)
        eager_step(rays_dev[i % POOL], tgt_dev[i % POOL])
    torch.cuda.synchronize()
    kern = {name: {'ms': sum(a.elapsed_time(b) for a, b in evs) / len(evs), 'launches_per_step': len(evs) / nprof}
            for name, evs in lib.profile.items()}
    lib.profile = None
    peak, peak_src = peaks()
    ms_step = ms / args.steps
    k1, m1 = kept / world, marched / world          # per GPU
    # samples the per-ray forward kernel evaluates (gathers + both MLPs): whole 32-sample chunks of every ray up to and including the
    # chunk in which its transmittance falls below early_stop_eps (the kept samples of a ray are a prefix of its marched ones)
    evaluated = 0.0
    with torch.no_grad():
        for j in range(POOL):
            o = model.forward_(rays_dev[j], static=True)
            tot = o['counts_loose'].double()
            kp = (o['offsets_packed'][1:] - o['offsets_packed'][:-1]).double()
            evaluated += float(torch.where(kp < tot, torch.minimum(tot, (torch.floor(kp / 32) + 1) * 32), tot).sum()) / POOL
    alg = {'nsr_nerf_prepass': 512.0 * m1, 'nsr_nerf_render_fwd': 512.0 * k1, 'nsr_nerf_field_bwd': 512.0 * k1,
           'nsr_nerf_field_bwd_tc': 512.0 * k1, 'nsr_nerf_table_scatter': 512.0 * k1, 'nsr_nerf_rays_fwd': 512.0 * evaluated}
    dom = max((n for n in alg if n in kern), key=lambda n: kern[n]['ms'] * kern[n]['launches_per_step'], default=None)
    roofline = None
    if dom is not None:
        ach = alg[dom] / (kern[dom]['ms'] * 1e-3) / 1e9
        step_bytes = 1024.0 * k1 + 512.0 * m1
        roofline = {'bound': 'hbm', 'kernel': dom, 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': None,
                    'peak_source': peak_src, 'algorithmic_bytes_per_launch': alg[dom], 'kernel_ms': kern[dom]['ms'],
                    'per_kernel': {n: {'algorithmic_bytes': alg[n], 'ms': kern[n]['ms'], 'achieved': alg[n] / (kern[n]['ms'] * 1e-3) / 1e9,
                                       'frac': alg[n] / (kern[n]['ms'] * 1e-3) / 1e9 / peak} for n in alg if n in kern},
                    'whole_step': {'algorithmic_bytes': step_bytes, 'achieved': step_bytes / (ms_step * 1e-3) / 1e9,
                                   'frac': step_bytes / (ms_step * 1e-3) / 1e9 / peak}}
    # ---- adjacent row 8f-2 (not part of `value`): the fused AdamW pass over all parameters, timed alone with CUDA events, L2 flushed
    adamw = None
    if world == 1:
        from nsr_b200.optim import FusedAdamW
        opt = FusedAdamW.for_model(model, lr=1e-2, betas=(0.9, 0.99), eps=1e-15)   # nerf-blender.yaml:74-79
        for p in params:
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        for _ in range(3):
            opt.step()
        lib.profile = {}   # CUDA events around every C-ABI call: the kernel's own duration, not Python's launch pace
        for i in range(20):
            flush.fill_(float(i))
            opt.step()
        torch.cuda.synchronize()
        n_calls = len(lib.profile['nsr_adamw_step']) // 20   # one launch per parameter tensor
        calls = [[a.elapsed_time(b) for a, b in lib.profile['nsr_adamw_step'][j * n_calls:(j + 1) * n_calls]] for j in range(20)]
        lib.profile = None
        opt_ms_all = sum(sum(c) for c in calls) / len(calls)       # all parameter tensors (the tiny ones are launch-latency bound)
        opt_ms = sum(max(c) for c in calls) / len(calls)           # the hash-table tensor's launch: the HBM-bound one
        n_par = max(p.numel() for p in params)
        opt_bytes = 30.0 * n_par   # p, g, m, v read (16 B) + p, m, v written (12 B) + fp16 copy written (2 B)
        adamw = {'kernel': 'adamw_kernel<1> (nsr_adamw_step), largest parameter tensor', 'params': n_par, 'ms': opt_ms,
                 'algorithmic_bytes': opt_bytes, 'achieved_GBps': opt_bytes / (opt_ms * 1e-3) / 1e9,
                 'frac_of_hbm_peak': opt_bytes / (opt_ms * 1e-3) / 1e9 / peak, 'all_tensors_ms': opt_ms_all,
                 'train_step_ms_with_optimizer': ms_step + opt_ms_all}
    # DRAM traffic of the dominant kernel from the committed ncu capture (per launch, same workload): far BELOW the algorithmic bytes
    # because the table and its gradient are L2 resident
    ncu_info = {}
    try:
        prof = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles')
        name = 'r2_ncu_traffic.json' if os.path.exists(os.path.join(prof, 'r2_ncu_traffic.json')) else 'r1_ncu_traffic.json'
        with open(os.path.join(prof, name)) as fh:
            ncu_info = json.load(fh)
    except (OSError, ValueError):
        pass
    if roofline is not None and dom in ncu_info:
        roofline['traffic'] = ncu_info[dom].get('dram_bytes_per_launch')
        roofline['traffic_source'] = ncu_info.get('source')
    if roofline is not None and dom in ('nsr_nerf_field_bwd', 'nsr_nerf_field_bwd_tc') and dom in ncu_info:
        # the table (25 MB fp16) and its gradient (50 MB fp32) live in the 126 MB L2: the kernel's real ceiling is the L2 atomic unit.
        # ~80 REDs (8-byte red.global.add.v2.f32) per kept sample after run merging = ncu RED sectors / K
        # (profiles/r1_ncu_traffic.json); 140 G RED/s = scatter-only micro-benchmark at full occupancy
        # (profiles/r1_gather_scatter_microbench.md).
        info = ncu_info.get(dom, {})
        reds = (info['red_sectors_per_launch'] / info['kept_samples'] if 'red_sectors_per_launch' in info else 79.2) * k1
        roofline['secondary'] = {'bound': 'l2_red', 'unit': 'G RED/s', 'achieved': reds / (kern[dom]['ms'] * 1e-3) / 1e9, 'peak': 140.0,
                                 'frac': reds / (kern[dom]['ms'] * 1e-3) / 1e9 / 140.0,
                                 'source': 'REDs/sample from ncu (profiles/r1_ncu_traffic.json); peak = measured scatter-only floor (profiles/r1_gather_scatter_microbench.md)'}
    cpu = time_cpu(4, 1, n_rays=CPU_SAMPLE_RAYS) if world == 1 else None   # ~5 s of CPU work: the C2 port (secondary)
    cpu_c1 = time_cpu_c1(4, 1) if world == 1 else None                       # ~10-15 s: BASELINE.json config 1 (primary)
    extra = {}
    if world == 1 and not args.no_extra:
        del gstep
        torch.cuda.empty_cache()
        for name in ('C3', 'C4'):
            try:
                extra[name] = neus_config(name, dev, min(args.steps, 20), max(3, min(args.warmup, 5)), flush, peak, peak_src)
            except Exception as e:   # a sub-line must never take the headline down
                extra[name] = {'error': f'{type(e).__name__}: {e}'}
    line = {
        'metric': 'rays/sec fwd+bwd (NeRF-Synthetic lego shape)', 'value': N_RAYS * world * args.steps / (ms * 1e-3), 'unit': 'rays/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': max(3, args.warmup), 'ms_per_step': ms_step, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
        'timing': {'statistic': 'median of the per-step CUDA-event times (max over ranks)', 'ms_per_step_mean': ms_mean,
                   'e2e_ms_per_step_median': ms_e2e / args.steps, 'e2e_ms_per_step_mean': ms_e2e_mean},
        'config': {'workload': WORKLOAD['C2'],
                   'rays_per_gpu': N_RAYS, 'evaluated_samples_per_step_per_gpu': evaluated, 'marched_samples_per_step': marched, 'kept_samples_per_step': kept,
                   'samples_per_s': kept * args.steps / (ms * 1e-3), 'l2': 'flushed (256 MB write) before every timed step',
                   'parallelism': f'dp{world}' if world > 1 else 'single',
                   'step': 'mask march + per-ray forward (early termination) + fused smooth-L1 loss + backward, one CUDA graph (nsr_b200.graph.GraphedStep)' + (f' + gradient mean over the ranks: {sync_desc}' if world > 1 else ''),
                   'eager_api_ms_per_step': ms_eager},
        'e2e': {'value': N_RAYS * world * args.steps / (ms_e2e * 1e-3), 'unit': 'rays/s',
                'h2d_bytes_per_step': N_RAYS * 6 * 4 + N_RAYS * 3 * 4, 'd2h_bytes_per_step': 4},
        'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline, 'kernels_ms': {k: round(v['ms'], 5) for k, v in kern.items()},
    }
    if adamw is not None:
        line['optimizer'] = adamw
    if cpu_c1 is not None:
        line['cpu_baseline'] = {'value': cpu_c1['rays_per_s'], 'unit': 'rays/s', 'cores': cpu_c1['cores'], 'kind': 'port',
                                'config': 'C1 (BASELINE.json configs[0]): nerf-blender with VanillaFrequency (10 / 4 frequencies) + VanillaMLP fields, 4096 rays, CPU only',
                                'sample': f"4 steps x {cpu_c1['n_rays']} rays (marched {cpu_c1['marched']:.0f}, kept {cpu_c1['kept']:.0f} samples/step), fwd+bwd, "
                                          f"the reference's torch field classes restated in oracle/mlp.py (pinned bit-for-bit by tests/test_oracle_golden.py) inside "
                                          f"the CPU oracle's marching / compositing, fp32, {cpu_c1['cores']} threads"}
    if cpu is not None:
        line['cpu_baseline_secondary'] = {'value': cpu['rays_per_s'], 'unit': 'rays/s', 'cores': cpu['cores'], 'kind': 'port',
                                          'config': 'C2 arithmetic (hash grid + 64-wide MLPs) on the CPU',
                                          'sample': f"4 steps x {cpu['n_rays']} rays of the C2 workload (kept {cpu['kept']:.0f} samples/step), fwd+bwd, "
                                                    f"fp32 CPU oracle, {cpu['cores']} threads"}
    if extra:
        line['extra'] = extra
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)  # see above: skip the NCCL teardown


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='C2', choices=['C2', 'C3', 'C4'], help='headline config (C3 / C4: single GPU)')
    ap.add_argument('--no-extra', action='store_true', help='skip the C3 / C4 sub-lines of the default run')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs and gradients of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the GPU path (--impl ours)')
    if args.impl == 'reference':
        reference_arm(args)
    elif args.config == 'C2':
        gpu_arm(args)
    else:
        neus_arm(args)


if __name__ == '__main__':
    main()
