"""The fused NeRF step against the CPU oracle on inputs built to reach the edges of its kernels, which the seeded synthetic scene of
test_gpu_nerf.py never reaches (there no ray needs more than 8 chunks of 32 samples):

* long rays: every cell occupied and a low density, so that rays along the box diagonals keep ~1024 samples (32 chunks of the per-ray
  forward's transmittance carry, every queue bin of nsr_chunk_bin, the reverse suffix carry of the ray backwards);
* prescribed counts: rays whose origin sits (n - 1/4) steps before the exit face have exactly n lattice samples without jitter; batches of
  them have a kept total K of 1, 63, 64, 65, 127, 128, 129 and 32 m +- 1 (the tail tiles of the 64-row and 128-row backwards);
* walls: a density step the rays end on, swept along the ray direction in fractions of a step so that the kept count takes every residue
  mod 32 (early termination at and next to chunk edges); on the steep wall (the density feature of the table x100) the raw density of
  kept samples passes 15, where the backward of trunc_exp clamps (and where an exclusive transmittance sum taken as incl - sd loses its
  earlier terms to rounding); the same steepness from an MLP output weight of 4000 marks the fp16 headroom of the tile backwards' loss scale;
* faces and degenerate rays: rays lying in a box face or edge (unit-cube coordinate exactly 0 or 1), grazing rays with 0, 1 and 2
  samples, zero direction components, misses, and the same ray repeated 2, 3 and 33 times (run merging of the table scatter across ray
  boundaries; 33 one-sample rays make a whole scatter warp of equal cells);
* batch sizes 1, 7, 9, 257 and 4097 (ragged CTAs, the per-256-ray block sums of nsr_pack_kept_scan), with and without the fused kept scan;
* single-term losses (colour, opacity, depth, a weights-only distortion loss and the combined loss with it) and scaled losses
  c * L, c = 2^-16 .. 2^16, against the oracle for every backward form.

Same oracle and tolerances as test_gpu_nerf.check_parity: kept sets exactly equal except samples within 1e-3 (relative) of early_stop_eps;
colour |d| <= 5e-3, opacity <= 2e-3, depth <= 5e-3; network gradients cosine >= 0.995, table gradient cosine >= 0.99 and max error
<= 6e-2 of the largest entry.  The tests without the gpu mark assert, from the oracle alone, that the scenes reach what they are built for."""
import functools
import math

import numpy as np
import pytest
import torch

from oracle import march as omarch, models as omodels
from test_gpu_nerf import build, cos

R = 1.5
STEP = np.float32(1.732 * 2 * R / 1024)   # NeRFModel.render_step_size as the kernels receive it (fp32)
BG = torch.tensor([0.3, 0.6, 0.9])         # test_gpu_nerf.build's background
EPS = 1e-4                                 # early_stop_eps
MODES = ['per_ray', 'per_ray_split', 'per_ray_tc', 'per_ray_bwd', 'two_pass', False]
FUSED = MODES[:-1]
K_TARGETS = {1: [1], 63: [63], 64: [32, 32], 65: [33, 32], 95: [31, 64], 97: [33, 64], 127: [63, 64], 128: [64, 64], 129: [65, 64],
             1023: [1023], 1025: [1024, 1], 2047: [1023, 1024]}
BATCHES = [1, 7, 9, 257, 4097]


# ---------------------------------------------------------------------------------------------------------------------------------------
# rays
# ---------------------------------------------------------------------------------------------------------------------------------------
def _ray(o, d):
    return np.array(list(o) + list(d), np.float32)


def counted_ray(n, axis=0, sign=1.0, across=(0.1, -0.2)):
    """origin inside the box, (n - 1/4) steps before the exit face: with no jitter t_min = 0 and the midpoints (k + 1/2) step, k < n, are
    exactly the ones inside.  Along a coordinate axis up to 590 samples; longer rays run along the body diagonal (sign * (1, 1, 1))."""
    dist = (n - 0.25) * float(STEP)
    if dist < 2 * R - 0.02:
        o, d = [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]
        others = [a for a in range(3) if a != axis]
        o[others[0]], o[others[1]] = across
        o[axis], d[axis] = sign * (R - dist), sign
        return _ray(o, d)
    s = sign / math.sqrt(3.0)
    return _ray([sign * (R - dist / math.sqrt(3.0))] * 3, [s] * 3)


def grazing_ray(n, z=0.2):
    """cuts the box edge x = y = +R along (1, -1, 0) / sqrt(2) on a chord of (n + 1/4) steps: n samples without jitter."""
    c = (n + 0.25) * float(STEP) / math.sqrt(2.0)
    h = 1.0 / math.sqrt(2.0)
    return _ray([R - c - 0.5, R + 0.5, z], [h, -h, 0.0])


def camera_rays(n, seed):
    from nsr_b200 import synthetic
    return synthetic.sample_rays(n, seed=seed)


def diagonal_rays():
    """the four body diagonals, entered just outside a corner: ~1024 samples each"""
    out = []
    for s in ((1, 1, 1), (1, 1, -1), (1, -1, 1), (-1, 1, 1)):
        s = np.array(s, np.float64)
        out.append(_ray(-(R + 0.02) * s, s / math.sqrt(3.0)))
    return np.stack(out)


def inside_rays(n, seed):
    rng = np.random.default_rng(seed)
    o = rng.uniform(-1.2, 1.2, (n, 3))
    d = rng.normal(size=(n, 3))
    return np.concatenate([o, d / np.linalg.norm(d, axis=1, keepdims=True)], 1).astype(np.float32)


def face_rays():
    """(rays, role) for the faces-and-degenerate scene"""
    tiny = 1e-20   # keeps the slab test finite (0 / 0 is NaN there: a ray with an exactly zero component inside a face plane misses)
    rows = [
        (_ray([-R, 0.3, -1.6], [tiny, 0, 1]), 'face x01 = 0'),
        (_ray([R, -0.4, -1.6], [-tiny, 0, 1]), 'face x01 = 1'),
        (_ray([0.2, R, 1.6], [0, -tiny, -1]), 'face y01 = 1'),
        (_ray([0.35, -0.6, -R], [0.6, 0.8, tiny]), 'face z01 = 0'),
        (_ray([-R, -R, -1.6], [tiny, tiny, 1]), 'edge x01 = y01 = 0'),
        (_ray([R, R, 1.6], [-tiny, -tiny, -1]), 'edge x01 = y01 = 1'),
        (_ray([-R, 0.3, -1.6], [0, 0, 1]), 'in a face, exactly parallel: a miss'),
        (_ray([0.2, 0.3, -2.0], [0, 0, 1]), 'zero components'),
        (_ray([-1.6, 0.1, -1.7], [0.6, 0, 0.8]), 'zero component'),
        (_ray([0.1, -0.2, 0.3], [0, -1, 0]), 'zero components, inside'),
        (_ray([3, 3, 3], [1, 0, 0]), 'miss'),
        (_ray([0, 0, -3], [0, 0, -1]), 'miss: box behind'),
        (_ray([1.6, 0, 0], [0, 0, 1]), 'miss: parallel outside a face'),
        (grazing_ray(0), 'grazing 0'),
        (grazing_ray(1), 'grazing 1'),
        (grazing_ray(2), 'grazing 2'),
    ]
    cam = camera_rays(24, seed=61)
    rows += [(cam[0], 'camera x2')] * 2 + [(cam[1], 'camera')]
    rows += [(grazing_ray(2, z=-0.3), 'grazing 2 x3')] * 3 + [(cam[2], 'camera')]
    rows += [(counted_ray(1, axis=1, across=(0.4, 0.2)), 'one sample x33')] * 33 + [(cam[3], 'camera')]
    rows += [(counted_ray(40, axis=2, sign=-1.0), '40 samples x3')] * 3
    rows += [(r, 'camera') for r in cam[4:]]
    return np.stack([r for r, _ in rows]), [t for _, t in rows]


# ---------------------------------------------------------------------------------------------------------------------------------------
# scenes: rays + occupancy + density peak (+ jitter)
# ---------------------------------------------------------------------------------------------------------------------------------------
WALL_SWEEP = 100


def _all_occupied():
    return np.ones((128, 128, 128), bool)


@functools.lru_cache(maxsize=None)
def scene(name):
    from nsr_b200 import synthetic
    if name == 'long':
        rays = np.concatenate([camera_rays(160, seed=31), diagonal_rays(), inside_rays(40, seed=32)])
        jit = np.random.default_rng(33).random(len(rays)).astype(np.float32)
        jit[160:164] = 0.0   # the diagonals keep all 1024 lattice points
        return dict(rays=rays, binary=_all_occupied(), peak=0.5, jitter=jit)
    if name.startswith('K'):
        rays = [counted_ray(n, axis=i % 3, sign=(-1.0) ** i, across=(0.05 * i - 0.3, 0.2)) for i, n in enumerate(K_TARGETS[int(name[1:])])]
        rays.insert(1, _ray([3, 3, 3], [1, 0, 0]))   # a ray without samples between them
        rays = np.stack(rays)
        return dict(rays=rays, binary=_all_occupied(), peak=0.5, jitter=np.zeros(len(rays), np.float32))
    if name in ('wall', 'wall_steep', 'wall_peak4000'):
        # rays along +x ending on the ball's density step; the origins advance by 0.37 steps: the kept count takes every value on ~37 steps
        o = np.stack([-1.45 + np.arange(WALL_SWEEP) * 0.37 * float(STEP), np.full(WALL_SWEEP, 0.05), np.full(WALL_SWEEP, 0.03)], 1)
        sweep = np.concatenate([o, np.tile([1.0, 0.0, 0.0], (WALL_SWEEP, 1))], 1).astype(np.float32)
        rays = np.concatenate([sweep, camera_rays(48, seed=41)])
        # steep: raw density rises by ~27 per step at the wall (peak 40 on a density feature x100), so the last kept sample often has raw
        # density > 15.  wall_peak4000: the same steepness from the density MLP's output weight (see test_wall_from_mlp_weight)
        zero = np.zeros(len(rays), np.float32)
        return {'wall': dict(rays=rays, binary=_all_occupied(), peak=60.0, jitter=zero),
                'wall_steep': dict(rays=rays, binary=_all_occupied(), peak=40.0, feature_gain=100.0, jitter=zero),
                'wall_peak4000': dict(rays=rays, binary=_all_occupied(), peak=4000.0, jitter=zero)}[name]
    if name == 'faces':
        rays, _ = face_rays()
        return dict(rays=rays, binary=_all_occupied(), peak=0.5, jitter=np.zeros(len(rays), np.float32))
    if name.startswith('batch'):
        n = int(name[5:])
        rays = camera_rays(n, seed=70 + n % 13)
        return dict(rays=rays, binary=synthetic.occupancy(), peak=10.0, jitter=np.random.default_rng(n).random(n).astype(np.float32))
    raise KeyError(name)


SCENES = ['long', 'wall', 'wall_steep', 'faces'] + [f'K{k}' for k in K_TARGETS] + [f'batch{n}' for n in BATCHES]


@functools.lru_cache(maxsize=1)
def _init_params():
    from nsr_b200 import models, configs
    torch.manual_seed(1234)   # test_gpu_nerf.build's initialisation
    m = models.make('nerf', configs.nerf_blender())
    net, cnet = m.geometry.encoding_with_network, m.texture.network
    return net.params.detach().clone(), cnet.params.detach().clone(), net.mlp.n_params, net.grid


@functools.lru_cache(maxsize=4)
def _params(peak, gain, feature_gain):
    from nsr_b200 import synthetic
    d0, c0, nm, grid = _init_params()
    p = d0.clone()
    g = torch.Generator().manual_seed(7)
    p[nm:] = (torch.rand(grid.n_params, generator=g) * 2 - 1) * 0.1
    synthetic.shape_density(p, grid, nm, peak_logit=peak)
    off, res = int(grid.offset[4]), int(grid.res[4])   # shape_density's density feature: feature 0 of dense level 4
    p[nm:].view(-1, 2)[off:off + res ** 3, 0] *= feature_gain
    p[:nm] *= gain
    return p, c0 * gain


def scene_params(sc, gain=1.0):
    """test_gpu_nerf.build's parameters (table U(-0.1, 0.1) + synthetic.shape_density(peak)); gain multiplies every MLP weight"""
    return _params(sc['peak'], gain, sc.get('feature_gain', 1.0))


def marched_counts(name):
    sc = scene(name)
    o, d = sc['rays'][:, :3], sc['rays'][:, 3:6]
    aabb = np.array([-R] * 3 + [R] * 3, np.float32)
    t0, t1 = omarch.ray_interval(o, d, aabb, None, None, STEP, sc['jitter'])
    return omarch.march_lattice(o, d, aabb, sc['binary'], STEP, t0, t1)[3][:, 1]


def chunk_bin(cnt):
    """nsr_chunk_bin (csrc/common.cuh): queue bin of a ray with `cnt` marched samples"""
    ch = (cnt + 31) // 32
    return 0 if ch >= 17 else 1 if ch >= 13 else 2 if ch >= 9 else 3 if ch >= 5 else 4 if ch >= 3 else 5 if ch == 2 else 6 if ch == 1 else 7


# ---------------------------------------------------------------------------------------------------------------------------------------
# losses: the same torch code on the kernels' outputs and on the oracle's
# ---------------------------------------------------------------------------------------------------------------------------------------
def _coef(n, cols, seed, dev):
    return (torch.rand(n, cols, generator=torch.Generator().manual_seed(seed)) * 2 - 1).to(dev)


def distortion(out, n):
    """MipNeRF-360's distortion loss (torch_efficient_distloss.flatten_eff_distloss, systems/nerf.py:101-106), from the packed samples:
    sum over ray pairs w_i w_j |m_i - m_j| + 1/3 sum w_i^2 delta_i, per ray, averaged over the rays.  fp64 prefix sums."""
    w, m = out['weights'].double().view(-1), out['points'].double().view(-1)
    dl, ri = out['intervals'].double().view(-1), out['ray_indices'].long().view(-1)
    if w.numel() == 0:
        return w.sum()
    counts = torch.bincount(ri, minlength=n)
    first = (torch.cumsum(counts, 0) - counts)[ri]
    ew, ewm = torch.cumsum(w, 0) - w, torch.cumsum(w * m, 0) - w * m   # exclusive prefix sums over the batch
    pw, pwm = ew - ew[first], ewm - ewm[first]                         # ... within the ray
    return (2.0 * (w * (m * pw - pwm)).sum() + (w * w * dl).sum() / 3.0) / n


def loss_of(kind, out, n):
    dev = out['comp_rgb'].device
    rgb = lambda: omodels.smooth_l1_masked(out['comp_rgb'], torch.rand(n, 3, generator=torch.Generator().manual_seed(3)).to(dev), out['rays_valid'])
    opacity = lambda: (out['opacity'] * _coef(n, 1, 4, dev)).sum() / n
    depth = lambda: (out['depth'] * _coef(n, 1, 5, dev)).sum() / n
    combined = lambda: rgb() + 0.1 * out['opacity'].mean() + 0.05 * out['depth'].mean()
    return {'rgb': rgb, 'opacity': opacity, 'depth': depth, 'distortion': lambda: distortion(out, n).float(),
            'combined': combined, 'combined+distortion': lambda: combined() + distortion(out, n).float()}[kind]()


# ---------------------------------------------------------------------------------------------------------------------------------------
# oracle (one forward graph kept at a time; gradients cached per loss)
# ---------------------------------------------------------------------------------------------------------------------------------------
_FWD = {}
_GRADS = {}


def oracle(name, gain=1.0):
    key = (name, gain)
    if key not in _FWD:
        _FWD.clear()
        _GRADS.clear()
        from nsr_b200 import configs
        sc = scene(name)
        pd, pc = scene_params(sc, gain)
        dflat, cflat = pd.clone().requires_grad_(True), pc.clone().requires_grad_(True)
        P = omodels.NerfParams(configs.nerf_blender()['geometry']['xyz_encoding_config'], dflat, cflat)
        out = omodels.nerf_render(P, sc['rays'], sc['binary'], R, STEP, BG, jitter=sc['jitter'], emulate_fp16=True)
        _FWD[key] = (out, dflat, cflat)
    return _FWD[key][0]


def oracle_grads(name, kind, gain=1.0):
    key = (name, gain, kind)
    if key not in _GRADS:
        out = oracle(name, gain)
        _, dflat, cflat = _FWD[(name, gain)]
        L = loss_of(kind, out, len(scene(name)['rays']))
        gd, gc = torch.autograd.grad(L, [dflat, cflat], retain_graph=True, allow_unused=True)
        _GRADS[key] = (L.detach(), torch.zeros_like(dflat) if gd is None else gd, torch.zeros_like(cflat) if gc is None else gc)
    return _GRADS[key]


def kept_per_ray(out, n):
    return torch.bincount(out['ray_indices'].long(), minlength=n).numpy()


# ---------------------------------------------------------------------------------------------------------------------------------------
# coverage: the scenes reach what they are built for (oracle only, no GPU)
# ---------------------------------------------------------------------------------------------------------------------------------------
def test_coverage_every_queue_bin():
    bins = set()
    for name in SCENES:
        bins |= {chunk_bin(int(c)) for c in marched_counts(name)}
    assert bins == set(range(8))


def test_coverage_long_rays():
    n = len(scene('long')['rays'])
    out = oracle('long')
    kept, marched = kept_per_ray(out, n), marched_counts('long')
    assert kept.max() >= 1000 and (kept[160:164] >= 1023).all()   # the diagonals: 32 chunks
    assert np.array_equal(kept, marched)                            # T stays above early_stop_eps on every ray
    assert float(out['trans_pre'].min()) > 100 * EPS


@pytest.mark.parametrize('name', ['wall', 'wall_steep', 'wall_peak4000'])
def test_coverage_wall_residues(name):
    out = oracle(name)
    kept = kept_per_ray(out, len(scene(name)['rays']))[:WALL_SWEEP]
    marched = marched_counts(name)[:WALL_SWEEP]
    assert (kept < marched).all() and (kept > 64).all()       # every sweep ray ends on the wall, after two chunks or more
    assert set((kept % 32).tolist()) == set(range(32))         # ... with every residue of the 32-sample chunk
    if name != 'wall':   # kept samples whose raw density passes 15: trunc_exp's backward clamp is used
        assert float(out['density'].detach().max()) > math.exp(15.0) * 10


@pytest.mark.parametrize('k', list(K_TARGETS))
def test_coverage_k_targets(k):
    name = f'K{k}'
    out = oracle(name)
    assert int(out['num_samples']) == k
    kept = kept_per_ray(out, len(scene(name)['rays']))
    want = list(K_TARGETS[k])
    want.insert(1, 0)
    assert kept.tolist() == want and marched_counts(name).tolist() == want


def test_coverage_faces_and_duplicates():
    rays, roles = face_rays()
    out = oracle('faces')
    kept = kept_per_ray(out, len(rays))
    role = lambda t: [i for i, r in enumerate(roles) if r == t]
    for n in (0, 1, 2):
        assert kept[role(f'grazing {n}')].tolist() == [n]
    assert all(kept[i] == 0 for t in ('miss', 'miss: box behind', 'miss: parallel outside a face', 'in a face, exactly parallel: a miss')
               for i in role(t))
    assert kept[role('one sample x33')].tolist() == [1] * 33 and kept[role('grazing 2 x3')].tolist() == [2] * 3
    i33 = role('one sample x33')
    assert i33 == list(range(i33[0], i33[0] + 33))   # contiguous: 33 equal packed rows, a whole warp of the scatter
    # samples on the faces: unit-cube coordinates exactly 0 and 1 reach the hash grid and its scatter
    o, d = torch.from_numpy(rays[:, :3]), torch.from_numpy(rays[:, 3:6])
    ri = out['ray_indices'].long()
    x01 = (o[ri] + d[ri] * out['points'][:, None] + R) / (2 * R)
    assert (x01 == 0).any(dim=0)[:2].all() and (x01 == 1).any(dim=0)[:2].all()
    for t in ('face x01 = 0', 'face x01 = 1', 'edge x01 = y01 = 0', 'edge x01 = y01 = 1'):
        assert kept[role(t)[0]] > 500


# ---------------------------------------------------------------------------------------------------------------------------------------
# GPU: kernels against the oracle
# ---------------------------------------------------------------------------------------------------------------------------------------
def gpu_model(mode, name, gain=1.0, fuse_kept_scan=None, march_alloc=None):
    sc = scene(name)
    model = build(mode, n_rays=8, peak=sc['peak'])[0]
    pd, pc = scene_params(sc, gain)
    net, cnet = model.geometry.encoding_with_network, model.texture.network
    with torch.no_grad():
        net.params.copy_(pd.to(net.params.device))
        cnet.params.copy_(pc.to(cnet.params.device))
    model.occupancy_grid.set_binary(torch.from_numpy(sc['binary']))
    if fuse_kept_scan is not None:
        model._fused.fuse_kept_scan = fuse_kept_scan
    if march_alloc is not None:
        model._fused.march_alloc = march_alloc
    return model


def gpu_step(model, name, kind='combined', scale=1.0):
    sc = scene(name)
    D = torch.device('cuda:0')
    for p in model.parameters():
        p.grad = None
    out = model.forward_(torch.from_numpy(sc['rays']).to(D), jitter=torch.from_numpy(sc['jitter']))
    L = loss_of(kind, out, len(sc['rays']))
    (L * scale).backward()
    grad = lambda p: torch.zeros(p.shape) if p.grad is None else p.grad.cpu() / scale   # (the composed path leaves unreached .grad None)
    return out, L.detach(), grad(model.geometry.encoding_with_network.params), grad(model.texture.network.params)


def check_forward(out, ref):
    k, k_r = int(out['num_samples'].sum()), int(ref['num_samples'])
    ambiguous = int(((ref['trans_pre'] / EPS - 1).abs() < 1e-3).sum())
    assert abs(k - k_r) <= ambiguous
    if k == k_r:
        assert torch.equal(out['ray_indices'].cpu(), ref['ray_indices'])
        assert np.array_equal(out['points'].detach().cpu().numpy(), ref['points'].numpy())
        assert torch.allclose(out['weights'].detach().cpu(), ref['weights'].detach(), rtol=0.0, atol=2e-3)
    assert (out['comp_rgb'].detach().cpu() - ref['comp_rgb'].detach()).abs().max().item() <= 5e-3
    assert (out['opacity'].detach().cpu() - ref['opacity'].detach()).abs().max().item() <= 2e-3
    assert (out['depth'].detach().cpu() - ref['depth'].detach()).abs().max().item() <= 5e-3


def check_grads(gd, gc, gd_r, gc_r, nm=3072):
    assert torch.isfinite(gd).all() and torch.isfinite(gc).all()
    for got, ref, c in ((gc, gc_r, 0.995), (gd[:nm], gd_r[:nm], 0.995), (gd[nm:], gd_r[nm:], 0.99)):
        top = ref.abs().max().item()
        if top == 0.0:   # the term does not reach this parameter block (e.g. the colour network under an opacity-only loss)
            assert got.abs().max().item() == 0.0
            continue
        assert cos(got, ref) >= c
        assert (got - ref).abs().max().item() <= 6e-2 * top


def check_against_oracle(mode, name, kind='combined', gain=1.0, scale=1.0, **opts):
    model = gpu_model(mode, name, gain, **opts)
    out, L, gd, gc = gpu_step(model, name, kind, scale)
    ref = oracle(name, gain)
    check_forward(out, ref)
    L_r, gd_r, gc_r = oracle_grads(name, kind, gain)
    assert abs(L.item() - L_r.item()) <= 2e-3 * abs(L_r.item()) + 1e-5
    check_grads(gd, gc, gd_r, gc_r, model.geometry.encoding_with_network.mlp.n_params)
    return model, out


# The composed path keeps tcnn's fixed fp16 loss scale (ops.LOSS_SCALE): on the long-ray scene its table gradients (~1e-8 an entry) fall
# into fp16's subnormal range and lose the precision the tolerances ask for, as the reference's would.  It runs on every other scene.
# Like tcnn, it also hands the colour network's input gradient back in fp16 without the loss scale.  On the steep wall the density output
# (~4000) saturates the colour sigmoid, and that gradient falls below fp16's normal range.  Under the colour-only loss it is the whole
# gradient of the density MLP's feature rows.  Rounding just that gradient to fp16 in the oracle gives the same cosine (0.967).
_COMPOSED_FP16_DX = pytest.mark.xfail(strict=True, reason="composed path: the colour network's input gradient is fp16 and unscaled "
                                                         "(tcnn's contract); it underflows behind the saturated sigmoid of the steep wall")


def _cases(name, *args):
    """(name, *args, mode) for every form the scene runs on"""
    if name == 'long':
        return [(name, *args, m) for m in FUSED]
    xfail = (name, *args) == ('wall_steep', 'rgb')
    return [(name, *args, m) for m in FUSED] + [pytest.param(name, *args, False, marks=_COMPOSED_FP16_DX) if xfail else (name, *args, False)]


@pytest.mark.gpu
@pytest.mark.parametrize('name,mode', [c for s in SCENES if not s.startswith('batch') for c in _cases(s)])
def test_scene_parity(name, mode):
    """combined loss (test_gpu_nerf's), forward and gradients, every form"""
    check_against_oracle(mode, name)


@pytest.mark.gpu
@pytest.mark.parametrize('n,fuse,mode', [(n, f, m) for n in BATCHES for f in (False, True) for m in MODES if f is False or m])
def test_batch_sizes(n, fuse, mode):
    """ragged CTAs in the marcher, the per-ray forward, the pack kernel and the ray backwards; fuse: nsr_pack_kept_scan (its per-256-ray
    block sums are read from 257 rays on)"""
    check_against_oracle(mode, f'batch{n}', fuse_kept_scan=fuse if mode else None)


@pytest.mark.gpu
@pytest.mark.parametrize('name,kind,mode', [c for s in ('long', 'wall', 'wall_steep')
                                            for k in ('rgb', 'opacity', 'depth', 'distortion', 'combined+distortion') for c in _cases(s, k)])
def test_single_term_losses(name, kind, mode):
    """each term of the loss on its own: a wrong depth or weights term cannot hide under the colour term"""
    check_against_oracle(mode, name, kind)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', FUSED)
@pytest.mark.parametrize('log2c', [-16, -6, 0, 6, 16])
def test_loss_scale_invariance(mode, log2c):
    """grad(c L) / c == grad(L) of the oracle: the automatic fp16 loss scale neither flushes nor overflows"""
    check_against_oracle(mode, 'long', 'combined', scale=2.0 ** log2c)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', MODES)
def test_amplifying_mlp_weights(mode):
    """every MLP weight x3: the hidden layers amplify the dgrad chain against the headroom of the automatic loss scale"""
    check_against_oracle(mode, 'long', 'combined+distortion', gain=3.0)


# The tile backwards (and the two-pass one) scale the loss so that the largest d_sraw / d_rgb becomes 2^8 and then run the dgrad chain in
# fp16 through the MLP weights: an output weight w keeps it finite only while about |w| * 2^8 < 65504, i.e. |w| < 256.  A density wall made
# steep by an output weight of 4000 (instead of by the table, as in wall_steep) overflows there.  The per-ray backward derives its scale
# from a bound on dL/dw (target 2^6), which leaves it enough headroom on this scene.
_FP16_DGRAD_BOUND = pytest.mark.xfail(strict=True, reason='fp16 dgrad overflow: MLP output weight 4000 x loss-scale target 2^8 > 65504')


@pytest.mark.gpu
@pytest.mark.parametrize('mode', [pytest.param(m, marks=_FP16_DGRAD_BOUND) if m in ('per_ray', 'per_ray_split', 'per_ray_tc', 'two_pass') else m
                                  for m in MODES])
def test_wall_from_mlp_weight(mode):
    check_against_oracle(mode, 'wall_peak4000')


def _outputs(model, name):
    out, _, gd, gc = gpu_step(model, name)
    return out, gd, gc


@pytest.mark.gpu
@pytest.mark.parametrize('name', SCENES)
def test_allocating_and_scan_marchers_agree(name):
    """nsr_march_rays_alloc and nsr_march_rays_mask + nsr_scan_counts_order: the same samples and the same per-ray results, bit for bit"""
    model = gpu_model('per_ray', name, march_alloc=True)
    a, gd_a, gc_a = _outputs(model, name)
    model._fused.march_alloc = False
    b, gd_b, gc_b = _outputs(model, name)
    assert int(a['num_samples']) == int(b['num_samples'])
    for key in ('ray_indices', 'points', 'comp_rgb', 'opacity', 'depth', 'weights'):
        assert torch.equal(a[key], b[key]), key
    assert cos(gd_a, gd_b) >= 0.999999 and cos(gc_a, gc_b) >= 0.999999   # (fp32 atomics: order differs)


@pytest.mark.gpu
@pytest.mark.parametrize('name', SCENES)
def test_per_ray_and_two_pass_agree(name):
    """the two fused forwards share the density code and the 32-sample chunking of the transmittance scan: identical kept sets"""
    a, _, _ = _outputs(gpu_model('per_ray', name), name)
    b, _, _ = _outputs(gpu_model('two_pass', name), name)
    assert int(a['num_samples']) == int(b['num_samples']) and torch.equal(a['ray_indices'], b['ray_indices'])
    assert torch.equal(a['points'], b['points']) and torch.allclose(a['weights'], b['weights'], rtol=0.0, atol=1e-6)
    assert (a['comp_rgb'] - b['comp_rgb']).abs().max().item() <= 1e-5
