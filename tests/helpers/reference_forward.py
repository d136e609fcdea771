"""Run in a subprocess by tests/test_reference_dropin.py.  Executes ``forward_`` of the UNMODIFIED reference models (models/nerf.py:61-127,
models/neus.py:205-287) on the CPU -- their third-party ops replaced by per-op stand-ins built from the oracle (tests/helpers/cpu_thirdparty.py)
-- and compares every output with the oracle's restatement of the same orchestration (oracle/models.py: nerf_render, neus_render).  Both
sides use the weights of the drop-in model built from seeds on the same stand-ins; the reference's outputs, gradients and constants are
stored in tests/golden/reference_forward.npz (tests/helpers/golden_ref.py; ``--record DIR`` re-creates it)."""
import contextlib
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden_ref import Tape, pick  # noqa: E402


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def main():
    T = Tape('reference_forward')
    import cpu_thirdparty as tp
    from nsr_b200.config import Config, to_primitive
    from nsr_b200 import configs, synthetic
    from oracle import models as om
    sys.modules['tinycudann'] = tp.tinycudann_module()
    nerfacc, inter = tp.nerfacc_modules()
    sys.modules['nerfacc'], sys.modules['nerfacc.intersection'] = nerfacc, inter
    quiet = lambda *a, **k: None
    rz = _stub('pytorch_lightning.utilities.rank_zero', rank_zero_info=quiet, rank_zero_debug=quiet, rank_zero_warn=quiet)
    ut = _stub('pytorch_lightning.utilities', rank_zero=rz)
    _stub('pytorch_lightning', utilities=ut, LightningModule=torch.nn.Module, LightningDataModule=object, Callback=object)
    _stub('torch_efficient_distloss', flatten_eff_distloss=None)

    class _OmegaConf:
        @staticmethod
        def register_new_resolver(*a, **k):
            pass

        @staticmethod
        def to_container(c, resolve=True):
            return to_primitive(c)
    _stub('omegaconf', OmegaConf=_OmegaConf)
    for name in ('imageio', 'cv2', 'trimesh', 'mcubes'):
        _stub(name, marching_cubes=None)
    mc, mp = _stub('matplotlib.colors'), _stub('matplotlib.pyplot')
    _stub('matplotlib', colors=mc, pyplot=mp, cm=types.SimpleNamespace())
    sysm = _stub('systems')
    sysm.utils = _stub('systems.utils', update_module_step=lambda m, e, s: m.update_step(e, s) if hasattr(m, 'update_step') else None)
    torch.cuda.device = lambda idx: contextlib.nullcontext()
    if T.recording:
        sys.path.insert(0, T.reference)
        import models as ref_models
    from nsr_b200 import models as ours, tcnn as our_tcnn

    def swap_tcnn(module):
        for name, child in list(module.named_children()):
            if isinstance(child, our_tcnn.NetworkWithInputEncoding):
                setattr(module, name, tp.NetworkWithInputEncoding(child.n_input_dims, child.n_output_dims, child.encoding_config, child.network_config))
            elif isinstance(child, our_tcnn.Encoding):
                setattr(module, name, tp.Encoding(child.n_input_dims, child.encoding_config))
            elif isinstance(child, our_tcnn.Network):
                setattr(module, name, tp.Network(child.n_input_dims, child.n_output_dims, child.network_config))
            else:
                swap_tcnn(child)

    def weights(kind, cfg, seed, prepare, name):
        """the drop-in model on the stand-ins, built from ``seed`` and prepared: the weights both sides use"""
        c = dict(cfg, fused=False)
        if 'geometry' in c:
            c['geometry'] = dict(c['geometry'], fused=False)
        torch.manual_seed(seed)
        m = ours.make(kind, c)
        swap_tcnn(m)
        with torch.no_grad():
            prepare(m)
        T.check_state(m, f'{name}/state')
        return m

    def reference(kind, cfg, m, run):
        """the unmodified reference model with the weights of ``m``, handed to run()"""
        ref = ref_models.make(kind, Config(cfg))
        missing, unexpected = ref.load_state_dict(m.state_dict(), strict=False)   # (the stand-in grid has no grid_coords / grid_indices)
        assert not missing and all('occupancy_grid' in k for k in unexpected), (missing, unexpected)
        return run(ref)

    binary = synthetic.occupancy()
    n = 192
    rays = synthetic.sample_rays(n, seed=21)
    bg = torch.tensor([0.3, 0.6, 0.9])
    res = {}

    def diff(a, b):   # a: the oracle's (or ours), b: the reference's
        a, b = pick(a, b)
        a, b = a.double(), b.double()
        assert a.shape == b.shape, (a.shape, b.shape)
        return float((a - b).abs().max()) if a.numel() else 0.0

    # ---- NeRF (nerf-blender.yaml)
    from oracle import neus as oneus
    from nsr_b200 import ops
    pts = (torch.rand(300, 3, generator=torch.Generator().manual_seed(9)) * 2 - 1) * 1.2
    keys = ('comp_rgb', 'opacity', 'depth', 'weights', 'points', 'intervals', 'ray_indices')
    cfg = configs.nerf_blender()
    cfg['randomized'] = False

    def prep_nerf(m):   # the bench's density bump: opaque ball => the sigma_fn pre-pass / visibility filter drops samples
        net = m.geometry.encoding_with_network
        flat = net.params.detach().clone()
        synthetic.shape_density(flat, ops.GridSpec(cfg['geometry']['xyz_encoding_config']), net.n_mlp)
        net.params.copy_(flat)
        m.occupancy_grid._binary.copy_(torch.from_numpy(binary))
    m = weights('nerf', cfg, 0, prep_nerf, 'nerf')

    def run_nerf(model):
        model.train()
        model.background_color = bg
        out = model.forward_(torch.from_numpy(rays))
        loss = out['comp_rgb'].square().mean() + 0.1 * out['opacity'].mean()
        loss.backward()
        model.update_step(0, 16)                                    # models/nerf.py:45-55: occ = density * render_step_size
        call = model.occupancy_grid.last_call
        with torch.no_grad():
            occ = call['occ_eval_fn'](pts)
        return {'keys': sorted(out), 'num_samples': int(out['num_samples']), 'out': {k: out[k].detach() for k in keys + ('rays_valid',)},
                'grads': [p.grad.clone() for p in (model.geometry.encoding_with_network.params, model.texture.network.params)],
                'render_step_size': float(model.render_step_size), 'occ': occ, 'occ_thre': call['occ_thre']}
    ref = T.ref('nerf', lambda: reference('nerf', cfg, m, run_nerf))
    out, g_ref = ref['out'], ref['grads']
    dflat = m.geometry.encoding_with_network.params.detach().clone().requires_grad_(True)
    cflat = m.texture.network.params.detach().clone().requires_grad_(True)
    P = om.NerfParams(cfg['geometry']['xyz_encoding_config'], dflat, cflat)
    P.one_gather = True
    o = om.nerf_render(P, rays, binary, 1.5, np.float32(ref['render_step_size']), bg, jitter=None, emulate_fp16=False)
    (o['comp_rgb'].square().mean() + 0.1 * o['opacity'].mean()).backward()
    res['nerf'] = {'keys': ref['keys'], 'num_samples': ref['num_samples'], 'num_samples_oracle': int(o['num_samples']),
                   'num_marched': int(o['num_marched']),
                   'diff': {k: diff(o[k], out[k]) for k in keys},
                   'rays_valid_equal': diff(o['rays_valid'], out['rays_valid']) == 0.0,
                   'grad_diff': [diff(dflat.grad, g_ref[0]) / (float(dflat.grad.abs().max()) + 1e-30),
                                 diff(cflat.grad, g_ref[1]) / (float(cflat.grad.abs().max()) + 1e-30)]}
    with torch.no_grad():
        dens, _ = om.nerf_field(P, pts, None, 1.5, emulate_fp16=False, density_only=True)
        res['nerf']['occ_fn'] = diff(dens[:, None] * ref['render_step_size'], ref['occ'])
    res['nerf']['occ_thre'] = ref['occ_thre']

    # ---- unbounded NeRF (nerf-colmap.yaml): sphere contraction, 256^3 grid, cone marching between the near and far planes
    cfg = configs.nerf_colmap()
    cfg['randomized'] = False
    bgb_nerf = np.random.default_rng(1).random((256, 256, 256)) < 0.3

    def prep_colmap(m):
        net = m.geometry.encoding_with_network
        flat = net.params.detach().clone()
        synthetic.shape_density(flat, ops.GridSpec(cfg['geometry']['xyz_encoding_config']), net.n_mlp, radius=1.0)
        net.params.copy_(flat)
        m.occupancy_grid._binary.copy_(torch.from_numpy(bgb_nerf))
    m = weights('nerf', cfg, 3, prep_colmap, 'nerf_colmap')
    rays_u = rays.copy()
    rays_u[:, :3] *= 1.0 / 1.5 * 0.4

    def run_colmap(model):
        model.train()
        model.background_color = bg
        out = model.forward_(torch.from_numpy(rays_u))
        (out['comp_rgb'].square().mean() + 0.1 * out['opacity'].mean() + 0.05 * out['depth'].mean()).backward()
        return {'num_samples': int(out['num_samples']), 'out': {k: out[k].detach() for k in keys},
                'grads': [p.grad.clone() for p in (model.geometry.encoding_with_network.params, model.texture.network.params)],
                'constants': [float(model.render_step_size), float(model.cone_angle), float(model.near_plane), float(model.far_plane)]}
    ref = T.ref('nerf_colmap', lambda: reference('nerf', cfg, m, run_colmap))
    out, g_ref, (step_u, cone_u, near_u, far_u) = ref['out'], ref['grads'], ref['constants']
    dflat = m.geometry.encoding_with_network.params.detach().clone().requires_grad_(True)
    cflat = m.texture.network.params.detach().clone().requires_grad_(True)
    P = om.NerfParams(cfg['geometry']['xyz_encoding_config'], dflat, cflat)
    P.one_gather = True
    o = om.nerf_unbounded_render(P, rays_u, bgb_nerf, 1.0, step_u, cone_u, near_u, far_u, bg, emulate_fp16=False)
    (o['comp_rgb'].square().mean() + 0.1 * o['opacity'].mean() + 0.05 * o['depth'].mean()).backward()
    res['nerf_colmap'] = {'num_samples': ref['num_samples'], 'num_samples_oracle': int(o['num_samples']), 'num_marched': int(o['num_marched']),
                          'diff': {k: diff(o[k], out[k]) for k in keys},
                          'grad_diff': [diff(dflat.grad, g_ref[0]) / (float(dflat.grad.abs().max()) + 1e-30),
                                        diff(cflat.grad, g_ref[1]) / (float(cflat.grad.abs().max()) + 1e-30)],
                          'constants': ref['constants']}

    # ---- NeuS (neus-blender.yaml)
    cfg = configs.neus_blender()
    cfg['randomized'] = False
    g = (np.arange(128) + 0.5) / 128 * 3.0 - 1.5
    X, Y, Z = np.meshgrid(g, g, g, indexing='ij')
    dist = np.sqrt(X ** 2 + Y ** 2 + Z ** 2)
    shell = (dist > 0.55) & (dist < 0.95)

    def prep_neus(m):   # sphere init zeroes the weights on the hash features: wake them up so the table matters
        v = m.geometry.network.layers[0].weight_v
        v[:, 3:] = torch.randn(v.shape[0], v.shape[1] - 3) * 0.05
        m.occupancy_grid._binary.copy_(torch.from_numpy(shell))
    m = weights('neus', cfg, 1, prep_neus, 'neus')
    names = ['geometry.encoding.encoding.params', 'texture.network.params', 'variance.variance', 'geometry.network.layers.0.weight_v']
    nkeys = ('comp_rgb', 'comp_normal', 'opacity', 'depth', 'sdf_samples', 'sdf_grad_samples', 'weights', 'points', 'intervals', 'ray_indices',
             'comp_rgb_full')

    def run_neus(model):
        model.train()
        model.update_step(0, 5000)
        model.background_color = bg
        out = model.forward_(torch.from_numpy(rays))
        eik = ((torch.linalg.norm(out['sdf_grad_samples'], ord=2, dim=-1) - 1.) ** 2).mean()
        (out['comp_rgb_full'].square().mean() + 0.1 * eik).backward()
        params = dict(model.named_parameters())
        call = model.occupancy_grid.last_call                   # models/neus.py:90-111 handed over by update_step(0, 5000) above
        with torch.no_grad():
            occ = call['occ_eval_fn'](pts * 0.6)
        return {'keys': sorted(out), 'num_samples': int(out['num_samples']), 'out': {k: out[k].detach() for k in nkeys},
                'grads': {k: params[k].grad.clone() for k in names}, 'inv_s': model.variance.inv_s.detach(),
                'cos_anneal_ratio': float(model.cos_anneal_ratio), 'render_step_size': float(model.render_step_size),
                'occ': occ, 'occ_thre': call['occ_thre']}
    ref = T.ref('neus', lambda: reference('neus', cfg, m, run_neus))
    out, g_ref = ref['out'], ref['grads']
    params = dict(m.named_parameters())
    P = om.NeusParams(cfg['geometry']['xyz_encoding_config'], params[names[0]], m.geometry.network, params[names[1]], params[names[2]])
    o = om.neus_render(P, rays, shell, 1.5, np.float32(ref['render_step_size']), bg, ref['cos_anneal_ratio'], jitter=None, emulate_fp16=False)
    eik = ((torch.linalg.norm(o['sdf_grad_samples'], ord=2, dim=-1) - 1.) ** 2).mean()
    (o['comp_rgb_full'].square().mean() + 0.1 * eik).backward()
    res['neus'] = {'keys': ref['keys'], 'num_samples': ref['num_samples'], 'num_samples_oracle': int(o['num_samples']),
                   'cos_anneal_ratio': ref['cos_anneal_ratio'],
                   'diff': {k: diff(o[k], out[k]) for k in nkeys},
                   'inv_s_diff': diff(o['inv_s'], ref['inv_s']),
                   'grad_diff': {k: diff(params[k].grad, g_ref[k]) / (float(params[k].grad.abs().max()) + 1e-30) for k in names}}
    with torch.no_grad():
        sdf = m.geometry(pts * 0.6, with_grad=False, with_feature=False)
        res['neus']['occ_fn'] = diff(oneus.occ_alpha(sdf, oneus.inv_s_from_variance(params[names[2]]), ref['render_step_size']), ref['occ'])
    res['neus']['occ_thre'] = ref['occ_thre']

    # ---- NeuS with learned background (neus-dtu.yaml: config C4)
    cfg = configs.neus_dtu()
    cfg['randomized'] = False
    r = cfg['radius']
    g = (np.arange(128) + 0.5) / 128 * 2 * r - r
    X, Y, Z = np.meshgrid(g, g, g, indexing='ij')
    dist = np.sqrt(X ** 2 + Y ** 2 + Z ** 2)
    shell = (dist > 0.35 * r) & (dist < 0.65 * r)
    bgb = np.random.default_rng(0).random((256, 256, 256)) < 0.3

    def prep_dtu(m):
        v = m.geometry.network.layers[0].weight_v
        v[:, 3:] = torch.randn(v.shape[0], v.shape[1] - 3) * 0.05
        m.geometry_bg.encoding_with_network.network.layers[-1].bias[0] = 2.5      # background densities ~ exp(1.5): visibly opaque
        m.occupancy_grid._binary.copy_(torch.from_numpy(shell))
        m.occupancy_grid_bg._binary.copy_(torch.from_numpy(bgb))
    m = weights('neus', cfg, 2, prep_dtu, 'neus_dtu')
    rays_c4 = rays.copy()
    rays_c4[:, :3] *= r / 1.5 * 0.6
    keys = ['comp_rgb', 'opacity', 'sdf_samples', 'sdf_grad_samples', 'weights', 'ray_indices', 'comp_rgb_bg', 'opacity_bg', 'depth_bg',
            'weights_bg', 'points_bg', 'intervals_bg', 'ray_indices_bg', 'comp_rgb_full']

    def run_dtu(model):
        model.train()
        model.update_step(0, 5000)
        model.background_color = bg
        out = model.forward_(torch.from_numpy(rays_c4))
        eik = ((torch.linalg.norm(out['sdf_grad_samples'], ord=2, dim=-1) - 1.) ** 2).mean()
        (torch.nn.functional.l1_loss(out['comp_rgb_full'], torch.full_like(out['comp_rgb_full'], 0.5)) + 0.1 * eik).backward()
        call_bg = model.occupancy_grid_bg.last_call             # models/neus.py:103-111: density * render_step_size_bg, its own threshold key
        with torch.no_grad():
            occ_bg = call_bg['occ_eval_fn'](pts * 3.0)
        return {'keys': sorted(out), 'num_samples': int(out['num_samples']), 'num_samples_bg': int(out['num_samples_bg']),
                'num_samples_full': int(out['num_samples_full']), 'out': {k: out[k].detach() for k in keys + ['rays_valid_full']},
                'grads': {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None},
                'constants': [float(model.render_step_size), float(model.render_step_size_bg), float(model.cone_angle_bg),
                              float(model.near_plane_bg), float(model.far_plane_bg), float(model.cos_anneal_ratio)],
                'occ_bg': occ_bg, 'occ_thre': [model.occupancy_grid.last_call['occ_thre'], call_bg['occ_thre']]}
    ref = T.ref('neus_dtu', lambda: reference('neus', cfg, m, run_dtu))
    out, g_ref = ref['out'], ref['grads']
    step, step_bg, cone_bg, near_bg, far_bg, ratio = ref['constants']
    params = dict(m.named_parameters())
    P = om.NeusParams(cfg['geometry']['xyz_encoding_config'], params['geometry.encoding.encoding.params'], m.geometry.network, None,
                      params['variance.variance'])
    P.color_mlp = m.texture.network
    ewn = m.geometry_bg.encoding_with_network
    Pbg = om.NeusBgParams(cfg['geometry_bg']['xyz_encoding_config'], ewn.encoding.encoding.params, ewn.network, m.texture_bg.network)
    o = om.neus_dtu_render(P, Pbg, rays_c4, shell, bgb, r, np.float32(step), step_bg, cone_bg, near_bg, far_bg, bg, ratio, emulate_fp16=False)
    eik = ((torch.linalg.norm(o['sdf_grad_samples'], ord=2, dim=-1) - 1.) ** 2).mean()
    (torch.nn.functional.l1_loss(o['comp_rgb_full'], torch.full_like(o['comp_rgb_full'], 0.5)) + 0.1 * eik).backward()
    res['neus_dtu'] = {'keys': ref['keys'], 'oracle_keys_missing': sorted(set(ref['keys']) - set(o)),
                       'num_samples': ref['num_samples'], 'num_samples_bg': ref['num_samples_bg'],
                       'num_samples_bg_oracle': int(o['num_samples_bg']), 'num_marched_bg': int(o['num_marched_bg']) if 'num_marched_bg' in o else -1,
                       'num_samples_full_equal': ref['num_samples_full'] == int(o['num_samples_full']),
                       'rays_valid_full_equal': diff(o['rays_valid_full'], out['rays_valid_full']) == 0.0,
                       'diff': {k: diff(o[k], out[k]) for k in keys},
                       'grad_diff': {k: diff(params[k].grad, gr) / (float(params[k].grad.abs().max()) + 1e-30) for k, gr in g_ref.items()},
                       'n_grads': len(g_ref)}
    with torch.no_grad():
        dens, _ = om.neus_bg_field(Pbg, pts * 3.0, None, r, emulate_fp16=False, density_only=True)
        res['neus_dtu']['occ_fn_bg'] = diff(dens[:, None] * step_bg, ref['occ_bg'])
    res['neus_dtu']['occ_thre'] = ref['occ_thre']
    if T.recording:
        T.save()
    print('RESULT ' + json.dumps(res))


if __name__ == '__main__':
    main()
