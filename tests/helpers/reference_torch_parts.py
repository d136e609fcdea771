"""Run in a subprocess by tests/test_reference_dropin.py.  Compares the PRODUCT's pure-torch pieces (nsr_b200.models.common / networks /
fields / neus_model: the parts of the drop-in models that are not CUDA kernels) DIRECTLY with the reference's own functions and classes
(models/utils.py, models/network_utils.py, models/geometry.py, models/neus.py) on the CPU: same inputs, same seeds.  The original's
values are stored in tests/golden/reference_torch_parts.npz (tests/helpers/golden_ref.py; ``--record DIR`` re-creates it)."""
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
    T = Tape('reference_torch_parts')
    from nsr_b200.config import Config, to_primitive
    import nsr_b200.nerfacc as nsr_nerfacc
    nsr_nerfacc.install_as_reference_modules()
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
        from models import utils as rutils, network_utils as rnet, geometry as rgeo, neus as rneus
    from nsr_b200 import models as ours, configs
    from nsr_b200.models import common as ocommon, networks as onet, fields as ofields, neus_model as oneus
    from nsr_b200.nerfacc import ContractionType

    res = {}
    g = torch.Generator().manual_seed(0)

    def mx(a, b):
        a, b = pick(a, b)
        return float((a.double() - b.double()).abs().max()) if a.numel() else 0.0

    # 1. activations: value and gradient
    x = torch.randn(400, generator=g) * 3
    acts = {}
    for name in ('none', None, 'scale2.5', 'clamp1.5', 'mul0.5', 'lin2srgb', 'trunc_exp', '+1.5', '-0.25', 'sigmoid', 'tanh', 'relu', 'softplus',
                 'Sigmoid', 'ReLU'):
        a = x.clone().requires_grad_(True)
        ya = ocommon.get_activation(name)(a)
        ya.sum().backward()

        def ref_act():
            b = x.clone().requires_grad_(True)
            yb = rutils.get_activation(name)(b)
            yb.sum().backward()
            return yb.detach(), b.grad
        yb, gb = T.ref(f'act/{name}', ref_act)
        acts[str(name)] = max(mx(ya.detach(), yb), mx(a.grad, gb))
    res['activations'] = acts
    # 2. scale_anything, contraction
    d = torch.randn(50, 3, generator=g) * 4
    res['scale_anything'] = max(mx(ocommon.scale_anything(d, (-1.5, 1.5), (0, 1)), T.ref('scale/box', lambda: rutils.scale_anything(d, (-1.5, 1.5), (0, 1)))),
                                mx(ocommon.scale_anything(d, None, (2, 5)), T.ref('scale/none', lambda: rutils.scale_anything(d, None, (2, 5)))))
    res['contract'] = max(mx(ofields.contract_to_unisphere(d.clone(), 1.5, ContractionType.AABB),
                             T.ref('contract/aabb', lambda: rgeo.contract_to_unisphere(d.clone(), 1.5, ContractionType.AABB))),
                          mx(ofields.contract_to_unisphere(d.clone(), 1.5, ContractionType.UN_BOUNDED_SPHERE),
                             T.ref('contract/sphere', lambda: rgeo.contract_to_unisphere(d.clone(), 1.5, ContractionType.UN_BOUNDED_SPHERE))))
    # 3. chunk_batch: dict / tuple / tensor / None results, with and without the move to the CPU
    data = torch.randn(1000, 3, generator=g)
    fns = {'dict': lambda t: {'a': t * 2, 'b': t.sum(-1)}, 'tuple': lambda t: (t + 1, t.norm(dim=-1)), 'tensor': lambda t: t * t,
           'none': lambda t: None}
    cb = {}
    for name, fn in fns.items():
        for to_cpu in (True, False):
            a, b = ocommon.chunk_batch(fn, 256, to_cpu, data), T.ref(f'chunk_batch/{name}/{to_cpu}', lambda: rutils.chunk_batch(fn, 256, to_cpu, data))
            if a is None or b is None:
                cb[f'{name}/{to_cpu}'] = 0.0 if (a is None and b is None) else 1.0
            elif isinstance(a, dict):
                cb[f'{name}/{to_cpu}'] = max(mx(a[k], b[k]) for k in b) if sorted(a) == sorted(b) else 1.0
            elif isinstance(a, (tuple, list)):
                cb[f'{name}/{to_cpu}'] = max(mx(u, v) for u, v in zip(a, b)) if type(a) == type(b) and len(a) == len(b) else 1.0
            else:
                cb[f'{name}/{to_cpu}'] = mx(a, b)
    res['chunk_batch'] = cb
    # 4. VanillaFrequency with the masking schedule
    fq = {}
    for n_mask in (0, 1000):
        cfgf = {'n_frequencies': 6, 'n_masking_step': n_mask}
        a, b = onet.VanillaFrequency(3, dict(cfgf)), rnet.VanillaFrequency(3, dict(cfgf)) if T.recording else None
        for step in (0, 1, 250, 999, 5000):
            a.update_step(0, step)
            xx = torch.rand(40, 3, generator=g)
            fq[f'{n_mask}/{step}'] = mx(a(xx), T.ref(f'freq/{n_mask}/{step}', lambda: (b.update_step(0, step), b(xx))[1]))
        fq[f'{n_mask}/dims'] = float(a.n_output_dims != T.ref(f'freq/{n_mask}/dims', lambda: b.n_output_dims))
    res['vanilla_frequency'] = fq
    # 5. VanillaMLP: same seed => the same initial parameters (draw for draw) and outputs, every init variant of the reference's configs
    vm = {}
    for name, (din, dout, c) in {'relu_1': (32, 8, dict(n_hidden_layers=1)), 'relu_2': (24, 3, dict(n_hidden_layers=2)),
                                 'sphere_wn': (35, 13, dict(n_hidden_layers=1, sphere_init=True, sphere_init_radius=0.5, weight_norm=True)),
                                 'sphere_2': (35, 13, dict(n_hidden_layers=2, sphere_init=True, sphere_init_radius=0.7))}.items():
        c = dict(c, n_neurons=64, output_activation='none', activation='ReLU')
        torch.manual_seed(123)
        a = onet.VanillaMLP(din, dout, dict(c))
        if T.recording:
            torch.manual_seed(123)
            b = rnet.VanillaMLP(din, dout, dict(c))
        sa, sb = a.state_dict(), T.ref(f'vanilla_mlp/{name}/state', lambda: b.state_dict())
        xx = torch.randn(30, din, generator=g)
        vm[name] = {'keys': sorted(sa) == sorted(sb), 'params': max(mx(sa[k], sb[k]) for k in sb),
                    'out': mx(a(xx), T.ref(f'vanilla_mlp/{name}/out', lambda: b(xx).detach()))}
    res['vanilla_mlp'] = vm
    # 5b. sphere initialisation written into a tcnn-layout flat parameter vector (models/network_utils.py:142-173)
    class Flat(torch.nn.Module):
        def __init__(self, n):
            super().__init__()
            self.params = torch.nn.Parameter(torch.zeros(n))
    tc = {}
    for otype, n_hidden in (('FullyFusedMLP', 1), ('FullyFusedMLP', 3), ('CutlassMLP', 2)):
        c = Config(dict(otype=otype, n_neurons=64, n_hidden_layers=n_hidden))
        pad = 16 if otype == 'FullyFusedMLP' else 8
        n_in, n_out = (35 + pad - 1) // pad * pad, (13 + pad - 1) // pad * pad
        n = (n_in + n_out) * 64 + (n_hidden - 1) * 64 * 64
        a, b = Flat(n), Flat(n)
        torch.manual_seed(7)
        onet.sphere_init_tcnn_network(35, 13, c, a)

        def ref_init():
            torch.manual_seed(7)
            rnet.sphere_init_tcnn_network(35, 13, c, b)
            return b.params.detach()
        tc[f'{otype}/{n_hidden}'] = mx(a.params.detach(), T.ref(f'sphere_init_tcnn/{otype}/{n_hidden}', ref_init))
    res['sphere_init_tcnn'] = tc
    # 6. VarianceNetwork incl. the modulation schedule; NeuSModel.get_alpha through the models
    vn = {}
    for c in (dict(init_val=0.3, modulate=False), dict(init_val=0.5, modulate=True, mod_start_steps=100, reach_max_steps=1000, max_inv_s=64.0)):
        a, b = oneus.VarianceNetwork(Config(c)), rneus.VarianceNetwork(Config(c)) if T.recording else None
        for step in (0, 50, 100, 101, 500, 2000):
            a.update_step(0, step)
            inv_s, val = T.ref(f"variance/{c['modulate']}/{step}", lambda: (b.update_step(0, step), b.inv_s.detach(), b(torch.zeros(4, 3)).detach())[1:])
            vn[f"{c['modulate']}/{step}"] = max(mx(a.inv_s.detach(), inv_s), mx(a(torch.zeros(4, 3)).detach(), val))
    res['variance'] = vn
    cfg = configs.neus_blender()
    ma, mb = ours.make('neus', cfg), ref_models.make('neus', Config(configs.neus_blender())) if T.recording else None
    ga = {}
    for step in (0, 5000, 40000):
        ma.train()
        ma.update_step(0, step + 1)    # +1: not a multiple of 16 => no occupancy refresh (needs CUDA in the product)
        if T.recording:
            mb.train()
            mb.update_step(0, step + 1)
        k = 200
        sdf, nrm = torch.randn(k, generator=g) * 0.1, torch.nn.functional.normalize(torch.randn(k, 3, generator=g), dim=-1)
        dirs, dists = torch.nn.functional.normalize(torch.randn(k, 3, generator=g), dim=-1), torch.rand(k, 1, generator=g) * 0.01
        alpha, ratio = T.ref(f'get_alpha/{step}', lambda: (mb.get_alpha(sdf, nrm, dirs, dists).detach(), mb.cos_anneal_ratio))
        ga[str(step)] = max(mx(ma.get_alpha(sdf, nrm, dirs, dists).detach(), alpha), abs(ma.cos_anneal_ratio - ratio))
    res['get_alpha'] = ga
    step_size, aabb = T.ref('render_constants', lambda: (mb.render_step_size, mb.scene_aabb))
    res['render_constants'] = {'step': abs(ma.render_step_size - step_size), 'aabb': mx(ma.scene_aabb, aabb)}
    md = ours.make('neus', configs.neus_dtu())
    me = T.ref('render_constants_bg', lambda: (lambda e: dict(cone=e.cone_angle_bg, step=e.render_step_size_bg, near=e.near_plane_bg,
                                                              far=e.far_plane_bg))(ref_models.make('neus', Config(configs.neus_dtu()))))
    res['render_constants_bg'] = {'cone': abs(md.cone_angle_bg - me['cone']), 'step': abs(md.render_step_size_bg - me['step']),
                                  'near': abs(md.near_plane_bg - me['near']), 'far': abs(md.far_plane_bg - me['far'])}
    na = ours.make('nerf', configs.nerf_blender())
    nb_step, nb_aabb = T.ref('render_constants_nerf', lambda: (lambda e: (e.render_step_size, e.scene_aabb))(ref_models.make('nerf', Config(configs.nerf_blender()))))
    res['render_constants_nerf'] = {'step': abs(na.render_step_size - nb_step), 'aabb': mx(na.scene_aabb, nb_aabb)}
    if T.recording:
        T.save()
    print('RESULT ' + json.dumps(res))


if __name__ == '__main__':
    main()
