"""Run in a subprocess by tests/test_reference_dropin.py.  The torch fallback paths of the product's VolumeSDF (models/fields.py: analytic
normals through autograd when the fused kernel is off, finite-difference normals + laplacian with the ProgressiveBandHashGrid of the
Neuralangelo config) executed on the CPU -- their hash-grid encoding swapped for the oracle-backed stand-in
(tests/helpers/cpu_thirdparty.py) -- against the reference's own VolumeSDF (models/geometry.py:141-238) built on the same stand-in with the
same weights.  The original's values are stored in tests/golden/reference_sdf_paths.npz (tests/helpers/golden_ref.py; ``--record DIR``
re-creates it)."""
import contextlib
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden_ref import Tape, pick, amax  # noqa: E402


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def main():
    T = Tape('reference_sdf_paths')
    import cpu_thirdparty as tp
    from nsr_b200.config import Config, to_primitive
    from nsr_b200 import configs
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
        import models as ref_models                      # noqa: F401  (registers the reference classes)
        from models import geometry as rgeo, network_utils as rnet
        rnet.get_rank = lambda: 'cpu'                    # ProgressiveBandHashGrid allocates its mask on device=get_rank()
    from nsr_b200.models import fields as ofields
    from nsr_b200.nerfacc import ContractionType as OurCT

    res = {}

    def mx(a, b):
        a, b = pick(a, b)
        return float((a.double() - b.double()).abs().max())

    def pair(name, geo_cfg, steps):
        torch.manual_seed(0)
        our = ofields.VolumeSDF(Config(geo_cfg))
        our.contraction_type = OurCT.AABB
        # swap our CUDA-backed hash grid for the stand-in the reference was built on, then share every weight
        holder = our.encoding.encoding
        grid_cfg = dict(geo_cfg['xyz_encoding_config'], otype='HashGrid')
        if type(holder).__name__ == 'ProgressiveBandHashGrid':
            holder.encoding = tp.Encoding(3, grid_cfg)
        else:
            our.encoding.encoding = tp.Encoding(3, grid_cfg)
        with torch.no_grad():
            v = our.network.layers[0].weight_v if hasattr(our.network.layers[0], 'weight_v') else our.network.layers[0].weight
            v[:, 3:] = torch.randn(v.shape[0], v.shape[1] - 3) * 0.05
        if T.recording:   # the reference's VolumeSDF on the same stand-in, with our weights
            torch.manual_seed(0)
            ref = rgeo.VolumeSDF(Config(geo_cfg))
            ref.contraction_type = tp.ContractionType.AABB
            ref.load_state_dict(our.state_dict(), strict=True)
        T.check_state(our, f'{name}/state')
        out = {}
        pts = (torch.rand(300, 3, generator=torch.Generator().manual_seed(1)) * 2 - 1) * 0.8 * geo_cfg['radius']
        for step in steps:
            for mode in ('train', 'eval'):
                getattr(our, mode)()
                our.update_step(0, step)
                fd = geo_cfg['grad_type'] == 'finite_difference'
                a = our(pts.clone(), with_grad=True, with_feature=True, with_laplace=fd)

                def ref_run():
                    getattr(ref, mode)()
                    ref.update_step(0, step)
                    b = ref(pts.clone(), with_grad=True, with_feature=True, with_laplace=fd)
                    r = {'out': [x.detach() for x in b], 'level': ref.forward_level(pts).detach(),
                         'sdf_only': ref(pts.clone(), with_grad=False, with_feature=False).detach()}
                    if mode == 'train':
                        for p in ref.parameters():
                            p.grad = None
                        (((b[1].norm(dim=-1) - 1) ** 2).mean() + b[0].mean()).backward()
                        r['param_grad'] = {k: p.grad for k, p in ref.named_parameters() if p.grad is not None}
                        r['requires_grad'] = b[0].requires_grad
                    return r
                b = T.ref(f'{name}/{step}/{mode}', ref_run)
                names = ['sdf', 'grad', 'feature'] + (['laplace'] if fd else [])
                d = {n: mx(x, y) for n, x, y in zip(names, a, b['out'])}
                d['level'] = mx(our.forward_level(pts), b['level'])
                d['sdf_only'] = mx(our(pts.clone(), with_grad=False, with_feature=False), b['sdf_only'])
                if mode == 'train':   # eikonal-style loss through the normals: second-order path of the torch fallback
                    for p in our.parameters():
                        p.grad = None
                    (((a[1].norm(dim=-1) - 1) ** 2).mean() + a[0].mean()).backward()
                    go, gr = dict(our.named_parameters()), b['param_grad']
                    d['param_grad'] = max(mx(go[k].grad, gr[k]) / (amax(gr[k]) + 1e-30) for k in gr)
                    d['requires_grad_outputs'] = float(a[0].requires_grad != b['requires_grad'])
                else:
                    d['detached'] = float(any(t.requires_grad for t in a))
                out[f'{step}/{mode}'] = d
        return out

    na = configs.neuralangelo_dtu()['geometry']
    res['finite_difference_progressive'] = pair('finite_difference_progressive', na, (0, 2500, 20000))
    an = configs.neus_blender()['geometry']
    an['fused'] = False                              # the torch fallback of the analytic-normal path
    res['analytic_fallback'] = pair('analytic_fallback', an, (0,))
    fixed = dict(configs.neus_blender()['geometry'], grad_type='finite_difference', finite_difference_eps=0.01)
    res['finite_difference_fixed_eps'] = pair('finite_difference_fixed_eps', fixed, (0,))
    colmap = dict(configs.neuralangelo_dtu()['geometry'], grad_type='analytic', radius=0.6)   # neus-colmap.yaml: progressive grid + analytic normals
    colmap.pop('finite_difference_eps', None)
    res['analytic_progressive'] = pair('analytic_progressive', colmap, (0, 3500))
    if T.recording:
        T.save()
    print('RESULT ' + json.dumps(res))


if __name__ == '__main__':
    main()
