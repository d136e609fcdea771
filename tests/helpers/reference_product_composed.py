"""Run in a subprocess by tests/test_reference_dropin.py.  The PRODUCT's drop-in models (nsr_b200.models 'nerf' / 'neus') executed on the
CPU through their composed (per-op) code path -- the CUDA-backed tcnn modules swapped for the oracle-backed stand-ins and the nerfacc-shaped
functions rebound to the stand-ins (tests/helpers/cpu_thirdparty.py) -- against the UNMODIFIED reference models built on the same stand-ins
with the same weights: the Python orchestration of the drop-in models (everything that is not a kernel) for C2, C3 and C4.  The original
models' weights, outputs and gradients are stored in tests/golden/reference_product_composed.npz (tests/helpers/golden_ref.py;
``--record DIR`` re-creates it)."""
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
from golden_ref import Tape, pick, amax, is_array  # noqa: E402


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def main():
    T = Tape('reference_product_composed')
    import cpu_thirdparty as tp
    from nsr_b200.config import Config, to_primitive
    from nsr_b200 import configs, synthetic, models as ours, tcnn as our_tcnn
    from nsr_b200.models import nerf_model, neus_model
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

    # the product's nerfacc-shaped entry points -> CPU stand-ins (only inside this process)
    for mod in (nerf_model, neus_model):
        for fn in ('ray_marching', 'render_weight_from_density', 'render_weight_from_alpha', 'accumulate_along_rays', 'ray_aabb_intersect'):
            if hasattr(mod, fn):
                setattr(mod, fn, getattr(tp, fn) if hasattr(tp, fn) else inter.ray_aabb_intersect)

    def swap_tcnn(module):
        """replace every CUDA-backed tcnn module inside ``module`` by the stand-in of the same kind (parameters are loaded afterwards)"""
        for name, child in list(module.named_children()):
            if isinstance(child, our_tcnn.NetworkWithInputEncoding):
                setattr(module, name, tp.NetworkWithInputEncoding(child.n_input_dims, child.n_output_dims, child.encoding_config, child.network_config))
            elif isinstance(child, our_tcnn.Encoding):
                setattr(module, name, tp.Encoding(child.n_input_dims, child.encoding_config))
            elif isinstance(child, our_tcnn.Network):
                setattr(module, name, tp.Network(child.n_input_dims, child.n_output_dims, child.network_config))
            else:
                swap_tcnn(child)

    def mx(a, b):
        a, b = pick(a, b)
        a, b = a.double(), b.double()
        assert a.shape == b.shape, (a.shape, b.shape)
        return float((a - b).abs().max()) if a.numel() else 0.0

    binary = synthetic.occupancy()
    rays = synthetic.sample_rays(160, seed=31)
    bg = torch.tensor([0.2, 0.5, 0.8])
    res = {}

    def run(kind, cfg_fn, prepare, loss_fn, ray_scale=1.0):
        cfg = cfg_fn()
        cfg['randomized'] = False
        cfg['fused'] = False
        if 'geometry' in cfg:
            cfg['geometry']['fused'] = False
        name = f'{kind}:{cfg_fn.__name__}'
        torch.manual_seed(0)
        our = ours.make(kind, cfg)
        swap_tcnn(our)
        prepare(our)
        if T.recording:   # the unmodified reference model with our weights
            ref = ref_models.make(kind, Config(cfg_fn() | {'randomized': False}))
            missing, unexpected = ref.load_state_dict(our.state_dict(), strict=False)   # (the stand-in grid has no grid_coords / grid_indices)
            assert not missing and all('occupancy_grid' in k for k in unexpected), (missing, unexpected)
        T.check_state(our, f'{name}/state')
        r = rays.copy()
        r[:, :3] *= ray_scale

        def run_model(m):
            m.train()
            m.update_step(0, 5001)            # not a multiple of 16: the product's occupancy refresh needs CUDA
            m.background_color = bg
            for p in m.parameters():
                p.grad = None
            out = m.forward_(torch.from_numpy(r))
            loss_fn(out).backward()
            grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
            # eval mode: chunked, detached, parked on the CPU, plus inv_s for NeuS
            m.eval()
            with torch.no_grad():
                ev = m(torch.from_numpy(r))
            return {k: v.detach() if torch.is_tensor(v) else v for k, v in out.items()}, grads, ev
        a, ga, ea = run_model(our)
        b, gb, eb = T.ref(f'{name}/run', lambda: run_model(ref))
        entry = {'keys_equal': sorted(a) == sorted(b), 'only_ours': sorted(set(a) - set(b)), 'only_ref': sorted(set(b) - set(a)),
                 'num_samples': int(b['num_samples']), 'diff': {k: mx(a[k].float(), b[k]) for k in b if is_array(b[k])},
                 'dtype_equal': all(a[k].dtype == b[k].dtype for k in b if is_array(b[k]) and k in a),
                 'grad_keys_equal': sorted(ga) == sorted(gb),
                 'grad_diff': max(mx(ga[k], gb[k]) / (amax(gb[k]) + 1e-30) for k in gb if k in ga)}
        entry['eval_keys_equal'] = sorted(ea) == sorted(eb)
        entry['eval_diff'] = max(mx(ea[k].float(), eb[k]) for k in eb if is_array(eb[k]) and k in ea)
        res[name] = entry

    def prep_nerf(m):
        from nsr_b200 import ops
        net = m.geometry.encoding_with_network
        with torch.no_grad():
            flat = net.params.detach().clone()
            synthetic.shape_density(flat, ops.GridSpec(configs.nerf_blender()['geometry']['xyz_encoding_config']), net.n_mlp)
            net.params.copy_(flat)
            m.occupancy_grid._binary.copy_(torch.from_numpy(binary))

    def shell(radius, lo, hi):
        g = (np.arange(128) + 0.5) / 128 * 2 * radius - radius
        X, Y, Z = np.meshgrid(g, g, g, indexing='ij')
        d = np.sqrt(X ** 2 + Y ** 2 + Z ** 2)
        return (d > lo * radius) & (d < hi * radius)

    def prep_neus(m):
        with torch.no_grad():
            v = m.geometry.network.layers[0].weight_v
            v[:, 3:] = torch.randn(v.shape[0], v.shape[1] - 3) * 0.05
            m.occupancy_grid._binary.copy_(torch.from_numpy(shell(1.5, 0.37, 0.63)))

    def prep_dtu(m):
        with torch.no_grad():
            v = m.geometry.network.layers[0].weight_v
            v[:, 3:] = torch.randn(v.shape[0], v.shape[1] - 3) * 0.05
            m.geometry_bg.encoding_with_network.network.layers[-1].bias[0] = 2.5
            m.occupancy_grid._binary.copy_(torch.from_numpy(shell(1.0, 0.35, 0.65)))
            m.occupancy_grid_bg._binary.copy_(torch.from_numpy(np.random.default_rng(0).random((256, 256, 256)) < 0.3))

    def neus_loss(out):
        eik = ((torch.linalg.norm(out['sdf_grad_samples'], ord=2, dim=-1) - 1.) ** 2).mean()
        return out['comp_rgb_full'].square().mean() + 0.1 * eik + 0.05 * out['opacity'].mean()

    run('nerf', configs.nerf_blender, prep_nerf, lambda out: out['comp_rgb'].square().mean() + 0.1 * out['opacity'].mean() + 0.05 * out['depth'].mean())
    def prep_colmap(m):
        from nsr_b200 import ops
        net = m.geometry.encoding_with_network
        with torch.no_grad():
            flat = net.params.detach().clone()
            synthetic.shape_density(flat, ops.GridSpec(configs.nerf_colmap()['geometry']['xyz_encoding_config']), net.n_mlp, radius=1.0)
            net.params.copy_(flat)
            m.occupancy_grid._binary.copy_(torch.from_numpy(np.random.default_rng(1).random((256, 256, 256)) < 0.3))

    run('nerf', configs.nerf_colmap, prep_colmap, lambda out: out['comp_rgb'].square().mean() + 0.1 * out['opacity'].mean() + 0.05 * out['depth'].mean(),
        ray_scale=1.0 / 1.5 * 0.4)
    run('neus', configs.neus_blender, prep_neus, neus_loss)
    run('neus', configs.neus_dtu, prep_dtu, neus_loss, ray_scale=1.0 / 1.5 * 0.6)
    if T.recording:
        T.save()
    print('RESULT ' + json.dumps(res))


if __name__ == '__main__':
    main()
