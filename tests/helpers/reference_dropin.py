"""Run in a subprocess by tests/test_reference_dropin.py (it rebinds sys.modules entries and torch.cuda.device, which must not leak into
the pytest process).  Builds the UNMODIFIED reference models (/root/reference/models/*.py) on top of nsr_b200's tinycudann / nerfacc
replacements (INTEGRATION.md level 1) and prints a JSON summary.  Only third-party packages that are not installed here and have
nothing to do with the path (lightning, omegaconf, imageio, ...) are stubbed.  What the original models report is stored in
tests/golden/reference_dropin.npz (tests/helpers/golden_ref.py; ``--record DIR`` re-creates it); the drop-in side runs every time."""
import contextlib
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden_ref import Tape  # noqa: E402


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def main():
    T = Tape('reference_dropin')
    from nsr_b200.config import Config, to_primitive
    import nsr_b200.nerfacc as nsr_nerfacc
    nsr_nerfacc.install_as_reference_modules()       # what INTEGRATION.md asks a maintainer to add to launch.py
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
    sysm = _stub('systems')   # the Lightning systems package: only update_module_step is used by models/
    sysm.utils = _stub('systems.utils', update_module_step=lambda m, e, s: m.update_step(e, s) if hasattr(m, 'update_step') else None)
    if not torch.cuda.is_available():   # the reference constructs tcnn modules under torch.cuda.device(rank)
        torch.cuda.device = lambda idx: contextlib.nullcontext()
    if T.recording:
        sys.path.insert(0, T.reference)
        import models as ref_models   # the reference's registry; imports its nerf, neus, geometry, texture modules
    from nsr_b200 import configs, models as our_models, tcnn
    nerfacc = sys.modules['nerfacc']  # what `import nerfacc` gives the reference's models

    def cpu_forward(model):
        model.train()
        model.background_color = torch.ones(3)
        try:
            model(torch.zeros(4, 6))
            return 'ran'
        except NotImplementedError:       # nerfacc 0.3.3 / tinycudann behaviour: CUDA only
            return 'NotImplementedError'

    def reference_model(kind, cfg_fn):
        ref = ref_models.make(kind, Config(cfg_fn()))
        return {'module': type(ref).__module__, 'n_params': sum(p.numel() for p in ref.parameters()),
                'shapes': {k: list(v.shape) for k, v in ref.state_dict().items()},
                'tcnn_modules': sorted({type(m).__name__ for m in ref.modules() if type(m).__module__ == tcnn.__name__}),
                'grid_module': type(ref.occupancy_grid).__name__, 'cpu_forward': cpu_forward(ref)}

    out = {'registry': T.ref('registry', lambda: sorted(ref_models.models))}
    for name, cfg_fn in (('nerf', configs.nerf_blender), ('neus', configs.neus_blender), ('neus-dtu', configs.neus_dtu)):
        kind = name.split('-')[0]
        ref = T.ref(name, lambda: reference_model(kind, cfg_fn))
        ours = our_models.make(kind, cfg_fn())
        rs, os_ = ref['shapes'], ours.state_dict()
        entry = {
            'module': ref['module'],
            'n_params': ref['n_params'],
            'n_params_ours': sum(p.numel() for p in ours.parameters()),
            'keys_equal': sorted(rs) == sorted(os_),
            'shapes_equal': all(tuple(rs[k]) == tuple(os_[k].shape) for k in rs if k in os_),
            'only_ref': sorted(set(rs) - set(os_)), 'only_ours': sorted(set(os_) - set(rs)),
            # the tcnn classes the reference instantiates, as our tcnn module provides them
            'tcnn_modules': [n for n in ref['tcnn_modules'] if getattr(tcnn, n, None) is not None],
            'grid_is_ours': getattr(nerfacc, ref['grid_module']).__module__,
        }
        # a checkpoint of the reference's layout loads into the drop-in model (the other direction: same keys and shapes, strict)
        g = torch.Generator().manual_seed(0)
        ours.load_state_dict({k: torch.rand(rs[k], generator=g).to(v.dtype) if v.is_floating_point() else v for k, v in os_.items()})
        entry['cpu_forward'] = cpu_forward(ours) if ref['cpu_forward'] == 'NotImplementedError' else 'reference ran on the CPU'
        out[name] = entry
    if T.recording:
        T.save()
    print('RESULT ' + json.dumps(out))


if __name__ == '__main__':
    main()
