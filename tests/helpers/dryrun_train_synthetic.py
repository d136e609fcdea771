"""Run in a subprocess by tests/test_abi_and_host.py: tools/train_synthetic.py end to end on the CPU -- a logic check of the tool (dataset
builder, batch assembly, loss, optimizer / scheduler, ray budget, evaluation) without a GPU.  Everything CUDA-backed is swapped inside THIS
process only: tcnn modules and nerfacc-shaped functions by the oracle-backed stand-ins (tests/helpers/cpu_thirdparty.py), the ray kernels
by oracle/rays.py, the fused losses by oracle/losses.py, FusedAdamW by torch.optim.AdamW, the occupancy refresh by a full grid."""
import sys, os, types, importlib.util, json, time
import numpy as np, torch
ROOT=os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))); sys.path.insert(0, ROOT); sys.path.insert(0, ROOT+'/tests/helpers')
import cpu_thirdparty as tp
from nsr_b200 import models as ours, tcnn as our_tcnn, rays as nrays, optim as noptim, configs
from nsr_b200.models import nerf_model, neus_model
from oracle import rays as orays
for mod in (nerf_model, neus_model):
    for fn in ('ray_marching','render_weight_from_density','render_weight_from_alpha','accumulate_along_rays'):
        if hasattr(mod, fn): setattr(mod, fn, getattr(tp, fn))
def swap_tcnn(module):
    for name, child in list(module.named_children()):
        if isinstance(child, our_tcnn.NetworkWithInputEncoding): setattr(module, name, tp.NetworkWithInputEncoding(child.n_input_dims, child.n_output_dims, child.encoding_config, child.network_config))
        elif isinstance(child, our_tcnn.Encoding): setattr(module, name, tp.Encoding(child.n_input_dims, child.encoding_config))
        elif isinstance(child, our_tcnn.Network): setattr(module, name, tp.Network(child.n_input_dims, child.n_output_dims, child.network_config))
        else: swap_tcnn(child)
_make = ours.make
def make_cpu(name, cfg):
    if name in ('nerf','neus'):
        cfg = dict(cfg); cfg['fused']=False; cfg['randomized']=False
        cfg['geometry'] = dict(cfg['geometry']); cfg['geometry']['fused']=False
    m = _make(name, cfg)
    if name in ('nerf','neus'): swap_tcnn(m)
    return m
ours.make = make_cpu
def tb(directions, c2w, images, masks, idx, x, y, background_color=None, apply_mask=False):
    r, c, f = orays.training_batch(directions.numpy(), c2w.numpy(), images.numpy(), masks.numpy(), idx.numpy(), x.numpy(), y.numpy())
    return {'rays': torch.from_numpy(r), 'rgb': torch.from_numpy(c), 'fg_mask': torch.from_numpy(f)}
nrays.training_batch = tb
nrays.image_batch = lambda d, c2w, i, *a, **k: {'rays': torch.from_numpy(orays.image_batch(d.numpy(), c2w.numpy(), int(i)))}
class CpuAdamW(torch.optim.AdamW):
    @classmethod
    def for_model(cls, model, params=None, **kw): return cls(params if params is not None else [p for p in model.parameters() if p.requires_grad], **kw)
noptim.FusedAdamW = CpuAdamW
torch.cuda.synchronize = lambda *a, **k: None
from nsr_b200 import losses as nl
from oracle import losses as ol
nl.neus_losses = lambda out, rgb, mask, **lam: ol.neus_loss(out, rgb, mask, dict(rgb_mse=lam.get('lambda_rgb_mse',0), eikonal=lam.get('lambda_eikonal',0), mask=lam.get('lambda_mask',0)))
# occupancy refresh needs CUDA: no-op it and use a fixed grid
from nsr_b200 import nerfacc as nacc
def every_n_step(self, step, occ_eval_fn, **k):
    if step == 0:
        from nsr_b200 import synthetic
        self._binary = torch.ones_like(self._binary)
nacc.OccupancyGrid.every_n_step = every_n_step
spec = importlib.util.spec_from_file_location('train_synthetic', ROOT+'/tools/train_synthetic.py'); ts = importlib.util.module_from_spec(spec); spec.loader.exec_module(ts)
import argparse
for model in ('nerf', 'neus'):
    args = argparse.Namespace(model=model, steps=3, images=4, size=12, rays=48, max_rays=64, device='cpu', export=False, dataset_only=False)
    ts.train(args)
