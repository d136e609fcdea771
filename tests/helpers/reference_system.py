"""Run in a subprocess by tests/test_reference_dropin.py.  Executes the UNMODIFIED reference training-step code -- ``preprocess_data`` and
``training_step`` of systems/nerf.py and systems/neus.py -- on the CPU with a tiny in-memory dataset and a fake model, and compares with
the oracle restatements the GPU kernels are tested against: oracle/rays.py (pixel -> ray front end), oracle/losses.py (loss blocks,
dynamic ray count).  Only packages that are not installed and not on the path (lightning, omegaconf, imaging libraries) are stubbed.
The reference's values are stored in tests/golden/reference_system.npz (tests/helpers/golden_ref.py; ``--record DIR`` re-creates it).
Its training steps driving the drop-in models are checked against the same steps restated from those oracle pieces."""
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
    T = Tape('reference_system')
    import cpu_thirdparty as tp
    from nsr_b200.config import Config, to_primitive
    from oracle import rays as orays, losses as olosses
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
    mc, mp = _stub('matplotlib.colors', LinearSegmentedColormap=object), _stub('matplotlib.pyplot')
    _stub('matplotlib', colors=mc, pyplot=mp, cm=types.SimpleNamespace())
    torch.cuda.device = lambda idx: contextlib.nullcontext()
    if T.recording:
        sys.path.insert(0, T.reference)
        import systems as ref_systems          # the reference's systems package: nerf.py, neus.py, base.py, criterions.py, utils.py
        from systems.utils import parse_optimizer as ref_parse_optimizer, update_module_step as ref_update_module_step

    def mx(a, b):
        a, b = pick(a, b)
        return float((a.double() - b.double()).abs().max())

    # ---- a tiny dataset in memory (what datasets/blender.py puts on the device)
    rng = np.random.default_rng(0)
    n_img, H, W = 5, 24, 32
    directions = orays.get_ray_directions(W, H, 40.0, 40.0, W / 2, H / 2)
    c2w = np.zeros((n_img, 3, 4), np.float32)
    for i in range(n_img):
        q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
        c2w[i, :, :3], c2w[i, :, 3] = q, rng.standard_normal(3) * 3
    images = rng.random((n_img, H, W, 3)).astype(np.float32)
    masks = (rng.random((n_img, H, W)) > 0.4).astype(np.float32)
    dataset = types.SimpleNamespace(all_images=torch.from_numpy(images), all_c2w=torch.from_numpy(c2w), all_fg_masks=torch.from_numpy(masks),
                                    directions=torch.from_numpy(directions), w=W, h=H, apply_mask=True, has_mask=True)
    res = {}

    def make_system(cls, model_cfg, loss_cfg):
        s = object.__new__(cls)
        torch.nn.Module.__init__(s)
        s.config = Config(dict(model=model_cfg, system=dict(loss=loss_cfg)))
        s.rank = 'cpu'                     # the reference moves batches with .to(self.rank)
        s.dataset = dataset
        s.log = lambda *a, **k: None
        s.global_step, s.current_epoch = 700, 0
        s.prepare()
        return s

    class FakeModel(torch.nn.Module):
        def __init__(self, out):
            super().__init__()
            self.out, self.background_color = out, None

        def forward(self, rays):
            return self.out

        def regularizations(self, out):
            return {}

    # ---- NeRF system: preprocess_data (systems/nerf.py:33-91) and training_step (:93-125)
    n_rays = 257
    model_cfg = dict(name='nerf', train_num_rays=n_rays, num_samples_per_ray=64, max_train_num_rays=1024, dynamic_ray_sampling=True,
                     batch_image_sampling=True, background_color='random')
    g = torch.Generator().manual_seed(3)
    out = {'comp_rgb': torch.rand(n_rays, 3, generator=g, requires_grad=True), 'rays_valid': torch.rand(n_rays, 1, generator=g) > 0.3,
           'num_samples': torch.tensor([9000], dtype=torch.int32)}

    def ref_nerf():
        s = make_system(ref_systems.systems['nerf-system'], model_cfg, dict(lambda_rgb=1.0, lambda_distortion=0.0))
        s.model = FakeModel(out)
        torch.manual_seed(11)
        batch = {}
        s.preprocess_data(batch, 'train')
        bg_train = s.model.background_color
        loss = s.training_step(batch, 0)['loss']
        loss.backward()
        grad = out['comp_rgb'].grad.clone()
        out['comp_rgb'].grad = None
        vb = {'index': torch.tensor([2])}   # validation path: every pixel of one image (systems/nerf.py:57-64)
        s.preprocess_data(vb, 'validation')
        return {'batch': batch, 'bg': bg_train, 'loss': float(loss.detach()), 'grad': grad, 'train_num_rays': s.train_num_rays,
                'image_rays': vb['rays']}
    ref = T.ref('nerf', ref_nerf)
    torch.manual_seed(11)                  # the same draws, in the reference's order: index, x, y, then the random background colour
    index = torch.randint(0, n_img, size=(n_rays,))
    x = torch.randint(0, W, size=(n_rays,))
    y = torch.randint(0, H, size=(n_rays,))
    bg = torch.rand((3,))
    o_rays, o_rgb, o_fg = orays.training_batch(directions, c2w, images, masks, index.numpy(), x.numpy(), y.numpy(), bg=bg.numpy(), apply_mask=True)
    o_loss = olosses.nerf_loss(out, torch.from_numpy(o_rgb))
    o_loss.backward()
    batch = ref['batch']
    res['nerf'] = {'rays': mx(o_rays, batch['rays']), 'rgb': mx(o_rgb, batch['rgb']), 'fg_mask': mx(o_fg, batch['fg_mask']),
                   'bg_equal': bool(torch.equal(ref['bg'], bg)),
                   'loss': ref['loss'], 'loss_oracle': float(o_loss.detach()),
                   'grad': mx(out['comp_rgb'].grad, ref['grad']),
                   'train_num_rays': ref['train_num_rays'],
                   'train_num_rays_oracle': olosses.next_train_num_rays(n_rays, n_rays * 64, 9000, 1024)}
    res['nerf']['image_rays'] = mx(orays.image_batch(directions, c2w, 2), ref['image_rays'])

    # ---- NeuS system: training_step (systems/neus.py:91-153)
    k = 4000
    model_cfg = dict(name='neus', train_num_rays=n_rays, num_samples_per_ray=64, max_train_num_rays=1024, dynamic_ray_sampling=True,
                     batch_image_sampling=True, background_color='white', learned_background=False)
    lam = dict(lambda_rgb_mse=10.0, lambda_rgb_l1=0.7, lambda_mask=0.1, lambda_eikonal=0.1, lambda_curvature=0.0, lambda_sparsity=0.02,
               lambda_distortion=0.0, lambda_distortion_bg=0.0, lambda_opaque=0.05, sparsity_scale=3.0)
    leaf = lambda *shape: torch.rand(*shape, generator=g).requires_grad_(True)
    out = {'comp_rgb_full': leaf(n_rays, 3), 'rays_valid_full': torch.rand(n_rays, 1, generator=g) > 0.3, 'opacity': leaf(n_rays, 1),
           'sdf_grad_samples': (torch.randn(k, 3, generator=g) * 1.3).requires_grad_(True),
           'sdf_samples': (torch.randn(k, generator=g) * 0.2).requires_grad_(True), 'num_samples_full': torch.tensor([5000], dtype=torch.int32),
           'inv_s': torch.tensor(20.0)}
    batch = {'rays': torch.zeros(n_rays, 6), 'rgb': torch.rand(n_rays, 3, generator=g), 'fg_mask': (torch.rand(n_rays, generator=g) > 0.5).float()}
    names = ('comp_rgb_full', 'opacity', 'sdf_grad_samples', 'sdf_samples')

    def ref_neus():
        s = make_system(ref_systems.systems['neus-system'], model_cfg, lam)
        s.model = FakeModel(out)
        loss = s.training_step(batch, 0)['loss']
        loss.backward()
        grads = {n: out[n].grad.clone() for n in names}
        for n in names:
            out[n].grad = None
        return {'loss': float(loss.detach()), 'grads': grads, 'train_num_rays': s.train_num_rays}
    ref = T.ref('neus', ref_neus)
    neus_lambdas = dict(rgb_mse=10.0, rgb_l1=0.7, eikonal=0.1, mask=0.1, opaque=0.05, sparsity=0.02, sparsity_scale=3.0)
    o_loss, terms = olosses.neus_loss(out, batch['rgb'], batch['fg_mask'], neus_lambdas)
    o_loss.backward()
    res['neus'] = {'loss': ref['loss'], 'loss_oracle': float(o_loss.detach()),
                   'grad': {n: mx(out[n].grad, ref['grads'][n]) for n in names},
                   'train_num_rays': ref['train_num_rays'],
                   'train_num_rays_oracle': olosses.next_train_num_rays(n_rays, n_rays * 64, 5000, 1024)}
    # ---- the reference's systems driving the DROP-IN models (INTEGRATION.md level 2), a few real training steps on the CPU: the models'
    # CUDA modules swapped for the stand-ins, everything else -- preprocess_data, update_module_step, training_step, the optimizer built by
    # the reference's parse_optimizer -- is the reference's own code calling our model classes.  The same steps restated from the oracle
    # pieces above (restated_system) must reproduce what the reference's systems reported.
    from nsr_b200 import models as our_models, configs, tcnn as our_tcnn, nerfacc as our_nerfacc, mcubes as nmc, ops, synthetic
    from nsr_b200.models import nerf_model, neus_model
    from oracle import mcubes as omc
    for mod in (nerf_model, neus_model):
        for fn in ('ray_marching', 'render_weight_from_density', 'render_weight_from_alpha', 'accumulate_along_rays'):
            if hasattr(mod, fn):
                setattr(mod, fn, getattr(tp, fn))
    # the GPU marching cubes of export() replaced by the oracle's inside this process
    nmc.marching_cubes = lambda level, threshold=0.0, lo=(0., 0., 0.), hi=(1., 1., 1.), negate=True: tuple(
        torch.from_numpy(a) for a in omc.marching_cubes(level.detach().cpu().numpy(), threshold, lo=lo, hi=hi, negate=negate))
    nmc.check_cuda = lambda *a, **k: None

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
    our_nerfacc.OccupancyGrid.every_n_step = lambda self, step, occ_eval_fn, **k: setattr(self, '_binary', torch.ones_like(self._binary))

    def make_model(kind, mcfg):
        torch.manual_seed(5)
        model = our_models.make(kind, mcfg)
        swap_tcnn(model)
        model.train()
        return model

    def prepare_export(kind, model, mcfg):
        if kind == 'nerf':   # give the density field a surface to extract: the bench's density bump (a ball of high density)
            net = model.geometry.encoding_with_network
            with torch.no_grad():
                flat = net.params.detach().clone()
                synthetic.shape_density(flat, ops.GridSpec(mcfg['geometry']['xyz_encoding_config']), net.n_mlp)
                net.params.copy_(flat)
        iso = dict(method='mc', resolution=20, chunk=4096, threshold=0.0 if kind == 'neus' else 5.0)
        model.geometry.config['isosurface'] = Config(iso)
        return iso, Config(dict(chunk_size=4096, export_vertex_color=True))

    def reference_system(kind, sysname, mcfg, lam_cfg):
        s = make_system(ref_systems.systems[sysname], mcfg, lam_cfg)
        s.train_num_samples = 64 * 40                      # a sample budget this tiny scene can meet
        s.model = make_model(kind, mcfg)
        opt = ref_parse_optimizer(Config(dict(name='AdamW', args=dict(lr=0.01, betas=[0.9, 0.99], eps=1.e-15))), s.model)
        losses_, rays_, train_rays = [], [], []
        for step in range(4):
            s.global_step = step
            batch = {}
            torch.manual_seed(100)                         # the same pixels every step: the loss on them must go down
            s.preprocess_data(batch, 'train')
            train_rays.append(batch['rays'])
            ref_update_module_step(s.model, 0, step)       # BaseSystem.on_train_batch_start
            loss = s.training_step(batch, step)['loss']
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses_.append(float(loss.detach()))
            rays_.append(int(s.train_num_rays))
        # validation_step (systems/nerf.py:136-149 / systems/neus.py:171-190): whole-image eval through model.eval() + chunk_batch
        s.model.eval()
        dataset.img_wh = (W, H)
        grids = []
        s.save_image_grid = lambda name, imgs: grids.append((name, [list(i['img'].shape) for i in imgs]))
        vb = {'index': torch.tensor([1])}
        s.preprocess_data(vb, 'validation')
        with torch.no_grad():
            vout = s.validation_step(vb, 0)
        # export() (systems/nerf.py:213-218): model.export(config.export) -> save_mesh(name, **mesh)
        iso, s.config['export'] = prepare_export(kind, s.model, mcfg)
        s.config['model']['geometry']['isosurface'] = Config(iso)
        meshes = []
        s.save_mesh = lambda name, **mesh: meshes.append((name, {k: list(v.shape) for k, v in mesh.items()}))
        s.export()
        return {'losses': losses_, 'train_num_rays': rays_, 'model_class': type(s.model).__module__,
                'val_psnr': float(vout['psnr']), 'val_index': int(vout['index'][0]), 'val_grid': grids[0][1],
                'mesh_name': meshes[0][0], 'mesh': meshes[0][1], 'rays': train_rays}

    def restated_system(kind, mcfg, lam_cfg, train_rays):
        """the same steps from the oracle pieces pinned above: the reference's draws, batch, losses, ray budget and AdamW; the training rays
        are the reference's (the oracle's agree to 1 ulp)"""
        model = make_model(kind, mcfg)
        opt = torch.optim.AdamW(model.parameters(), lr=0.01, betas=[0.9, 0.99], eps=1.e-15)   # parse_optimizer without param groups
        n_train, losses_, rays_ = mcfg['train_num_rays'], [], []
        for step in range(4):
            torch.manual_seed(100)
            index, x, y = (torch.randint(0, hi, size=(n_train,)) for hi in (n_img, W, H))
            bg = torch.rand((3,))
            _, rgb, fg = orays.training_batch(directions, c2w, images, masks, index.numpy(), x.numpy(), y.numpy(), bg=bg.numpy(), apply_mask=True)
            rgb, fg = torch.from_numpy(rgb), torch.from_numpy(fg)
            model.background_color = bg
            model.update_step(0, step)
            out = model(train_rays[step])
            n_samples = int(out['num_samples' if kind == 'nerf' else 'num_samples_full'].sum())
            n_train = olosses.next_train_num_rays(n_train, 64 * 40, n_samples, mcfg['max_train_num_rays'])
            loss = olosses.nerf_loss(out, rgb, lam_cfg['lambda_rgb']) if kind == 'nerf' else olosses.neus_loss(out, rgb, fg, neus_lambdas)[0]
            for name, value in model.regularizations(out).items():
                loss = loss + value * lam_cfg[f'lambda_{name}']
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses_.append(float(loss.detach()))
            rays_.append(n_train)
        model.eval()
        fg = torch.from_numpy(masks[1]).view(-1, 1)
        rgb = torch.from_numpy(images[1]).view(-1, 3) * fg + torch.ones(3) * (1 - fg)    # validation: white background
        model.background_color = torch.ones(3)
        with torch.no_grad():
            out = model(torch.from_numpy(orays.image_batch(directions, c2w, 1)))
        key = 'comp_rgb' if kind == 'nerf' else 'comp_rgb_full'
        grid = [rgb.view(H, W, 3), out[key].view(H, W, 3), out['depth'].view(H, W)] + \
            ([out['opacity'].view(H, W)] if kind == 'nerf' else [out['comp_normal'].view(H, W, 3)])
        iso, export_cfg = prepare_export(kind, model, mcfg)
        mesh = model.export(export_cfg)
        return {'losses': losses_, 'train_num_rays': rays_, 'val_psnr': float(-10 * torch.log10(torch.mean((out[key] - rgb) ** 2))),
                'val_grid': [list(t.shape) for t in grid], 'mesh_name': f"it3-{iso['method']}{iso['resolution']}.obj",
                'mesh': {k: list(v.shape) for k, v in mesh.items()}}

    res['integration'] = {}
    for kind, sysname, cfg_fn, lam_cfg in (('nerf', 'nerf-system', configs.nerf_blender, dict(lambda_rgb=1.0, lambda_distortion=0.0)),
                                           ('neus', 'neus-system', configs.neus_blender, lam)):
        mcfg = cfg_fn()
        mcfg.update(fused=False, train_num_rays=64, max_train_num_rays=128, num_samples_per_ray=1024, dynamic_ray_sampling=True,
                    batch_image_sampling=True, background_color='random')
        mcfg['geometry']['fused'] = False
        e = T.ref(f'integration/{kind}', lambda: reference_system(kind, sysname, mcfg, lam_cfg), whole=True)
        e['restated'] = restated_system(kind, mcfg, lam_cfg, e.pop('rays'))
        res['integration'][kind] = e

    # ---- parse_optimizer (systems/utils.py:314-325) on the same model and config section: param groups of the reference vs ours
    from nsr_b200.optim import parse_optimizer
    m = our_models.make('neus', configs.neus_dtu())
    ocfg = dict(name='AdamW', args=dict(lr=0.01, betas=[0.9, 0.99], eps=1.e-15),
                params=dict(geometry=dict(lr=0.01), texture=dict(lr=0.01), geometry_bg=dict(lr=0.01), texture_bg=dict(lr=0.01), variance=dict(lr=0.001)))
    keys = ('lr', 'betas', 'eps', 'weight_decay')
    param_names = {id(p): n for n, p in m.named_parameters()}

    def reference_groups():
        ro = ref_parse_optimizer(Config(ocfg), m)
        return {'class': type(ro).__name__, 'groups': [dict({k: g_[k] for k in ('name',) + keys}, params=[param_names[id(p)] for p in g_['params']])
                                                       for g_ in ro.param_groups]}
    ro, oo = T.ref('optimizer', reference_groups), parse_optimizer(Config(ocfg), m)
    res['optimizer'] = {
        'ref_class': ro['class'], 'our_class': type(oo).__name__,
        'names_equal': [g_['name'] for g_ in ro['groups']] == [g_['name'] for g_ in oo.param_groups],
        'hyper_equal': all(tuple(a[k]) == tuple(b[k]) if isinstance(a[k], (list, tuple)) else a[k] == b[k]
                           for a, b in zip(ro['groups'], oo.param_groups) for k in keys),
        'same_tensors': all(a['params'] == [param_names[id(p)] for p in b['params']] for a, b in zip(ro['groups'], oo.param_groups)),
        'n_groups': len(oo.param_groups)}
    if T.recording:
        T.save()
    print('RESULT ' + json.dumps(res))


if __name__ == '__main__':
    main()
