"""Drop-in check at INTEGRATION.md level 1: the UNMODIFIED reference models (instant-nsr-pl's models/*.py) import ``tinycudann`` and
``nerfacc`` and get nsr_b200's modules; they construct with the reference's own configs, expose the parameter counts SURVEY.md 8a
states, share state_dict keys / shapes with the drop-in models (checkpoints load both ways) and refuse CPU tensors the way
nerfacc 0.3.3 / tiny-cuda-nn do.  What the reference computes is stored under tests/golden/ (tests/helpers/golden_ref.py: each helper
re-creates its file with ``--record <instant-nsr-pl checkout>``), so these tests need nothing outside the repository."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_models_build_on_our_modules():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'helpers', 'reference_dropin.py')], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')][-1]
    res = json.loads(line[len('RESULT '):])
    assert res['registry'] == ['nerf', 'neus', 'volume-color', 'volume-density', 'volume-radiance', 'volume-sdf']
    nerf, neus, dtu = res['nerf'], res['neus'], res['neus-dtu']
    assert nerf['module'] == 'models.nerf' and neus['module'] == 'models.neus'            # the reference's classes, not ours
    # SURVEY 8a: table 12,599,920 + density MLP 3,072 + colour MLP 7,168; NeuS table 13,969,152 + SDF MLP (weight-norm: + 64 + 13 g) ...
    assert nerf['n_params'] == nerf['n_params_ours'] == 12599920 + 3072 + 7168
    assert neus['n_params'] == neus['n_params_ours'] == 13969152 + (35 * 64 + 64 + 64) + (64 * 13 + 13 + 13) + 7168 + 1
    for e in (nerf, neus, dtu):
        assert e['keys_equal'] and e['shapes_equal'] and not e['only_ref'] and not e['only_ours'], e
        assert e['cpu_forward'] == 'NotImplementedError'
        assert e['grid_is_ours'] == 'nsr_b200.nerfacc'
    assert nerf['tcnn_modules'] == ['Encoding', 'Network', 'NetworkWithInputEncoding']
    assert neus['tcnn_modules'] == ['Encoding', 'Network']
    assert dtu['n_params'] == dtu['n_params_ours'] and dtu['tcnn_modules'] == ['Encoding']  # neus-dtu: VanillaMLPs everywhere


def test_oracle_orchestration_is_pinned_to_the_reference_forward():
    """oracle/models.py (nerf_render, neus_render, neus_bg_render, neus_dtu_render) restates models/nerf.py:61-127 and models/neus.py:141-287.  Here the reference's
    OWN forward_ runs on the CPU -- tinycudann / nerfacc replaced by per-op stand-ins built from the oracle's primitives
    (tests/helpers/cpu_thirdparty.py), fp32 throughout -- and every output and parameter gradient (incl. the double backward of the
    eikonal term through the reference's VolumeSDF) must equal the oracle's: the glue is pinned, the third-party arithmetic stays ours
    on both sides."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'helpers', 'reference_forward.py')], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')][-1][len('RESULT '):])
    nerf, neus = res['nerf'], res['neus']
    assert nerf['keys'] == ['comp_rgb', 'depth', 'intervals', 'num_samples', 'opacity', 'points', 'ray_indices', 'rays_valid', 'weights']
    assert nerf['num_samples'] == nerf['num_samples_oracle'] and 0.3 * nerf['num_marched'] < nerf['num_samples'] < 0.9 * nerf['num_marched']
    assert nerf['rays_valid_equal'] and max(nerf['diff'].values()) < 1e-6 and max(nerf['grad_diff']) < 1e-5
    colmap = res['nerf_colmap']                      # unbounded NeRF (nerf-colmap.yaml): sphere contraction + cone marching + planes
    assert colmap['num_samples'] == colmap['num_samples_oracle'] > 1000 and colmap['num_marched'] > 10 * colmap['num_samples']
    assert max(colmap['diff'].values()) < 1e-6 and max(colmap['grad_diff']) < 1e-5
    assert colmap['constants'] == [0.01, pytest.approx(10 ** (4 / 2048) - 1, rel=1e-12), 0.2, 1e4]
    assert set(neus['keys']) >= {'comp_rgb', 'comp_normal', 'opacity', 'depth', 'rays_valid', 'num_samples', 'sdf_samples', 'sdf_grad_samples',
                                 'weights', 'points', 'intervals', 'ray_indices', 'comp_rgb_bg', 'num_samples_bg', 'rays_valid_bg',
                                 'comp_rgb_full', 'num_samples_full', 'rays_valid_full'}
    assert neus['num_samples'] == neus['num_samples_oracle'] > 5000 and neus['cos_anneal_ratio'] == 0.25
    assert max(neus['diff'].values()) < 5e-6 and neus['inv_s_diff'] == 0.0 and max(neus['grad_diff'].values()) < 1e-5
    # config C4 (neus-dtu.yaml): learned background = forward_bg_ (models/neus.py:141-203) + the *_bg / *_full composition (:268-281)
    dtu = res['neus_dtu']
    assert not dtu['oracle_keys_missing'] and dtu['num_samples'] > 5000
    assert dtu['num_samples_bg'] == dtu['num_samples_bg_oracle'] > 300 and dtu['num_samples_full_equal'] and dtu['rays_valid_full_equal']
    assert max(dtu['diff'].values()) < 5e-6
    assert dtu['n_grads'] == 25 and max(dtu['grad_diff'].values()) < 2e-4     # every trainable tensor of all five submodules
    # the occupancy functions update_step hands to OccupancyGrid.every_n_step (models/nerf.py:45-55, models/neus.py:90-111) and their thresholds
    assert nerf['occ_fn'] < 1e-7 and nerf['occ_thre'] == 0.01
    assert neus['occ_fn'] < 1e-6 and neus['occ_thre'] == 0.001                # grid_prune_occ_thre of neus-blender.yaml
    assert dtu['occ_fn_bg'] < 1e-6 and dtu['occ_thre'] == [0.001, 0.01]       # the background grid keeps the default threshold


def test_oracle_front_end_and_losses_are_pinned_to_the_reference_training_step():
    """The reference's OWN systems/nerf.py / systems/neus.py ``preprocess_data`` and ``training_step`` run on the CPU (tiny in-memory
    dataset, fake model; tests/helpers/reference_system.py): the batch they assemble equals oracle.rays.training_batch / image_batch (the
    checker of nsr_gather_rays), their losses and gradients equal oracle.losses (the restatement the fused loss kernels are tested
    against), and their dynamic ray count equals the rule RayBudget applies."""
    from nsr_b200.rays import RayBudget
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'helpers', 'reference_system.py')], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')][-1][len('RESULT '):])
    nerf, neus = res['nerf'], res['neus']
    assert nerf['rays'] < 3e-7 and nerf['image_rays'] < 3e-7 and nerf['rgb'] == 0.0 and nerf['fg_mask'] == 0.0 and nerf['bg_equal']
    assert abs(nerf['loss'] - nerf['loss_oracle']) < 1e-7 and nerf['grad'] < 1e-8
    assert nerf['train_num_rays'] == nerf['train_num_rays_oracle'] == RayBudget.rule(257, 257 * 64, 9000, 1024)
    assert abs(neus['loss'] - neus['loss_oracle']) < 1e-6 and max(neus['grad'].values()) < 1e-7
    assert neus['train_num_rays'] == neus['train_num_rays_oracle'] == RayBudget.rule(257, 257 * 64, 5000, 1024)
    # level 2: the reference's systems (preprocess_data, update_module_step, training_step, parse_optimizer) drive OUR model classes for a
    # few real optimizer steps on the CPU (CUDA modules swapped for the stand-ins): it trains, and the ray budget reacts
    for kind in ('nerf', 'neus'):
        e = res['integration'][kind]
        assert e['model_class'] == f'nsr_b200.models.{kind}_model' and len(e['losses']) == 4
        assert e['losses'][-1] < e['losses'][0] and all(v == v for v in e['losses'])
        assert e['train_num_rays'][-1] != 64 and all(1 <= v <= 128 for v in e['train_num_rays'])
        # ... and their validation_step renders a whole image through model.eval() / chunk_batch and lays the outputs out as H x W images
        assert 0 < e['val_psnr'] < 60 and e['val_index'] == 1 and e['val_grid'][:2] == [[24, 32, 3], [24, 32, 3]]
        # ... and their export() receives the mesh dictionary save_mesh expects (marching cubes: the oracle's, in that process)
        m = e['mesh']
        assert e['mesh_name'] == 'it3-mc20.obj' and set(m) == {'v_pos', 't_pos_idx', 'v_rgb'}
        assert m['v_pos'][0] > 500 and m['v_pos'] == m['v_rgb'] and m['t_pos_idx'][1] == 3
        # the same steps restated from the oracle pieces pinned above, on the same drop-in model, reproduce what the systems reported
        r = e['restated']
        assert r['train_num_rays'] == e['train_num_rays'] and r['val_grid'] == e['val_grid'] and r['mesh_name'] == e['mesh_name'], (kind, r)
        assert max(abs(a - b) / abs(b) for a, b in zip(r['losses'], e['losses'])) < 1e-5 and abs(r['val_psnr'] - e['val_psnr']) < 1e-4, (kind, r)
        assert r['mesh'] == e['mesh'], (kind, r['mesh'])
    # optim.parse_optimizer builds the reference's param groups (same tensors, names, hyper-parameters) around FusedAdamW
    opt = res['optimizer']
    assert opt['ref_class'] == 'AdamW' and opt['our_class'] == 'FusedAdamW' and opt['n_groups'] == 5
    assert opt['names_equal'] and opt['hyper_equal'] and opt['same_tensors']


def test_product_torch_side_equals_the_reference_functions():
    """every pure-torch piece of the drop-in models compared DIRECTLY with the reference's own (tests/helpers/reference_torch_parts.py):
    activations (value + gradient), scale_anything, contraction, chunk_batch, VanillaFrequency mask schedule, VanillaMLP / tcnn sphere
    initialisation (same seed => the same parameters, draw for draw), VarianceNetwork modulation, NeuSModel.get_alpha with cos annealing,
    the render constants (step sizes, cone angle, planes, boxes).  The bar is bit equality."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'helpers', 'reference_torch_parts.py')], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')][-1][len('RESULT '):])

    def worst(v):
        if isinstance(v, dict):
            return max(worst(x) for x in v.values())
        return float(v) if not isinstance(v, bool) else (0.0 if v else 1.0)

    assert len(res['activations']) == 15 and len(res['chunk_batch']) == 8 and len(res['vanilla_mlp']) == 4
    for name, section in res.items():
        assert worst(section) == 0.0, (name, section)


def test_product_volume_sdf_torch_paths_equal_the_reference():
    """VolumeSDF paths of the product that are torch code rather than kernels -- finite-difference normals + laplacian under the
    ProgressiveBandHashGrid schedule (configs/neuralangelo-dtu-wmask.yaml), fixed-eps finite differences, the autograd fallback of the
    analytic normal (plain grid, and the progressive grid of configs/neus-colmap.yaml) -- run on the CPU with the hash grid swapped for the oracle-backed stand-in, against the reference's VolumeSDF with the
    same weights (tests/helpers/reference_sdf_paths.py): values, level function, train / eval detaching, parameter gradients through an
    eikonal-style loss."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'helpers', 'reference_sdf_paths.py')], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')][-1][len('RESULT '):])
    assert set(res) == {'finite_difference_progressive', 'analytic_fallback', 'finite_difference_fixed_eps', 'analytic_progressive'}
    assert len(res['finite_difference_progressive']) == 6
    for section, cases in res.items():
        for case, d in cases.items():
            for name, v in d.items():
                tol = 1e-5 if name == 'param_grad' else (2e-6 if name == 'grad' else 0.0)
                assert v <= tol, (section, case, name, v)


def test_product_models_composed_path_equals_the_reference_models_on_cpu():
    """The drop-in 'nerf' / 'neus' models run their per-op (composed) code path on the CPU -- tcnn modules swapped for the oracle-backed
    stand-ins, nerfacc-shaped functions rebound to them (tests/helpers/reference_product_composed.py) -- against the unmodified reference
    models with the same weights, for C2 (nerf-blender), nerf-colmap (unbounded: sphere contraction + cone marching), C3 (neus-blender) and
    C4 (neus-dtu with the learned background): same output
    keys and dtypes, values and every parameter gradient to fp32 rounding, same eval-mode behaviour (chunking, detaching, inv_s)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'helpers', 'reference_product_composed.py')], capture_output=True,
                       text=True, timeout=1500)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('RESULT ')][-1][len('RESULT '):])
    assert sorted(res) == ['nerf:nerf_blender', 'nerf:nerf_colmap', 'neus:neus_blender', 'neus:neus_dtu']
    for name, e in res.items():
        assert e['keys_equal'] and e['dtype_equal'] and e['grad_keys_equal'] and e['eval_keys_equal'], (name, e['only_ours'], e['only_ref'])
        assert e['num_samples'] > (1000 if 'colmap' in name else 5000), name
        assert max(e['diff'].values()) < 5e-6 and e['grad_diff'] < 1e-5 and e['eval_diff'] < 5e-6, (name, e)
