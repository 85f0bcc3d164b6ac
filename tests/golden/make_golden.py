"""Generates the golden vectors under tests/golden/.  The files marked (*) need a checkout of the reference
(monniert/differentiable-blocksworld), given with --reference DIR; without it they are left untouched:

  ref_functions.npz   (*) outputs of the REFERENCE'S OWN pure-torch functions on seeded inputs, obtained by extracting them
                      with `ast` from the checkout (layered_rgb_blend, parametric_sq/signed_pow, get_icosphere_uvs,
                      point_to_uv_sphericalmap, elev/azim/roll rotations).  These pin the oracle's restatements.
  ref_restatements.npz  (*) the same functions over every blend mode (sigma x clip_inside x opacities) on a second seeded
                      input, and the reference's own DifferentiableBlocksWorld.compute_losses (parsimony / TV / overlap)
                      on a crowded 4-block scene for coarse / fine x each TV norm: inputs and outputs.
  ref_configs.json    (*) the `model` section of every configs/<dataset>/<name>.yml of the reference, overlaid on the
                      directory's default.yml as the reference's load_yaml does.
  primitives/*.obj    (*) the reference's primitive meshes (cube, plane), verbatim.
  render_cube.npz     oracle render of BASELINE configs[0] (one cube primitive, 2 views 64x64, K=10): soft + hard pass and
                      their gradients to the texture and the vertices, fp32.
  render_small.npz    oracle render of a small seeded scene (2 views 40x48, 3 blocks): blocks pass, env pass, composite,
                      loss and parameter gradients, fp32.  These pin the oracle against drift and give the CUDA path a
                      committed target.  (PARITY UNPINNED upstream: the reference ships no vectors, SURVEY 8c.)

    python tests/golden/make_golden.py [--reference DIR]
"""
import argparse
import json
import os
import shutil
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from oracle import dbw_path as D, pt3d  # noqa: E402
import _refextract  # noqa: E402
from _refextract import extract, extract_method, have_reference  # noqa: E402


def small_case(dtype=torch.float32):
    tpl = D.SceneTemplate(n_blocks=3, txt_size=32)
    p = D.init_params(3, 32, seed=11, boxy=True, dtype=dtype)
    R, T, K = D.ring_cameras(2, dtype=dtype, jitter=0.3, seed=11)
    g = torch.Generator().manual_seed(11)
    imgs = torch.rand(2, 3, 40, 48, generator=g).to(dtype)
    return tpl, p, R, T, K, imgs


def render_small(dtype=torch.float32):
    tpl, p, R, T, K, imgs = small_case(dtype)
    p = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    blocks, alpha = tpl.build_blocks(p)
    fa = alpha.repeat_interleave(tpl.BNF)
    fg = D.render(blocks, R, T, K, (40, 48), sigma=1e-4, faces_per_pixel=10, z_clip=0.001, detach_bary=True, faces_alpha=fa)
    env = D.render(tpl.build_env(p), R, T, K, (40, 48), sigma=0, faces_per_pixel=1, z_clip=0.001, detach_bary=False)
    rec = fg[:, :3] * fg[:, 3:] + (1 - fg[:, 3:]) * env[:, :3]
    loss = D.mse_loss(imgs, rec)
    loss.backward()
    out = {'fg': fg, 'env': env, 'rec': rec, 'loss': loss.reshape(1)}
    out.update({f'grad_{k}': (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in p.items()})
    return {k: v.detach().numpy() for k, v in out.items()}


def cube_case(dtype=torch.float32):
    """BASELINE configs[0]: one cube primitive, 2 views 64x64, K=10 (coarse settings)."""
    g = torch.Generator().manual_seed(3)
    tex = torch.sigmoid(torch.randn(32, 64, 3, generator=g)).to(dtype)
    Rm = pt3d.rotation_6d_to_matrix(torch.tensor([[0.9, 0.3, -0.2, -0.1, 0.8, 0.4]]))[0].to(dtype)
    R, T, K = D.ring_cameras(2, dtype=dtype, jitter=0.3, seed=3)
    return tex, Rm, torch.tensor([0.1, -0.05, 0.0], dtype=dtype), R, T, K


def render_cube(dtype=torch.float32):
    tex, Rm, Tm, R, T, K = cube_case(dtype)
    tex = tex.clone().requires_grad_(True)
    scene = D.cube_scene(tex, scale=0.45, R=Rm, T=Tm)
    scene['verts'].requires_grad_(True)
    out = D.render(scene, R, T, K, (64, 64), sigma=1e-4, faces_per_pixel=10, z_clip=0.001, detach_bary=True)
    hard = D.render(scene, R, T, K, (64, 64), sigma=0, faces_per_pixel=1, z_clip=0.001, detach_bary=False)
    (out.square().sum() + hard[:, :3].sum()).backward()
    return {k: v.detach().numpy() for k, v in dict(soft=out, hard=hard, grad_tex=tex.grad, grad_verts=scene['verts'].grad).items()}


def _read_obj(path):
    """minimal OBJ reader of the GENERATOR (v / f records, fan triangulation), independent of the product's loader"""
    vs, fs = [], []
    for line in open(path):
        t = line.split()
        if t[:1] == ['v']:
            vs.append([float(x) for x in t[1:4]])
        elif t[:1] == ['f']:
            ix = [int(x.split('/')[0]) - 1 for x in t[1:]]
            fs += [[ix[0], ix[k], ix[k + 1]] for k in range(1, len(ix) - 1)]
    return np.asarray(vs, np.float32), np.asarray(fs, np.int64)


def ref_functions():
    assert have_reference()
    out = {}
    g = torch.Generator().manual_seed(5)
    nsb = extract('src/model/renderer.py', ['layered_rgb_blend'])
    N, H, W, K = 2, 6, 7, 5
    p2f = torch.randint(-1, 30, (N, H, W, K), generator=g)
    d = torch.randn(N, H, W, K, generator=g) * 1e-4
    col = torch.rand(N, H, W, K, 3, generator=g)
    fa = torch.rand(40, generator=g)
    out.update(blend_p2f=p2f, blend_dists=d, blend_colors=col, blend_faces_alpha=fa)
    for name, sigma, ci, a in [('hard', 0, True, None), ('exp', 1e-4, True, fa), ('sigmoid', 1e-4, False, fa)]:
        out[f'blend_out_{name}'] = nsb['layered_rgb_blend'](col, SimpleNamespace(pix_to_face=p2f, dists=d),
                                                            SimpleNamespace(sigma=sigma, background_color=(0.1, 0.2, 0.3)),
                                                            clip_inside=ci, faces_alpha=a)
    ns = extract('src/utils/pytorch.py', ['signed_pow', 'safe_pow', 'SQRT_EPS'])
    ns2 = extract('src/utils/superquadric.py', ['parametric_sq'], {'signed_pow': ns['signed_pow']})
    eta, om = torch.rand(3, 42, generator=g) * 3 - 1.5, torch.rand(3, 42, generator=g) * 6 - 3
    e1, e2 = torch.rand(3, 1, generator=g) * 1.8 + 0.1, torch.rand(3, 1, generator=g) * 1.8 + 0.1
    out.update(sq_eta=eta, sq_omega=om, sq_e1=e1, sq_e2=e2, sq_out=ns2['parametric_sq'](eta, om, e1, e2))

    class M:
        def __init__(s, v, f): s.v, s.f = v, f
        def get_mesh_verts_faces(s, i): return s.v, s.f
    nsm = extract('src/utils/mesh.py', ['point_to_uv_sphericalmap', 'get_icosphere_uvs'],
                  {'get_icosphere': lambda level: M(*pt3d.ico_sphere(level))})
    for lvl in (1, 2):
        f, uv = nsm['get_icosphere_uvs'](lvl, fix_continuity=True, fix_poles=True)
        out[f'ico{lvl}_faces_uvs'], out[f'ico{lvl}_verts_uvs'] = f, uv
    cf, cuv = extract('src/utils/mesh.py', ['get_cube_uvs'])['get_cube_uvs']()
    out['cube_faces_uvs'], out['cube_verts_uvs'] = cf, cuv
    out['cube_verts'], out['cube_faces'] = _read_obj(os.path.join(_refextract.REF, 'primitives', 'cube.obj'))
    out['plane_verts'], out['plane_faces'] = _read_obj(os.path.join(_refextract.REF, 'primitives', 'plane.obj'))
    nst = extract('src/model/tools.py', ['azim_to_rotation_matrix', 'elev_to_rotation_matrix', 'roll_to_rotation_matrix'])
    out['R_world_115_20_m30'] = (nst['elev_to_rotation_matrix'](115) @ nst['azim_to_rotation_matrix'](20) @ nst['roll_to_rotation_matrix'](-30))[None]
    return {k: (v.numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()}


BLEND_CASES = [(sigma, ci, a) for sigma in (0, 1e-4) for ci in (True, False) for a in (False, True)]
REG_CASES = [(coarse, tv) for coarse in (True, False) for tv in ('l2sq', 'l2', 'l1')]


def regulariser_case():
    """a crowded 4-block scene whose overlap term is active; the fourth block is killed (kill_blocks)"""
    tpl = D.SceneTemplate(n_blocks=4, txt_size=16)
    p = D.init_params(4, 16, seed=2, boxy=True)
    p['alpha_logit'] = torch.tensor([3.0, 2.5, 2.0, -6.0])
    p['T'] = p['T'] * 0.02
    torch.manual_seed(77)
    u01 = torch.rand(4, 1000, 3)                                     # the draws of the reference's dbw.py:393
    return tpl, p, u01


def ref_restatements():
    assert have_reference()
    out = {}
    nsb = extract('src/model/renderer.py', ['layered_rgb_blend'])
    g = torch.Generator().manual_seed(9)
    N, H, W, K = 2, 5, 7, 4
    p2f = torch.randint(-1, 30, (N, H, W, K), generator=g)
    d = torch.randn(N, H, W, K, generator=g) * 1e-4
    col = torch.rand(N, H, W, K, 3, generator=g)
    fa = torch.rand(40, generator=g)
    out.update(blend_p2f=p2f, blend_dists=d, blend_colors=col, blend_faces_alpha=fa)
    for i, (sigma, ci, a) in enumerate(BLEND_CASES):
        out[f'blend_out_{i}'] = nsb['layered_rgb_blend'](col, SimpleNamespace(pix_to_face=p2f, dists=d),
                                                         SimpleNamespace(sigma=sigma, background_color=(0.1, 0.2, 0.3)),
                                                         clip_inside=ci, faces_alpha=fa if a else None)
    ns = extract('src/utils/pytorch.py', ['signed_pow', 'safe_pow', 'SQRT_EPS'])
    ns2 = extract('src/utils/superquadric.py', ['parametric_sq'], {'signed_pow': ns['signed_pow']})
    eta, om = torch.rand(3, 42, generator=g) * 3 - 1.5, torch.rand(3, 42, generator=g) * 6 - 3
    e1, e2 = torch.rand(3, 1, generator=g) * 1.8 + 0.1, torch.rand(3, 1, generator=g) * 1.8 + 0.1
    out.update(sq_eta=eta, sq_omega=om, sq_e1=e1, sq_e2=e2, sq_out=ns2['parametric_sq'](eta, om, e1, e2))

    class M:
        def __init__(s, v, f): s.v, s.f = v, f
        def get_mesh_verts_faces(s, i): return s.v, s.f
    nsm = extract('src/utils/mesh.py', ['point_to_uv_sphericalmap', 'get_icosphere_uvs'],
                  {'get_icosphere': lambda level: M(*pt3d.ico_sphere(level))})
    for lvl in (1, 2):
        out[f'ico{lvl}_faces_uvs'], out[f'ico{lvl}_verts_uvs'] = nsm['get_icosphere_uvs'](lvl, fix_continuity=True, fix_poles=True)

    # the reference's DifferentiableBlocksWorld.compute_losses (src/model/dbw.py:361-408), run on a stand-in `self` that
    # carries the state its build_* methods leave behind
    ns = extract('src/utils/pytorch.py', ['safe_pow', 'SQRT_EPS'])
    nsq = extract('src/utils/superquadric.py', ['implicit_sq'], {'safe_pow': ns['safe_pow']})
    nsl = extract('src/model/loss.py', ['tv_norm_funcs'], {'safe_pow': ns['safe_pow']})
    fn = extract_method('src/model/dbw.py', 'DifferentiableBlocksWorld', 'compute_losses',
                        {'safe_pow': ns['safe_pow'], 'implicit_sq': nsq['implicit_sq'], 'OVERLAP_N_POINTS': 1000,
                         'OVERLAP_N_BLOCKS': 1.95, 'OVERLAP_TEMPERATURE': 0.005})
    tpl, p, u01 = regulariser_case()
    out.update({f'reg_p_{k}': v for k, v in p.items()}, reg_u01=u01)
    keep = torch.sigmoid(p['alpha_logit']) > 0.01
    alpha_full = torch.sigmoid(p['alpha_logit']) * keep
    S, Rm = p['S'].exp() + tpl.scale_min, pt3d.rotation_6d_to_matrix(p['R_6d'])
    eps = torch.sigmoid(p['sq_eps']) * 1.8 + 0.1
    for coarse, tv_type in REG_CASES:
        me = SimpleNamespace(loss_weights={'parsimony': 0.01, 'tv': 0.1, 'overlap': 1.0}, is_live=lambda name: coarse,
                             _alpha_full=alpha_full, _bkg_maps=torch.sigmoid(p['texture_bkg']),
                             _ground_maps=torch.sigmoid(p['texture_ground']), _blocks_maps=torch.sigmoid(p['textures']),
                             tv_norm=nsl['tv_norm_funcs'][tv_type], n_blocks=4, ratio_block_scene=tpl.ratio,
                             _blocks_SRT=(S, Rm, p['T']), _blocks_eps=(eps[:, :1], eps[:, 1:]))
        torch.manual_seed(77)
        ref = fn(me, torch.zeros(1, 3, 4, 4), torch.zeros(1, 3, 4, 4))
        for k in ('parsimony', 'tv', 'overlap'):
            out[f'reg_{int(coarse)}_{tv_type}_{k}'] = torch.as_tensor(ref[k]).reshape(1)
    return {k: (v.numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()}


def ref_configs():
    """{'<dataset>/<file>': model section} of every reference config, overlaid on the directory's default.yml"""
    import yaml
    from copy import deepcopy
    root = os.path.join(_refextract.REF, 'configs')

    def overlay(dst, src):
        for k, v in (src or {}).items():
            if isinstance(v, dict) and isinstance(dst.get(k), dict):
                overlay(dst[k], v)
            else:
                dst[k] = v
    out = {}
    for ds in sorted(os.listdir(root)):
        dpath = os.path.join(root, ds, 'default.yml')
        default = yaml.safe_load(open(dpath)) if os.path.exists(dpath) else {}
        for fn in sorted(os.listdir(os.path.join(root, ds))):
            cfg = deepcopy(default)
            overlay(cfg, yaml.safe_load(open(os.path.join(root, ds, fn))))
            out[f'{ds}/{fn}'] = cfg['model']
    return out


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--reference', help='checkout of the reference (monniert/differentiable-blocksworld)')
    _refextract.REF = ap.parse_args().reference
    np.savez_compressed(os.path.join(HERE, 'render_small.npz'), **render_small())
    print('wrote render_small.npz')
    np.savez_compressed(os.path.join(HERE, 'render_cube.npz'), **render_cube())
    print('wrote render_cube.npz')
    if have_reference():
        np.savez_compressed(os.path.join(HERE, 'ref_functions.npz'), **ref_functions())
        print('wrote ref_functions.npz')
        np.savez_compressed(os.path.join(HERE, 'ref_restatements.npz'), **ref_restatements())
        print('wrote ref_restatements.npz')
        with open(os.path.join(HERE, 'ref_configs.json'), 'w') as f:
            json.dump(ref_configs(), f, indent=1, sort_keys=True)
        print('wrote ref_configs.json')
        os.makedirs(os.path.join(HERE, 'primitives'), exist_ok=True)
        for name in ('cube.obj', 'plane.obj'):
            shutil.copyfile(os.path.join(_refextract.REF, 'primitives', name), os.path.join(HERE, 'primitives', name))
        print('wrote primitives/cube.obj, primitives/plane.obj')
    else:
        print('no reference checkout given: ref_functions.npz, ref_restatements.npz, ref_configs.json, primitives/ left untouched')
