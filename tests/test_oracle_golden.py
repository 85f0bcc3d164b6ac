"""CPU: the oracle against the committed golden vectors (tests/golden/, generator make_golden.py), among them the outputs
of the reference's own functions (extracted with `ast` from a reference checkout when the vectors were generated)."""
import os

import numpy as np
import pytest
import torch

from oracle import dbw_path as D, pt3d

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _npz(name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLD, name)).items()}


def test_blend_matches_reference_golden():
    g = _npz('ref_functions.npz')
    for name, sigma, ci, a in [('hard', 0, True, None), ('exp', 1e-4, True, g['blend_faces_alpha']),
                               ('sigmoid', 1e-4, False, g['blend_faces_alpha'])]:
        out = D.layered_rgb_blend(g['blend_colors'], g['blend_p2f'], g['blend_dists'], sigma, (0.1, 0.2, 0.3), ci, a)
        assert torch.allclose(out, g[f'blend_out_{name}'], atol=1e-7, rtol=0), name


def test_superquadric_and_uv_builders_match_reference_golden():
    g = _npz('ref_functions.npz')
    out = D.parametric_sq(g['sq_eta'], g['sq_omega'], g['sq_e1'], g['sq_e2'])
    assert torch.allclose(out, g['sq_out'], atol=1e-7, rtol=0)
    for lvl in (1, 2):
        f, uv = D.get_icosphere_uvs(lvl)
        assert torch.equal(f, g[f'ico{lvl}_faces_uvs'])
        assert torch.allclose(uv, g[f'ico{lvl}_verts_uvs'], atol=1e-7, rtol=0)
    assert torch.allclose(D.world_rotation(115, 20, -30), g['R_world_115_20_m30'], atol=1e-6)


def test_cube_primitive_matches_reference_golden():
    """BASELINE configs[0]: the cube primitive (vertices / faces of primitives/cube.obj, UV cross of mesh.py:176-207) of
    the oracle AND of the product's geometry module, against vectors generated from the reference's files."""
    import dbw_b200  # noqa: F401
    from dbw_b200 import geometry as G
    g = _npz('ref_functions.npz')
    for verts, faces in (D.get_cube(), G.unit_cube()):
        assert torch.equal(verts, g['cube_verts']) and torch.equal(faces, g['cube_faces'])
    for f, uv in (D.get_cube_uvs(), G.cube_uvs()):
        assert torch.equal(f, g['cube_faces_uvs']) and torch.equal(uv, g['cube_verts_uvs'])
    pv, pf = G.unit_plane()
    assert torch.equal(pv, g['plane_verts']) and torch.equal(pf, g['plane_faces'])
    ov, of = D.get_plane()
    assert torch.equal(ov.reshape(-1, 3), g['plane_verts']) and torch.equal(of.reshape(-1, 3), g['plane_faces'])


def test_obj_loader_reads_the_reference_primitives():
    """the reference's primitives/*.obj, stored verbatim under tests/golden/primitives/"""
    import dbw_b200  # noqa: F401
    from dbw_b200 import geometry as G
    for name, (v, f) in (('cube', G.unit_cube()), ('plane', G.unit_plane())):
        lv, lf = G.load_obj(os.path.join(GOLD, 'primitives', f'{name}.obj'))
        assert torch.equal(lv, v) and torch.equal(lf, f), name


def test_render_cube_matches_golden():
    """BASELINE configs[0] on the CPU oracle (the config's own arm: 'PyTorch3D CPU rasterizer, plumbing, no GPU')."""
    from tests.golden.make_golden import render_cube
    cur = render_cube()
    g = np.load(os.path.join(GOLD, 'render_cube.npz'))
    assert (g['soft'][:, 3] > 0.5).mean() > 0.05 and (g['hard'][:, 3] == 1).mean() > 0.05      # the cube is in view
    for k in g.files:
        if k.startswith('grad_'):
            assert float(np.linalg.norm(cur[k] - g[k])) / max(float(np.linalg.norm(g[k])), 1e-12) < 1e-4, k
        else:
            assert np.abs(cur[k] - g[k]).max() <= 2e-6, k


def test_render_small_matches_golden():
    from tests.golden.make_golden import render_small
    cur = render_small()
    g = np.load(os.path.join(GOLD, 'render_small.npz'))
    for k in g.files:
        scale = max(1.0, float(np.abs(g[k]).max()))
        if k.startswith('grad_'):
            # gradients: libm / thread-count differences move a handful of texel contributions by an ulp
            denom = max(float(np.linalg.norm(g[k])), 1e-12)
            assert float(np.linalg.norm(cur[k] - g[k])) / denom < 1e-4, k
        else:
            assert np.abs(cur[k] - g[k]).max() <= 2e-6 * scale, k


def test_oracle_backward_matches_finite_differences():
    """float64 oracle: autograd (C backward + torch) vs central differences, constant textures so that detaching the
    barycentrics does not matter, K large enough that no face is evicted."""
    tpl = D.SceneTemplate(n_blocks=3, txt_size=16)
    p = D.init_params(3, 16, seed=2, dtype=torch.float64)
    p['textures'] = torch.randn(3, 1, 1, 3, dtype=torch.float64).expand(3, 16, 16, 3).clone()
    R, T, K = D.ring_cameras(2, dtype=torch.float64)
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(2, 3, 32, 40, generator=g, dtype=torch.float64)

    def loss_fn(pp):
        blocks, alpha = tpl.build_blocks(pp)
        out = D.render(blocks, R, T, K, (32, 40), sigma=1e-3, faces_per_pixel=60, z_clip=0.001, detach_bary=True,
                       faces_alpha=alpha.repeat_interleave(tpl.BNF))
        return D.mse_loss(imgs, out[:, :3]) + out[:, 3].mean()

    pg = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    loss_fn(pg).backward()
    for name, idx in [('T', (0, 0)), ('S', (1, 1)), ('R_6d', (2, 4)), ('alpha_logit', (1,)), ('sq_eps', (0, 1))]:
        h = 1e-6
        pp = {k: v.clone() for k, v in p.items()}
        pp[name][idx] += h
        lp = loss_fn(pp).item()
        pp[name][idx] -= 2 * h
        lm = loss_fn(pp).item()
        fd, ag = (lp - lm) / (2 * h), pg[name].grad[idx].item()
        assert abs(fd - ag) <= 1e-4 * max(abs(fd), abs(ag)) + 1e-9, (name, fd, ag)


def test_oracle_env_gradients_match_finite_differences():
    tpl = D.SceneTemplate(n_blocks=1, txt_size=16)
    p = D.init_params(1, 16, seed=4, dtype=torch.float64)
    R, T, K = D.ring_cameras(2, dtype=torch.float64)
    g = torch.Generator().manual_seed(0)
    w = torch.rand(2, 3, 24, 24, generator=g, dtype=torch.float64)

    def loss_fn(pp):
        return (D.render(tpl.build_env(pp), R, T, K, (24, 24), sigma=0, faces_per_pixel=1, z_clip=0.001)[:, :3] * w).sum()

    pg = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    loss_fn(pg).backward()
    for name, idx in [('T_ground', (0, 1)), ('R_6d_ground', (0, 2)), ('texture_ground', (0, 8, 8, 1))]:
        h = 1e-6
        pp = {k: v.clone() for k, v in p.items()}
        pp[name][idx] += h
        lp = loss_fn(pp).item()
        pp[name][idx] -= 2 * h
        lm = loss_fn(pp).item()
        fd, ag = (lp - lm) / (2 * h), pg[name].grad[idx].item()
        assert abs(fd - ag) <= 1e-4 * max(abs(fd), abs(ag)) + 1e-8, (name, fd, ag)


def test_oracle_edge_cases():
    """empty scene regions, a face fully behind the camera (culled), K larger than the number of faces."""
    verts = torch.tensor([[[-.5, -.5, 2.], [.5, -.5, 2.], [0., .5, 2.], [-.5, -.5, -1.], [.5, -.5, -1.], [0., .5, -1.]]])
    faces = torch.tensor([[0, 1, 2], [3, 4, 5]])
    fr = pt3d.rasterize_meshes(verts, faces, (16, 16), blur_radius=0.0, faces_per_pixel=4, z_clip_value=0.01)
    assert (fr.pix_to_face[..., 1:] == -1).all()                # never more than one face per pixel
    assert set(fr.pix_to_face.unique().tolist()) <= {-1, 0}     # the face behind the camera is culled
    assert (fr.pix_to_face[..., 0] == 0).sum() > 10
    assert (fr.zbuf[fr.pix_to_face >= 0] - 2.0).abs().max() < 1e-6


def test_restatements_match_reference_source():
    """bit-for-bit against the outputs of the reference's own code (tests/golden/ref_restatements.npz)."""
    from tests.golden.make_golden import BLEND_CASES
    g = _npz('ref_restatements.npz')
    col, p2f, d, fa = g['blend_colors'], g['blend_p2f'], g['blend_dists'], g['blend_faces_alpha']
    for i, (sigma, ci, a) in enumerate(BLEND_CASES):
        assert torch.equal(g[f'blend_out_{i}'], D.layered_rgb_blend(col, p2f, d, sigma, (0.1, 0.2, 0.3), ci, fa if a else None)), i
    assert torch.equal(g['sq_out'], D.parametric_sq(g['sq_eta'], g['sq_omega'], g['sq_e1'], g['sq_e2']))
    for lvl in (1, 2):
        fo, uvo = D.get_icosphere_uvs(lvl)
        assert torch.equal(g[f'ico{lvl}_faces_uvs'], fo) and torch.equal(g[f'ico{lvl}_verts_uvs'], uvo)


@pytest.mark.parametrize('coarse', [True, False])
@pytest.mark.parametrize('tv_type', ['l2sq', 'l2', 'l1'])
def test_regulariser_restatement_matches_reference_compute_losses(coarse, tv_type):
    """oracle.regularisers (parsimony / TV / overlap) against the reference's own DifferentiableBlocksWorld.compute_losses
    (src/model/dbw.py:361-408) on the same parameters and overlap samples (tests/golden/ref_restatements.npz)"""
    g = _npz('ref_restatements.npz')
    tpl = D.SceneTemplate(n_blocks=4, txt_size=16)
    p = {k[len('reg_p_'):]: v for k, v in g.items() if k.startswith('reg_p_')}
    keep = torch.sigmoid(p['alpha_logit']) > 0.01                    # kill_blocks
    ref = {k: g[f'reg_{int(coarse)}_{tv_type}_{k}'][0] for k in ('parsimony', 'tv', 'overlap')}
    got = D.regularisers(tpl, p, coarse=coarse, keep=keep, tv_type=tv_type, unit_samples=g['reg_u01'], weights=(0.01, 0.1, 1.0))
    for k in ('parsimony', 'tv', 'overlap'):
        assert torch.allclose(got[k], ref[k], rtol=1e-6, atol=1e-9), (k, got[k].item(), ref[k].item())
    if coarse:
        assert ref['overlap'] > 0 and ref['parsimony'] > 0
