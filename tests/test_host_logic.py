"""CPU: host-side logic of the product (no kernels are launched): topology/UV builders vs the oracle, the Meshes /
TexturesUV stand-ins, model construction from the reference's configs, view sharding, and the N>1 gradient
all-reduce path on the gloo backend (world_size 2)."""
import os
from copy import deepcopy

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import dbw_path as D, pt3d

REF_CFG = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_configs.json')

DTU_DEFAULT_MODEL = {          # restated values of configs/dtu/default.yml:1-26
    'name': 'dbw',
    'mesh': {'n_blocks': 10, 'S_world': 0.5, 'R_world': [115, 0, 0], 'txt_size': 256},
    'renderer': {'faces_per_pixel': 10, 'cameras': {'name': 'perspective'}, 'detach_bary': True, 'z_clip': 0.001},
    'rend_optim': {'coarse_learning': 1500, 'decimate_txt': 750, 'decimate_factor': 8, 'kill_blocks': True,
                   'decouple_rendering': True, 'opacity_noise': True},
    'loss': {'rgb_weight': 1, 'perceptual_weight': 0.1, 'parsimony_weight': 0.01, 'tv_weight': 0.1, 'overlap_weight': 1},
}


def test_geometry_builders_match_oracle():
    from dbw_b200 import geometry as G
    for lvl in (0, 1, 2):
        v, f = G.ico_sphere(lvl)
        vo, fo = pt3d.ico_sphere(lvl)
        assert torch.equal(f, fo) and torch.equal(v, vo)
    for lvl in (1, 2):
        f, uv = G.icosphere_uvs(lvl)
        fo, uvo = D.get_icosphere_uvs(lvl)
        assert torch.equal(f, fo) and torch.equal(uv, uvo)
    gv, gf = G.unit_plane()
    ov, of = D.get_plane()
    for _ in range(3):
        gv, gf = G.subdivide_mesh(gv, gf)
        ov, of = pt3d.subdivide(ov, of)
    assert torch.equal(gf, of) and torch.equal(gv, ov)
    assert torch.allclose(G.euler_world_rotation(115, 20, -30), D.world_rotation(115, 20, -30), atol=1e-7)
    d6 = torch.randn(5, 6)
    assert torch.allclose(G.rotation_6d_to_matrix(d6), pt3d.rotation_6d_to_matrix(d6), atol=1e-7)
    Rm = G.random_rotations(7)
    assert torch.allclose(Rm @ Rm.transpose(1, 2), torch.eye(3).expand(7, -1, -1), atol=1e-5)
    assert torch.allclose(torch.det(Rm), torch.ones(7), atol=1e-5)
    eta, om = torch.rand(3, 42) * 3 - 1.5, torch.rand(3, 42) * 6 - 3
    e1, e2 = torch.rand(3, 1) * 1.8 + 0.1, torch.rand(3, 1) * 1.8 + 0.1
    assert torch.equal(G.superquadric_points(eta, om, e1, e2), D.parametric_sq(eta, om, e1, e2))
    X = torch.randn(50, 3)
    assert torch.equal(G.spherical_uv(X), D.point_to_uv_sphericalmap(X))


def test_synthetic_cameras_match_oracle_and_look_at_origin():
    from dbw_b200.synthetic import ring_cameras
    R, T, K = ring_cameras(5, jitter=0.2, seed=3)
    Ro, To, Ko = D.ring_cameras(5, jitter=0.2, seed=3)
    assert torch.equal(R, Ro) and torch.equal(T, To) and torch.equal(K, Ko)
    origin_cam = (torch.zeros(5, 1, 3) @ R)[:, 0] + T          # X_cam = X_world @ R + T
    assert torch.allclose(origin_cam[:, :2], torch.zeros(5, 2), atol=1e-6) and (origin_cam[:, 2] > 2).all()
    assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3).expand(5, -1, -1), atol=1e-6)


def test_meshes_and_textures_join_scene():
    from dbw_b200 import Meshes, TexturesUV, join_meshes_as_scene
    v = torch.rand(2, 4, 3)
    f = torch.tensor([[[0, 1, 2], [0, 2, 3]]]).expand(2, -1, -1)
    maps = torch.rand(2, 5, 7, 3)
    fu = torch.tensor([[[0, 1, 2], [0, 2, 3]]]).expand(2, -1, -1)
    vu = torch.rand(2, 4, 2)
    a = Meshes(v, f, TexturesUV(maps, fu, vu))
    extra = Meshes(torch.rand(1, 3, 3), torch.tensor([[[0, 1, 2]]]), TexturesUV(torch.rand(1, 4, 4, 3), torch.tensor([[[0, 1, 2]]]), torch.rand(1, 3, 2)))
    scene = join_meshes_as_scene([a, extra])
    assert len(scene) == 1 and len(scene.extend(6)) == 6
    sv, sf = scene.get_mesh_verts_faces(0)
    assert sv.shape == (11, 3) and sf.shape == (5, 3) and sf.max() == 10
    assert torch.equal(sf[2:4], f[1] + 4) and torch.equal(sf[4], torch.tensor([8, 9, 10]))
    fvu, fmap = scene.textures.scene_arrays()
    assert fvu.shape == (5, 3, 2) and fmap.tolist() == [0, 0, 1, 1, 2]
    assert torch.equal(fvu[2], vu[1][fu[1][0]])
    flat, table = scene.textures.packed_maps()
    assert table == [(0, 5, 7), (105, 5, 7), (210, 4, 4)] and flat.numel() == 210 + 48
    assert torch.equal(flat[105:210].reshape(5, 7, 3), maps[1])


def _param_shapes(model):
    return {n: tuple(p.shape) for n, p in model.named_parameters()}


def test_model_constructs_with_reference_parameter_names():
    from dbw_b200.dbw import create_model
    cfg = {'model': deepcopy(DTU_DEFAULT_MODEL)}
    cfg['model']['mesh']['txt_size'] = 64
    model = create_model(cfg, (300, 400))
    assert _param_shapes(model) == {
        'sq_eps': (10, 2), 'R_6d_ground': (1, 6), 'T_ground': (1, 3), 'S': (10, 3), 'R_6d': (10, 6), 'T': (10, 3),
        'alpha_logit': (10,), 'texture_bkg': (1, 64, 64, 3), 'texture_ground': (1, 64, 64, 3), 'textures': (10, 64, 64, 3)}
    bufs = dict(model.named_buffers())
    assert set(bufs) == {'R_world', 'T_world', 'bkg_verts_uvs', 'ground_verts_uvs', 'sq_eta', 'sq_omega',
                         'block_faces_uvs', 'block_verts_uvs'}
    assert bufs['sq_eta'].shape == (10, 42) and bufs['block_faces_uvs'].shape == (80, 3) and bufs['block_verts_uvs'].shape == (63, 2)
    assert model.bkg_n_faces == 320 and model.ground_n_faces == 128 and model.blocks_n_faces == 800
    assert model.loss_names == ['loss_rgb', 'loss_perceptual', 'loss_parsimony', 'loss_tv', 'loss_overlap', 'loss_total']
    assert model.renderer.sigma == 1e-4 and model.renderer_fine.sigma == 5e-6 and model.renderer_env.faces_per_pixel == 1
    assert abs(model.renderer.blur_radius - 9.2102e-4) < 1e-7
    # the texture-prefixed Adam group of src/optimizer.py:9-14
    assert sorted(n for n, _ in model.named_parameters() if n.startswith('texture')) == ['texture_bkg', 'texture_ground', 'textures']
    # milestones
    assert model.is_live('coarse_learning') and model.is_live('decimate_txt')
    model.set_cur_epoch(1600)
    assert not model.is_live('coarse_learning')
    # checkpoint round trip incl. the spq_ -> sq_ rename of dbw.py:444-445
    sd = {k.replace('sq_', 'spq_'): v.clone() + 1 for k, v in model.state_dict().items()}
    model.load_state_dict(sd)
    assert torch.allclose(model.state_dict()['sq_eps'], sd['spq_eps'])


def test_every_reference_config_parses_unmodified():
    """the `model` section of every reference config (overlaid on its directory's default.yml, as the reference's
    load_yaml does), stored in tests/golden/ref_configs.json"""
    import json
    from dbw_b200.dbw import create_model
    n = 0
    for name, model_cfg in sorted(json.load(open(REF_CFG)).items()):
        cfg = {'model': model_cfg}
        cfg['model']['mesh']['txt_size'] = 16               # keep the CPU test light; every other key untouched
        model = create_model(cfg, (32, 48))
        assert model.n_blocks == cfg['model']['mesh']['n_blocks'], name
        n += 1
    assert n >= 18


def test_shard_views_is_a_balanced_partition():
    from dbw_b200.parallel import shard_views
    for B, W in [(49, 8), (49, 1), (64, 8), (5, 8), (256, 3)]:
        parts = [shard_views(B, W, r) for r in range(W)]
        assert parts[0].start == 0 and parts[-1].stop == B
        assert all(parts[i].stop == parts[i + 1].start for i in range(W - 1))
        sizes = [p.stop - p.start for p in parts]
        assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
    assert [p.stop - p.start for p in [shard_views(49, 8, r) for r in range(8)]] == [7, 6, 6, 6, 6, 6, 6, 6]


class _ToyScene(torch.nn.Module):
    """stands in for the scene model on CPU: per-view 'render' loss + a view-independent regulariser + opacity noise."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.arange(6, dtype=torch.float32).reshape(2, 3) / 10)
        self.textures = torch.nn.Parameter(torch.ones(4))
        self.n_total_views, self.noise_generator = None, None

    def forward(self, inp, labels=None):
        noise = torch.randn(4, generator=self.noise_generator)
        pred = inp['imgs'] * self.w.sum() + (self.textures * (1 + 0.1 * noise)).sum()
        rgb = ((pred - inp['R'].sum((1, 2))[:, None]) ** 2).sum() / (self.n_total_views * pred.shape[1])
        reg = (self.w ** 2).sum() + self.textures.abs().sum()
        return {'rgb': rgb, 'tv': reg, 'total': rgb + reg}


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from dbw_b200.parallel import ViewParallel
    torch.manual_seed(0)
    model = _ToyScene()
    vp = ViewParallel(model, seed=123)
    g = torch.Generator().manual_seed(1)
    inp = {'imgs': torch.rand(7, 5, generator=g), 'R': torch.rand(7, 3, 3, generator=g), 'T': torch.rand(7, 3, generator=g)}
    vp.forward_backward(inp)
    out[rank] = vp.bucket.flat.clone()
    dist.destroy_process_group()


class _ToyRows(torch.nn.Module):
    """per-pixel 'render' loss over (B,H,W) images that honours inp['rows'] the way the kernels do (dbw_render.h view_rows)"""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.linspace(0.1, 0.9, 5))
        self.textures = torch.nn.Parameter(torch.ones(3))
        self.n_total_views, self.noise_generator = None, None

    def forward(self, inp, labels=None):
        imgs = inp['imgs']
        B, H, W = imgs.shape
        pred = imgs * self.w[None, None] + self.textures.sum() * inp['R'].sum((1, 2))[:, None, None]
        err = (pred - 0.5) ** 2
        if inp.get('rows') is not None:
            y = torch.arange(H)[None, :, None]
            err = err * ((y >= inp['rows'][:, 0, None, None]) & (y < inp['rows'][:, 1, None, None]))
        rgb = err.sum() / (self.n_total_views * H * W)
        reg = self.textures.pow(2).sum()
        return {'rgb': rgb, 'tv': reg, 'total': rgb + reg}


def _worker_rows(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from dbw_b200.parallel import ViewParallel
    torch.manual_seed(0)
    vp = ViewParallel(_ToyRows(), seed=123, row_bands=True)
    g = torch.Generator().manual_seed(1)
    inp = {'imgs': torch.rand(5, 48, 5, generator=g), 'R': torch.rand(5, 3, 3, generator=g), 'T': torch.rand(5, 3, generator=g)}
    local, n_total = vp.shard(inp)
    out[f'rows{rank}'] = local['rows'].clone()
    vp.forward_backward(inp)
    out[rank] = vp.bucket.flat.clone()
    dist.destroy_process_group()


def test_row_band_view_parallel_gradients_equal_single_process_gloo():
    """world_size-2 gloo run with (view, row band) sharding: the ranks split a view in the middle; the summed gradient is the
    single-process gradient of the same step"""
    from dbw_b200.parallel import ViewParallel
    mgr = mp.Manager()
    out = mgr.dict()
    port = 31000 + os.getpid() % 2000
    mp.spawn(_worker_rows, args=(2, port, out), nprocs=2, join=True)
    assert out['rows0'].tolist() == [[0, 48], [0, 48], [0, 32]] and out['rows1'].tolist() == [[32, 48], [0, 48], [0, 48]]
    torch.manual_seed(0)
    vp = ViewParallel(_ToyRows(), seed=123)
    g = torch.Generator().manual_seed(1)
    inp = {'imgs': torch.rand(5, 48, 5, generator=g), 'R': torch.rand(5, 3, 3, generator=g), 'T': torch.rand(5, 3, generator=g)}
    vp.forward_backward(inp)
    ref = torch.nn.functional.pad(vp.bucket.grads_flat(), (0, vp.bucket.flat.numel() - vp.bucket.n))
    assert torch.allclose(out[0], out[1]) and torch.allclose(out[0], ref, rtol=1e-5, atol=1e-7)


def test_row_band_sharding_is_a_balanced_partition():
    """parallel.shard_row_bands: every (view, row) exactly once, contiguous pieces, loads within one 16-row band"""
    from dbw_b200.parallel import shard_row_bands, ROW_BAND
    for n_views, H, world in [(49, 400, 8), (49, 400, 2), (64, 576, 8), (256, 800, 8), (3, 50, 4), (1, 16, 4), (5, 400, 1)]:
        seen = torch.zeros(n_views, H, dtype=torch.int32)
        loads = []
        for r in range(world):
            pieces = shard_row_bands(n_views, H, world, r)
            assert [v for v, _, _ in pieces] == sorted(set(v for v, _, _ in pieces))       # one piece per touched view, in order
            for v, a, b in pieces:
                assert 0 <= a < b <= H and a % ROW_BAND == 0
                seen[v, a:b] += 1
            loads.append(sum(b - a for _, a, b in pieces))
        assert (seen == 1).all(), (n_views, H, world)
        assert max(loads) - min(loads) <= ROW_BAND, loads
    # 49 views over 8 ranks: 6.12 views' worth of rows each instead of 7 whole views on the busiest rank
    assert max(sum(b - a for _, a, b in shard_row_bands(49, 400, 8, r)) for r in range(8)) == 2464


def test_view_parallel_gradients_equal_single_process_gloo():
    """world_size-2 gloo run: sharded views + ONE all-reduce == the single-process gradient of the same step."""
    from dbw_b200.parallel import ViewParallel
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29000 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    torch.manual_seed(0)
    model = _ToyScene()
    vp = ViewParallel(model, seed=123, gather_grads=True)         # one rank: nothing reads the bucket unless asked for
    g = torch.Generator().manual_seed(1)
    inp = {'imgs': torch.rand(7, 5, generator=g), 'R': torch.rand(7, 3, 3, generator=g), 'T': torch.rand(7, 3, generator=g)}
    vp.forward_backward(inp)
    ref = vp.bucket.flat
    assert torch.allclose(out[0], out[1], atol=0)                 # every rank holds the same reduced gradient
    assert torch.allclose(out[0], ref, rtol=1e-5, atol=1e-6)
    assert vp.bucket.flat.data_ptr() == model.w.grad.data_ptr()   # grads are views into the single bucket


def test_grad_bucket_backward_gathers_like_accumulation():
    """GradBucket.backward (parameters enter the backward without .grad, ONE cat gathers the gradients into the flat
    buffer) == zero the bucket + autograd's accumulate-adds; parameters the loss does not reach read as zero; the .grad
    attributes are the bucket views again afterwards, and a second step does not accumulate onto the first."""
    from dbw_b200.parallel import GradBucket
    torch.manual_seed(3)
    a, b, unused = (torch.nn.Parameter(torch.randn(s)) for s in ((4, 3), (5,), (2, 2)))
    loss_fn = lambda: (a.sin().sum() * b.pow(2).sum() + (a[:, 0] * b[:4]).sum())
    bucket = GradBucket([a, b, unused])
    bucket.backward(loss_fn())
    got = bucket.flat.clone()
    assert bucket.n == 21 and bucket.flat.numel() == 24             # padded to whole 128-bit lanes for the all-reduce kernel
    ga, gb = torch.autograd.grad(loss_fn(), [a, b])
    ref = torch.cat([ga.reshape(-1), gb.reshape(-1), torch.zeros(4 + 3)])
    assert torch.allclose(got, ref, rtol=1e-6, atol=1e-7)
    for p in (a, b, unused):
        assert p.grad is not None and p.grad.untyped_storage().data_ptr() == bucket.flat.untyped_storage().data_ptr()
    assert torch.equal(a.grad, ga) and torch.equal(unused.grad, torch.zeros(2, 2))
    bucket.backward(2 * loss_fn())                                   # overwrites, does not accumulate
    assert torch.allclose(bucket.flat, 2 * ref, rtol=1e-6, atol=1e-7)
    bucket.zero_()                                                   # the classic path still works on the same views
    loss_fn().backward()
    assert torch.allclose(bucket.flat, ref, rtol=1e-6, atol=1e-7)
    # gather=False (no collective reads the bucket): .grad are autograd's own tensors, the flat buffer is left alone,
    # grads_flat() concatenates on demand, and zero_() re-installs the views for the classic protocol
    before = bucket.flat.clone()
    bucket.backward(3 * loss_fn(), gather=False)
    assert torch.equal(bucket.flat, before) and unused.grad is None
    assert a.grad.untyped_storage().data_ptr() != bucket.flat.untyped_storage().data_ptr()
    assert torch.allclose(bucket.grads_flat(), 3 * ref[:21], rtol=1e-6, atol=1e-7)
    bucket.zero_()
    assert a.grad.untyped_storage().data_ptr() == bucket.flat.untyped_storage().data_ptr()
    loss_fn().backward()
    assert torch.allclose(bucket.flat, ref, rtol=1e-6, atol=1e-7)


def test_scene_settings_of_a_render_pass():
    """host-side bookkeeping of one pass (no kernel runs): per-face vs per-view-and-face opacity strides, texel-atlas map
    sizes, the blur radius of renderer.py:51, and the saved-fragment-state switch following grad mode."""
    import numpy as np
    from dbw_b200.renderer import scene_settings
    from dbw_b200._lib import DbwError
    V, F, B = 12, 20, 3
    verts, faces = torch.zeros(V, 3), torch.zeros(F, 3, dtype=torch.int32)
    atlas = torch.zeros(2 * 8 * 8, 4)                                  # two 8x8 float4 maps
    table = [(0, 8, 8), (8 * 8 * 3, 8, 8)]
    intr = (2.0, 2.0, 0.0, 0.0)
    cfg, dev_table = scene_settings(verts, faces, atlas, table, B, intr, (16, 24), 1e-4, 10, 0.001, detach_bary=True,
                                    faces_alpha=torch.ones(F), maps_are_texels4=True)
    assert (cfg.n_views, cfg.height, cfg.width, cfg.faces_per_pixel, cfg.n_verts, cfg.n_faces, cfg.n_maps) == (B, 16, 24, 10, V, F, 2)
    assert cfg.alpha_view_stride == 0 and cfg.maps_are_texels4 == 1 and cfg.n_map_floats == 2 * 8 * 8 * 3
    assert abs(cfg.blur_radius - np.log(1. / 1e-4 - 1.) * 1e-4) < 1e-9 and abs(cfg.z_clip - 0.001) < 1e-9
    assert cfg.save_fragment_state == 1                                # detach_bary pass, grad mode on
    assert dev_table.reshape(-1, 4)[:, :3].tolist() == [[0, 8, 8], [192, 8, 8]]
    with torch.no_grad():
        cfg2, _ = scene_settings(verts, faces, atlas, table, B, intr, (16, 24), 1e-4, 10, None, detach_bary=True,
                                 faces_alpha=torch.ones(B * F), maps_are_texels4=True)
    assert cfg2.save_fragment_state == 0 and cfg2.alpha_view_stride == F and cfg2.z_clip == -1.0
    with pytest.raises(DbwError):
        scene_settings(verts, faces, atlas, table, B, intr, (16, 24), 1e-4, 10, faces_alpha=torch.ones(F + 1))


class _ToyScenePoint(torch.nn.Module):
    """a scene model that routes what its 'render' differentiates through the data-parallel gradient-sum point the way
    DifferentiableBlocksWorld does (dbw.py _scene_tensors): scene tensors = f(leaves), rgb = g(scene tensors), plus a
    view-independent regulariser that does NOT pass through the point"""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.linspace(0.1, 0.9, 5))
        self.textures = torch.nn.Parameter(torch.linspace(-1, 1, 6))
        self.n_total_views, self.noise_generator, self.grad_sum_point = None, None, None
        self.point_calls = 0

    def _fused_loss_ok(self, imgs):
        return True

    def can_sum_gradients_at_scene_tensors(self, imgs):
        return True

    def grad_sum_floats(self):
        return 5 + 3

    def forward(self, inp, labels=None):
        verts, cells = self.w.exp(), torch.sigmoid(self.textures).view(3, 2).mean(1)          # leaves -> scene tensors
        if self.grad_sum_point is not None:
            verts, cells = self.grad_sum_point(verts, cells)
            self.point_calls += 1
        imgs = inp['imgs']
        B, H, W = imgs.shape
        err = (imgs * verts[None, None] + cells.sum() * inp['R'].sum((1, 2))[:, None, None] - 0.5) ** 2
        if inp.get('rows') is not None:
            y = torch.arange(H)[None, :, None]
            err = err * ((y >= inp['rows'][:, 0, None, None]) & (y < inp['rows'][:, 1, None, None]))
        rgb = err.sum() / (self.n_total_views * H * W)
        reg = self.textures.pow(2).sum() + self.w.sum()
        return {'rgb': rgb, 'tv': reg, 'total': rgb + reg}


class _GlooBucket:
    """stands in for parallel.PeerAllReduce on CPU: a flat bucket and an in-place sum over the ranks of a prefix of it"""

    def __init__(self, n_floats, device):
        self.flat = torch.zeros(n_floats)
        self.sizes = []

    def all_reduce(self, buf):
        assert buf.data_ptr() == self.flat.data_ptr() and buf.numel() % 4 == 0
        self.sizes.append(buf.numel())
        dist.all_reduce(buf)


def _worker_point(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from dbw_b200.parallel import ViewParallel
    torch.manual_seed(0)
    model = _ToyScenePoint()
    vp = ViewParallel(model, seed=123, row_bands=True, peer_factory=_GlooBucket)
    g = torch.Generator().manual_seed(1)
    inp = {'imgs': torch.rand(5, 48, 5, generator=g), 'R': torch.rand(5, 3, 3, generator=g), 'T': torch.rand(5, 3, generator=g)}
    assert vp.sum_point is not None and vp.reduces_inside_backward(inp)
    vp.forward_backward(inp)
    vp.forward_backward(inp)                       # the bucket is reused
    out[rank] = (vp.bucket.grads_flat().clone(), model.point_calls, list(vp.bucket.peer.sizes),
                 model.w.grad.data_ptr() != vp.bucket.flat.data_ptr())
    dist.destroy_process_group()


def test_gradients_summed_at_the_scene_tensors_equal_single_process_gloo():
    """world_size-2 gloo run of the scene-level reduction (parallel.GradSumPoint over a gloo stand-in for the peer-memory
    bucket): ONE small exchange inside each backward, no leaf all-reduce, no gather; the leaf gradients -- chain rule applied
    to the summed scene-tensor gradients, regulariser counted once -- equal the single-process step's on both ranks"""
    from dbw_b200.parallel import ViewParallel
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker_point, args=(2, 33000 + os.getpid() % 2000, out), nprocs=2, join=True)
    torch.manual_seed(0)
    model = _ToyScenePoint()
    vp = ViewParallel(model, seed=123)
    g = torch.Generator().manual_seed(1)
    inp = {'imgs': torch.rand(5, 48, 5, generator=g), 'R': torch.rand(5, 3, 3, generator=g), 'T': torch.rand(5, 3, generator=g)}
    vp.forward_backward(inp)
    ref = vp.bucket.grads_flat()
    assert model.point_calls == 0                                     # one rank: no sum point in the graph
    for rank in (0, 1):
        got, calls, sizes, own_grads = out[rank]
        assert calls == 2 and sizes == [8, 8] and own_grads           # 5 + 3 floats per step; .grad not gathered into the bucket
        assert torch.allclose(got, ref, rtol=1e-5, atol=1e-7), (rank, got, ref)
    assert torch.equal(out[0][0], out[1][0])
