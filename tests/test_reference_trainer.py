"""CPU: the import shims of dbw_b200.compat through which the reference's UNMODIFIED trainer pipeline (src/trainer.py +
optimizer.py + scheduler.py + utils/*) runs on this repo's model.  tests/ref_trainer_driver.py runs that pipeline against
a checkout of the reference."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_compat_shims_are_thin_and_fail_loudly():
    """in a subprocess (the stand-ins must not leak into this session): real helpers work, placeholders raise when called"""
    code = r'''
import sys; sys.path.insert(0, %r)
import torch, dbw_b200, dbw_b200.compat as compat
names = compat.install()
import toolz
assert toolz.merge({'a': 1}, {'b': 2}) == {'a': 1, 'b': 2} and toolz.valmap(lambda v: v + 1, {'a': 1}) == {'a': 2}
assert toolz.keyfilter(lambda k: k != 'a', {'a': 1, 'b': 2}) == {'b': 2} and toolz.valfilter(lambda v: v > 1, {'a': 1, 'b': 2}) == {'b': 2}
if 'pytorch3d' in names:
    from pytorch3d.structures import Meshes
    from pytorch3d.utils import ico_sphere
    from pytorch3d.ops import SubdivideMeshes
    from pytorch3d.transforms import rotation_6d_to_matrix, matrix_to_rotation_6d, random_rotations
    from pytorch3d.io import save_ply
    m = ico_sphere(1)
    v, f = m.get_mesh_verts_faces(0)
    assert v.shape == (42, 3) and f.shape == (80, 3)
    v2, f2 = SubdivideMeshes()(m).get_mesh_verts_faces(0)
    assert v2.shape == (162, 3) and f2.shape == (320, 3)
    R = random_rotations(4)
    assert torch.allclose(rotation_6d_to_matrix(matrix_to_rotation_6d(R)), R, atol=1e-5)
    try:
        save_ply('x.ply', v)
        raise SystemExit('placeholder did not raise')
    except NotImplementedError:
        pass
if 'seaborn' in names:
    import seaborn as sns
    from matplotlib import colors as mplcolors
    from dbw_b200 import geometry as G
    pal = sns.color_palette('hls', 21)
    cm = mplcolors.LinearSegmentedColormap.from_list('Custom', [mplcolors.to_rgb('gold')] + pal[3:] + pal[:2])
    import numpy as np
    x = np.linspace(0, 1, 11)
    assert np.allclose(cm(x)[:, :3], G.fancy_cmap()(x))
print('OK')
''' % ROOT
    res = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and 'OK' in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]
