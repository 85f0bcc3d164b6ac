"""Drives the reference's UNMODIFIED `src/trainer.py` (+ optimizer.py, scheduler.py, utils/*, configs/dtu/*.yml) on this repo's
model, from a checkout of the reference (monniert/differentiable-blocksworld):

    python tests/ref_trainer_driver.py --reference <checkout> <run_dir> [--iters N]

It prints one `DRIVER_RESULT <json>` line: loss names, Adam groups, moved parameters, checkpoint keys, metrics rows, resume.

What is swapped (INTEGRATION.md A, nothing in the reference tree is edited or copied):
  * `model.create_model`                 -> dbw_b200.dbw.create_model   (the drop-in)
  * `dataset.create_train_val_test_loader` -> a synthetic multi-view loader (no DTU images on disk here)
  * missing third-party modules          -> dbw_b200.compat stand-ins

With a GPU the model renders for real.  WITHOUT one the product renderer refuses to run -- there is
no CPU fallback, by design -- so this driver replaces the model's three render entry points by parameter-touching dummies and
says so: what the run then proves is the whole trainer <-> model surface (config parsing, loss names, Adam groups,
schedules, metrics, visualisation calls, checkpoints, resume), not pixels."""
import argparse
import json
import os
import sys
from pathlib import Path

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

import dbw_b200  # noqa: E402,F401
import dbw_b200.compat as compat  # noqa: E402
import dbw_b200.dbw as b200  # noqa: E402
from dbw_b200.synthetic import ring_cameras  # noqa: E402


class SyntheticViews(torch.utils.data.Dataset):
    """what src/dataset/dtu.py:58-68 yields per item: ({'imgs','K','R','T'}, {'points'})"""
    name, tag = 'synthetic', 'ring'

    def __init__(self, split, img_size, n_views=8, **unused):
        self.img_size = tuple(img_size)
        self.R, self.T, self.K = ring_cameras(n_views)
        g = torch.Generator().manual_seed({'train': 1, 'val': 2, 'test': 3}[split])
        self.imgs = torch.rand(n_views, 3, *self.img_size, generator=g)
        self.pc_gt = torch.rand(500, 3, generator=g) - 0.5

    def __len__(self):
        return len(self.imgs)

    def __getitem__(self, i):
        return {'imgs': self.imgs[i], 'K': self.K, 'R': self.R[i], 'T': self.T[i]}, {'points': self.pc_gt[:100]}


def synthetic_loaders(cfg, rank=None, world_size=None):
    from torch.utils.data import DataLoader
    kwargs = dict(cfg['dataset'])
    kwargs.pop('name'), kwargs.pop('tag', None)
    bs = cfg['training']['batch_size']
    mk = lambda split, shuffle: DataLoader(SyntheticViews(split, **kwargs), batch_size=bs, num_workers=0, shuffle=shuffle)
    return mk('train', True), mk('val', False), mk('test', False)


def stub_render_entry_points():
    """no GPU: differentiable stand-ins for forward / predict / predict_synthetic that touch every parameter"""
    M = b200.DifferentiableBlocksWorld

    def forward(self, inp, labels=None):
        reg = sum(p.float().pow(2).mean() for p in self.parameters())
        terms = {k: reg * (i + 1) * 1e-3 for i, k in enumerate(self.loss_weights)}
        terms['total'] = sum(terms.values())
        return terms

    def predict(self, inp, labels=None, w_edges=False, filter_transparent=False):
        return torch.sigmoid(self.texture_bkg.mean()) * torch.ones_like(inp['imgs'])

    M.forward, M.predict, M.predict_synthetic = forward, predict, lambda self, inp, labels=None: torch.ones_like(inp['imgs'])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('run_dir')
    ap.add_argument('--reference', required=True, help='checkout of the reference')
    ap.add_argument('--iters', type=int, default=3)
    args = ap.parse_args()
    REF = os.path.realpath(args.reference)
    shimmed = compat.install()
    sys.path.insert(0, os.path.join(REF, 'src'))
    import dataset as ref_dataset
    import model as ref_model
    ref_model.create_model = b200.create_model
    ref_dataset.create_train_val_test_loader = synthetic_loaders
    import trainer as ref_trainer                          # the reference's file, unmodified
    from utils import load_yaml                            # the reference's config loader (scan24.yml + default.yml merge)
    assert os.path.realpath(ref_trainer.__file__).startswith(REF)
    stubbed = not torch.cuda.is_available()
    if stubbed:
        stub_render_entry_points()
    cfg = load_yaml(Path(REF) / 'configs' / 'dtu' / 'scan24.yml')
    cfg['dataset'].update(img_size=[48, 64])               # a small image; everything else as shipped
    cfg['model']['mesh']['txt_size'] = 32
    cfg['training'].update(batch_size=4, n_workers=0, n_epoches=2, train_stat_interval=1, val_stat_interval=2, visualizer_port=None)
    run_dir = Path(args.run_dir)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')                    # the LPIPS-unavailable warning is expected here
        T = ref_trainer.Trainer(cfg, run_dir, seed=cfg['training']['seed'])
    if T.model.loss_weights.get('perceptual') and getattr(T.model, 'perceptual_loss', None) is None:
        T.model.set_perceptual_loss(lambda imgs, rec: (imgs - rec).abs().mean())        # stand-in callable (no LPIPS weights here)
    groups = [len(g['params']) for g in T.optimizer.param_groups]
    lrs = [g['lr'] for g in T.optimizer.param_groups]
    before = {n: p.detach().clone() for n, p in T.model.named_parameters()}
    it = 0
    for images, labels in T.train_loader:
        T.run_single_batch_train(images, labels)           # trainer.py:137-147
        it += 1
        T.log_train_metrics(it, 1, it)
        if it >= args.iters:
            break
    T.run_val_and_log(it, 1, it)                           # opacities + colour map (trainer.py:150-163)
    T.log_visualizations(it)                               # predict(w_edges) / hard / synthetic / textures (trainer.py:177-199)
    T.step(2, batch=1)                                     # scheduler + model.step()
    T.save(epoch=1, batch=it)
    moved = sorted(n for n, p in T.model.named_parameters() if not torch.equal(p.detach(), before[n]))
    ckpt = torch.load(run_dir / 'model.pkl', map_location='cpu', weights_only=False)
    out = {'shimmed': shimmed, 'stubbed_render': stubbed, 'device': str(T.device), 'loss_names': T.model.loss_names,
           'param_groups': groups, 'lrs': lrs, 'moved': moved, 'cur_epoch': T.model.cur_epoch,
           'checkpoint_keys': sorted(ckpt['model_state'].keys()), 'model_name': ckpt['model_name'],
           'train_metrics_rows': len(open(run_dir / 'train_metrics.tsv').read().strip().splitlines()),
           'val_metrics_rows': len(open(run_dir / 'val_metrics.tsv').read().strip().splitlines()),
           'images': sorted(str(p.relative_to(run_dir)) for p in run_dir.glob('*/*.jpg'))[:3] + sorted(str(p.relative_to(run_dir)) for p in run_dir.glob('*/*.png'))[:2]}
    # resume from the checkpoint through the reference's own load_from (trainer.py:84-108)
    cfg2 = load_yaml(Path(REF) / 'configs' / 'dtu' / 'scan24.yml')
    cfg2['dataset'].update(img_size=[48, 64]); cfg2['model']['mesh']['txt_size'] = 32
    cfg2['training'].update(batch_size=4, n_workers=0, n_epoches=2, train_stat_interval=1, val_stat_interval=2, visualizer_port=None)
    ref_trainer.RUNS_PATH = run_dir.parent.parent                                  # runs/<dataset>/<tag>/model.pkl
    cfg2['training']['resume'] = run_dir.name
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        T2 = ref_trainer.Trainer(cfg2, run_dir, seed=1)
    out['resumed_epoch_start'] = T2.epoch_start
    out['resume_equal'] = all(torch.equal(a.detach().cpu(), b.detach().cpu())
                              for a, b in zip(T.model.state_dict().values(), T2.model.state_dict().values()))
    print('DRIVER_RESULT ' + json.dumps(out))


if __name__ == '__main__':
    main()
