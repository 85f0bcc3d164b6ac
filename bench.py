#!/usr/bin/env python
"""bench.py -- render+backward views/sec of the DBW render hot path (BASELINE.json metric).

A "step" = one optimisation step's render work on one batch of B synthetic views: build the scene from the leaf
parameters, render the environment pass (K=1, sigma=0) and the blocks pass (K, sigma=1e-4, per-block opacities),
composite + MSE against the target images, and back-propagate to every leaf parameter
(S, R_6d, T, sq_eps, alpha_logit, textures, texture_bkg, texture_ground, R_6d_ground, T_ground).  SURVEY.md 8d.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload dtu|bmvs|stress]     our arm (torchrun launches N ranks)
  python bench.py --impl reference ...                            the reference's algorithm on the host cores (oracle port)
  python bench.py ... --dump-outputs DIR       also write what the last timed step computed (losses, every leaf gradient)
                                               as DIR/<name>.npy, to compare two builds output for output

Workloads = BASELINE.json configs: dtu = configs[1]/[2] (the metric's configuration and the default), bmvs = configs[3],
stress = configs[4].  N > 1 is STRONG scaling: the step's views are split over the ranks at (view, 16-row band) granularity.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    'dtu': dict(baseline='configs[1] (1 GPU) / configs[2] (8 GPUs)', n_blocks=10, n_views=49, height=400, width=400,
                faces_per_pixel=10, txt_size=256, txt_bkg_upscale=1,
                what='DTU scan24 shape: 10 superquadric blocks (800 faces) + env (448 faces), 49 views 400x400, K=10, 256^2 textures'),
    'bmvs': dict(baseline='configs[3]', n_blocks=10, n_views=64, height=576, width=768, faces_per_pixel=10, txt_size=256,
                 txt_bkg_upscale=1, what='BlendedMVS shape: 10 blocks + env, 64 views 576x768, K=10, 256^2 textures'),
    'stress': dict(baseline='configs[4]', n_blocks=50, n_views=256, height=800, width=800, faces_per_pixel=25, txt_size=128,
                   txt_bkg_upscale=2, what='stress shape (configs/bmvs/gundam_50.yml): 50 blocks (4000 faces) + env, 256 views '
                                           '800x800, K=25, 128^2 block textures, 256^2 env textures'),
}
SEED = 227391          # configs/dtu/default.yml:42
DUMP_LIMIT = 64 << 20  # bytes --dump-outputs may write
PASS_BYTES = 30e9      # views of a step are processed in passes of at most this much workspace (gradients accumulate)


def model_cfg(w):
    return {
        'mesh': {'n_blocks': w['n_blocks'], 'S_world': 0.5, 'R_world': [115, 0, 0], 'txt_size': w['txt_size'],
                 'txt_bkg_upscale': w['txt_bkg_upscale']},
        'renderer': {'faces_per_pixel': w['faces_per_pixel'], 'cameras': {'name': 'perspective'}, 'detach_bary': True, 'z_clip': 0.001},
        'rend_optim': {'coarse_learning': 1500, 'decimate_txt': 750, 'decimate_factor': 8, 'kill_blocks': True,
                       'decouple_rendering': True, 'opacity_noise': True},
        'loss': {'rgb_weight': 1},
    }


def metric_name(w):
    return f'render+backward views/sec ({w["height"]}x{w["width"]}, {w["n_blocks"]} blocks)'


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def kernel_fingerprint():
    """sha256 over the sources of the raster kernels (dbw_render.cu and the headers it includes): ties a committed ncu capture
    (profiles/ncu_traffic.json) to the build that is benched"""
    h = hashlib.sha256()
    d = os.path.join(ROOT, 'differentiable-blocksworld_b200', 'csrc')
    for fn in ('dbw_render.cu', 'dbw_math.cuh', 'dbw_fraglist.cuh', 'dbw_clip.cuh'):
        h.update(open(os.path.join(d, fn), 'rb').read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel_label, workload, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_label` from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by scripts/summarize_profile.py) -- only if it was taken on THIS build of the kernels,
    this workload and one GPU; else None"""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if world != 1 or not os.path.exists(path):
        return None, 'no capture'
    d = json.load(open(path))
    if d.get('kernel_fingerprint') != kernel_fingerprint() or d.get('workload') != workload:
        return None, f'profiles/ncu_traffic.json is from another build ({d.get("kernel_fingerprint")}) or workload: not used'
    return d['bytes_per_launch'].get(kernel_label), f'{d.get("source", "profiles/ncu_traffic.json")} (same kernel sources: {d["kernel_fingerprint"]})'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line): one background
    `nvidia-smi -lms 100` process, started before the region and stopped after it."""
    QUERY = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.QUERY}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.25)                      # let the first sample land before the timed region starts
        except Exception:
            self.proc = None

    def summary(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ''
        rows = [[c.strip() for c in l.split(',')] for l in out.strip().splitlines() if l.count(',') >= 6]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        num = lambda x: float(x) if x.replace('.', '', 1).isdigit() else None
        sm = sorted(v for v in (num(r[0]) for r in rows) if v is not None)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in rows)]
        pw = [v for v in (num(r[2]) for r in rows) if v is not None]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': num(rows[0][1]), 'reasons': reasons,
                'samples': len(rows), 'power_w_max': max(pw) if pw else None}


def synthetic_inputs(w):
    from dbw_b200.synthetic import ring_cameras
    B, H, W = w['n_views'], w['height'], w['width']
    R, T, K = ring_cameras(B)
    g = torch.Generator().manual_seed(SEED)
    imgs = torch.rand(B, 3, H, W, generator=g)
    return {'imgs': imgs, 'R': R, 'T': T, 'K': K[None].expand(B, -1, -1).contiguous()}


def dump_outputs(out_dir, model, losses, loss_suffix=''):
    """the step's result as its caller holds it: the loss terms and the gradient of every leaf parameter (p.grad), float32"""
    import numpy as np
    arrays = {f'loss_{k}{loss_suffix}': v.detach().float().reshape(1) for k, v in losses.items()}
    for n, p in model.named_parameters():
        if p.requires_grad:
            arrays[f'grad_{n}'] = (p.grad if p.grad is not None else torch.zeros_like(p)).detach().float()
    total = sum(v.numel() * 4 for v in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f'--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte limit')
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), v.cpu().numpy())


def make_passes(local, rows, w):
    """split this rank's views into passes of equal shape: [{imgs, R, T, K, rows}] (host, pinned).  Padding entries of the
    last pass repeat view 0 with an EMPTY row range, so that one captured graph serves every pass."""
    B_local, H, W, K = len(local['imgs']), w['height'], w['width'], w['faces_per_pixel']
    per_view = H * W * (32 * K + 33 + 16 * 6 + 12)          # fragment records + count (both passes), RGBA-sized images, target
    cap = max(1, int(PASS_BYTES // per_view))
    n_pass = -(-B_local // cap)
    size = -(-B_local // n_pass)
    if rows is None:
        rows = torch.tensor([[0, H]] * B_local, dtype=torch.int32)
    passes = []
    for p in range(n_pass):
        idx = list(range(p * size, min((p + 1) * size, B_local)))
        pad = size - len(idx)
        sel = torch.tensor(idx + [0] * pad)
        chunk = {k: v[sel].contiguous() for k, v in local.items()}
        r = rows[sel].clone()
        if pad:
            r[len(idx):] = 0
        chunk['rows'] = r.contiguous()
        passes.append({k: v.pin_memory() for k, v in chunk.items()})
    return passes


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch.distributed as dist
    rank, world, local = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    assert world == args.gpus or world == 1, f'WORLD_SIZE={world} but --gpus {args.gpus}'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    import dbw_b200  # noqa: F401
    from dbw_b200 import _lib, fused_loss
    from dbw_b200.dbw import DifferentiableBlocksWorld
    from dbw_b200.parallel import ViewParallel
    from dbw_b200.graph import GraphedStep, PipelinedGraphedStep
    from copy import deepcopy
    fused_loss.OVERLAP_BACKWARD_PASSES = args.overlap_bwd == 'on' or (args.overlap_bwd == 'auto' and world >= 4)

    w = WORKLOADS[args.workload]
    B, H, W, K = w['n_views'], w['height'], w['width'], w['faces_per_pixel']
    torch.manual_seed(SEED)
    model = DifferentiableBlocksWorld((H, W), **deepcopy(model_cfg(w))).to(dev)
    model.train()
    vp = ViewParallel(model, seed=SEED, row_bands=True, collective=args.collective)
    host_local, _ = vp.shard(synthetic_inputs(w))
    rows = host_local.pop('rows', None)
    passes = make_passes(host_local, rows, w)
    n_pass, views_per_pass = len(passes), len(passes[0]['imgs'])
    local_px = int(sum(int((p['rows'][:, 1] - p['rows'][:, 0]).sum()) for p in passes)) * W
    dev_passes = [{k: v.to(dev) for k, v in p.items()} for p in passes]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)       # > 126 MB L2
    acc = torch.zeros_like(vp.bucket.flat) if n_pass > 1 else None
    if n_pass > 1:
        vp.gather_grads = True          # the passes' gradients are accumulated through the flat bucket
    # Where the step's gradients are summed over the ranks (parallel.py): inside the backward at the scene tensors (GradSumPoint:
    # vertices, opacities, decimated texture cells -- one small all-reduce per pass, no leaf all-reduce), else at the leaves
    # (one all-reduce of the parameter-gradient bucket per step)
    inside = vp.reduces_inside_backward(dev_passes[0])

    def step_eager(collective=True):
        for i, p in enumerate(dev_passes):
            losses = vp.forward_backward(p, None, already_sharded=True, n_total_views=B, all_reduce=collective and inside)
            if acc is not None:
                acc.copy_(vp.bucket.flat) if i == 0 else acc.add_(vp.bucket.flat)
        if acc is not None:
            vp.bucket.flat.copy_(acc)
        if collective and not inside:
            vp.bucket.all_reduce(vp.group)
        return losses

    graphed = piped = None
    nocoll = None
    if not args.no_graph:
        # the peer-memory all-reduce is captured inside the graph when the step is a single pass (it then cannot be skipped:
        # a second graph without it serves the "what does the collective add" measurement)
        in_graph = vp.graph_capturable_collective and (n_pass == 1 or inside)
        piped = PipelinedGraphedStep(vp, dev_passes[0], B, capture_all_reduce=in_graph)
        graphed = piped.steps[0]
        nocoll = GraphedStep(vp, dev_passes[0], B, capture_all_reduce=False) if (in_graph and world > 1) else graphed

    def step_resident(collective=True):
        if graphed is None:
            return step_eager(collective)
        g = graphed if collective else nocoll
        for i, p in enumerate(dev_passes):
            losses = g.run(p if n_pass > 1 else None, all_reduce=False)      # a collective captured in the graph runs regardless
            if acc is not None:
                acc.copy_(vp.bucket.flat) if i == 0 else acc.add_(vp.bucket.flat)
        if acc is not None:
            vp.bucket.flat.copy_(acc)
        if collective and not g.capture_all_reduce and not inside:
            vp.bucket.all_reduce(vp.group)
        return losses

    def step_e2e():
        """the public API with HOST buffers: every pass's inputs are copied H2D from pinned memory (the next pass's while
        this one computes: double-buffered), and the step's loss is read back"""
        loss = 0.0
        if piped is None:
            for i, p in enumerate(passes):
                inp = {k: v.to(dev, non_blocking=True) for k, v in p.items()}
                losses = vp.forward_backward(inp, None, already_sharded=True, n_total_views=B, all_reduce=inside)
                if acc is not None:
                    acc.copy_(vp.bucket.flat) if i == 0 else acc.add_(vp.bucket.flat)
                loss = loss + losses['rgb']
        else:
            for i, p in enumerate(passes):
                losses = piped.run(p, passes[(i + 1) % n_pass], all_reduce=False)
                if acc is not None:
                    acc.copy_(vp.bucket.flat) if i == 0 else acc.add_(vp.bucket.flat)
                loss = loss + losses['rgb']
        if acc is not None:
            vp.bucket.flat.copy_(acc)
        if not inside and (piped is None or not piped.steps[0].capture_all_reduce):
            vp.bucket.all_reduce(vp.group)
        return float(loss.item())                                                 # D2H read of the step's result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def timed(fn, steps):
        evs = []
        barrier()
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last['losses'] = fn()
            b.record()
            evs.append((a, b))
        barrier()
        return sum(a.elapsed_time(b) for a, b in evs)

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_resident()
    barrier()

    # ---- device-resident timing: per-step CUDA event pairs, L2 flushed between steps (outside the pairs)
    launches0 = _lib.launch_count()
    step_eager()
    launches_per_step = _lib.launch_count() - launches0      # our kernels per step (a graph replays exactly these)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    try:
        ms_local = timed(step_resident, args.steps)
    finally:
        clocks = sampler.summary() if sampler else None          # stops the sampling process
    if args.dump_outputs and rank == 0:
        # a step of several passes keeps only its last pass's loss terms (its gradients are the sum over the passes)
        dump_outputs(args.dump_outputs, model, last['losses'], '' if n_pass == 1 else '_last_pass')
    # the same steps without the gradient collective: what the all-reduce adds to a step when it is exposed
    ms_nocoll_local = timed(lambda: step_resident(False), args.steps) if world > 1 else ms_local

    # ---- per-kernel durations (roofline): the same steps run eagerly with CUDA events around the raster kernels on their
    # launch stream (events cannot be read back from inside a replayed graph; kernel durations do not depend on how
    # the launch was submitted)
    _lib.lib().dbw_timing_reset()
    _lib.lib().dbw_timing_enable(1)
    overlap, fused_loss.OVERLAP_BACKWARD_PASSES = fused_loss.OVERLAP_BACKWARD_PASSES, False      # one kernel at a time here
    for _ in range(args.steps):
        flush.zero_()
        step_eager(False)
    barrier()
    fused_loss.OVERLAP_BACKWARD_PASSES = overlap
    _lib.lib().dbw_timing_enable(0)
    kt = {(kind, kk): _lib.kernel_time_ms(kind, kk) for kind in (0, 1) for kk in (1, K)}
    _lib.lib().dbw_timing_reset()

    # ---- end-to-end timing through the public API with host buffers
    for _ in range(2):
        step_e2e()
    ms_e2e_local = timed(step_e2e, args.steps)

    comm_err = vp.bucket.peer.error() if vp.bucket.peer is not None else 0        # a barrier of the peer all-reduce timed out?
    t = torch.tensor([ms_local, ms_e2e_local, ms_nocoll_local, float(comm_err)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e_total, ms_nocoll_total, comm_err = t.tolist()
    if comm_err:
        raise RuntimeError(f'the peer-memory all-reduce reported a barrier time-out (code {int(comm_err)}): the timed steps are invalid; '
                           f're-run with --collective nccl')

    if rank == 0:
        ms_per_step = ms_total / args.steps
        value = B * args.steps / (ms_total / 1e3)
        e2e_value = B * args.steps / (ms_e2e_total / 1e3)
        peak, peak_src = peaks()
        names = {(0, 1): 'raster_forward[env K=1]', (0, K): f'raster_forward[blocks K={K}]',
                 (1, 1): 'raster_backward[env K=1]', (1, K): f'raster_backward[blocks K={K}]'}
        per_step = {names[k]: kt[k][0] / args.steps for k in kt}

        def roofline(key):
            """SURVEY 8d: each direction of a pass moves H*W*(16 + 4K) algorithmic bytes per view (RGBA + K ids); this rank's
            launches of one step cover local_px pixels"""
            ms = kt[key][0] / args.steps                       # all launches of this kernel in one step (one per pass)
            alg = local_px * (16 + 4 * key[1])
            traffic, src = ncu_traffic(names[key], args.workload, world)
            return {'bound': 'hbm', 'kernel': names[key], 'achieved': alg / (ms / 1e3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                    'frac': alg / (ms / 1e3) / 1e9 / peak, 'traffic': traffic, 'traffic_source': src, 'peak_source': peak_src,
                    'algorithmic_bytes_per_step': alg, 'kernel_ms_per_step': ms, 'launches_per_step': kt[key][1] / args.steps}

        dom = max(kt, key=lambda k: kt[k][0])                  # the raster kernel with the largest summed duration
        raster_ms = sum(per_step.values())
        h2d = sum(v.numel() * v.element_size() for p in passes for v in p.values())
        line = {
            'metric': metric_name(w), 'value': value, 'unit': 'views/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': warm, 'ms_per_step': ms_per_step,
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'{args.workload}: {w["what"]}; BASELINE {w["baseline"]}; coarse phase (sigma=1e-4, per-block '
                                   f'opacities + noise, 8x decimated textures); the step\'s {B} views are split over the ranks at '
                                   f'(view, 16-row band) granularity, gradients summed over the ranks '
                                   + ('inside the backward at the scene tensors (vertices, opacities, decimated texture cells: '
                                      f'{model.grad_sum_floats() * 4 / 1e6:.2f} MB) ' if inside else
                                      f'at the leaves ({vp.bucket.nbytes / 1e6:.1f} MB bucket) ')
                                   + f'by one all-reduce ({vp.collective_name})',
                       'views_per_step': B, 'views_per_pass_per_rank': views_per_pass, 'passes_per_step': n_pass,
                       'l2': 'flushed (256 MB memset) between steps, outside the per-step event pairs',
                       'loss': 'rgb (MSE) only; LPIPS excluded (SURVEY 8d)', 'seed': SEED,
                       'submission': 'eager' if graphed is None else 'each pass captured once in a CUDA graph and replayed',
                       'backward_passes': 'concurrent (two graph branches)' if fused_loss.OVERLAP_BACKWARD_PASSES else 'back to back',
                       'e2e_pipeline': 'none' if piped is None else 'inputs of the next pass copied H2D on a side stream during this pass (double-buffered)'},
            'e2e': {'value': e2e_value, 'unit': 'views/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4},
            'gpu_launches': launches_per_step * args.steps,
            'clocks': clocks,
            'roofline': dict(roofline(dom), kernels_ms_per_step=per_step),
            'roofline_backward': roofline((1, K)),
            'breakdown_ms_per_step': {'step': ms_per_step, 'raster_kernels_rank0': raster_ms,
                                      'other_kernels_and_launch_gaps': ms_nocoll_total / args.steps - raster_ms,
                                      'exposed_collective': (ms_total - ms_nocoll_total) / args.steps},
            'note': 'PyTorch3D-CUDA (the north star\'s comparator) is not installable here: unmeasured',
        }
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline(args.workload)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ CPU legs (oracle port)
def sample_views(n_views, n):
    """n view indices spread evenly over the ring: the CPU legs render a subset of the very views the GPU arm renders"""
    return [int(round(i * n_views / n)) % n_views for i in range(n)]


def oracle_step(workload, views):
    """One render+backward pass of the reference's algorithm (oracle port) over the given views of the workload."""
    from oracle import dbw_path as D
    w = WORKLOADS[workload]
    H, W, K = w['height'], w['width'], w['faces_per_pixel']
    tpl = D.SceneTemplate(n_blocks=w['n_blocks'], txt_size=w['txt_size'], txt_bkg_upscale=w['txt_bkg_upscale'])
    p = {k: v.requires_grad_(True) for k, v in D.init_params(w['n_blocks'], w['txt_size'], w['txt_bkg_upscale'], seed=SEED).items()}
    R, T, Km = D.ring_cameras(w['n_views'])
    g = torch.Generator().manual_seed(SEED)
    imgs = torch.rand(len(views), 3, H, W, generator=g)
    keep = torch.sigmoid(p['alpha_logit'].detach()) > 0.01
    t0 = time.perf_counter()
    rec = D.predict(tpl, p, R[views], T[views], Km, (H, W), sigma=1e-4, faces_per_pixel=K, z_clip=0.001, keep=keep, decimate=8)
    loss = D.mse_loss(imgs, rec)
    loss.backward()
    return time.perf_counter() - t0


def cpu_threads():
    """threads for the CPU legs: all host cores up to 32 (beyond that the small torch ops of the path get slower, not
    faster; measured on the 128-core GPU box)"""
    return min(os.cpu_count(), 32)


def cpu_baseline(workload, n_views=None):
    w = WORKLOADS[workload]
    # about 10-30 s of host work: 16 views of the DTU shape, scaled by pixels and faces
    n_views = n_views or max(1, int(16 * 160000 / (w['height'] * w['width']) * min(1.0, 10 / w['n_blocks'])))
    views = sample_views(w['n_views'], n_views)
    torch.set_num_threads(cpu_threads())
    oracle_step(workload, views[:1])                  # warm-up (page in the library, thread pools)
    dt = oracle_step(workload, views)
    return {'value': n_views / dt, 'unit': 'views/s', 'cores': cpu_threads(), 'kind': 'port', 'views_sampled': views,
            'sample': f'{n_views} of the {w["n_views"]} views ({w["height"]}x{w["width"]}, {w["n_blocks"]} blocks, K={w["faces_per_pixel"]}), '
                      f'forward+backward once, OpenMP rasterizer + torch ops on {cpu_threads()} of {os.cpu_count()} host threads; {dt:.1f} s'}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    torch.set_num_threads(cpu_threads())
    n = 2
    views = sample_views(w['n_views'], n)
    for _ in range(min(args.warmup, 1)):
        oracle_step(args.workload, views[:1])
    tot = 0.0
    for _ in range(args.steps):
        tot += oracle_step(args.workload, views)
    value = n * args.steps / tot
    sample = f'{n} of the {w["n_views"]} views per step ({w["height"]}x{w["width"]}, {w["n_blocks"]} blocks, K={w["faces_per_pixel"]}), forward+backward'
    print(json.dumps({
        'impl': 'reference', 'metric': metric_name(w), 'value': value, 'unit': 'views/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': min(args.warmup, 1), 'ms_per_step': tot / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{args.workload}: {w["what"]} (same scene, cameras and seed as our arm); bounded sample: ' + sample,
                   'views_per_step': w['n_views'], 'views_sampled': views, 'seed': SEED},
        'cpu_baseline': {'value': value, 'unit': 'views/s', 'cores': cpu_threads(), 'kind': 'port', 'sample': sample, 'views_sampled': views},
        'e2e': {'value': value, 'unit': 'views/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'note': 'PyTorch3D (the reference dependency that owns this arithmetic) is not installable here, so PyTorch3D-CUDA and '
                'PyTorch3D-CPU are both UNMEASURED; this arm times the CPU restatement of its algorithm (oracle/, "port") on the host cores',
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None,
                    help='timed steps (default: 100 on dtu, 10 on the larger workloads, 5 with --impl reference)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='dtu', choices=sorted(WORKLOADS))
    ap.add_argument('--collective', default='auto', choices=['auto', 'nccl', 'p2p'],
                    help='gradient all-reduce: hand-written NVLink peer-memory kernel (p2p), NCCL, or p2p when it initialises (auto)')
    ap.add_argument('--overlap-bwd', default='auto', choices=['auto', 'on', 'off'],
                    help="run the two passes' backward kernels concurrently (fused_loss.OVERLAP_BACKWARD_PASSES); auto: when the "
                         'step is split over 4 or more GPUs (short launches whose tails then overlap)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='submit the step eagerly instead of replaying a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="write the last timed step's loss terms and leaf gradients as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps is None:
        # the larger workloads take 10-100x longer per step, and a reference step is a bounded CPU sample: keep the
        # default run within minutes
        args.steps = 5 if args.impl == 'reference' else 100 if args.workload == 'dtu' else 10
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        if args.dump_outputs:
            ap.error('--dump-outputs applies to our arm')
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
