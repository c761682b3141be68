#!/usr/bin/env python
"""
bench.py -- megapixels/second through pipe_color2d_slic_features_model_graphcut (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's (segm, segm_soft) to DIR/*.npy

Workload (BASELINE.json configs[1], SURVEY.md section 8d "config 2"): one synthetic 2048x2048 RGB float64 image per
GPU per step -- Voronoi regions with 3 class means + gaussian noise, sp_size 29 (4 987 seeds), colour-mean descriptors,
3-class GMM, GraphCut with gc_regul 1 / 'model' edges.  A "step" is one pass of the whole path over that image.
N > 1 shards independent images over ranks (one process per GPU, weak scaling, no data-path collective).

  value : MPix/s with the image already resident in HBM and results left in HBM (device-resident)
  e2e   : MPix/s through the public numpy API -- pinned host image in, (segm, segm_soft) host arrays out
Timed with CUDA events on the launching stream between barrier + synchronize, max over ranks.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 2048
SP_SIZE, SP_REGUL, NB_CLASSES, GC_REGUL = 29, 0.2, 3, 1.0
FEATURES = {'color': ['mean']}
METRIC = 'megapixels/sec end-to-end SLIC+features+GC (pipe_color2d_slic_features_model_graphcut)'
WORKLOAD = 'config2: 2048x2048 RGB f64 synthetic, SLIC sp_size=29 (~5k superpixels) + colour-mean + 3-class GMM + GraphCut'
#: algorithmic bytes per pixel per sweep of the dominant kernel (slic_assign) as SURVEY.md section 8(d) counts them: image held
#: as f32 (12 B) + label i32 (4 B).  The kernel itself keeps Lab in f64 planes (the k-means is defined in float64), so the
#: bytes it has to move are 24 + 4 = 28 per pixel; both figures are reported.
ASSIGN_BYTES_PER_PX = 16
ASSIGN_LAYOUT_BYTES_PER_PX = 28
#: SURVEY.md section 8(d) per-pixel figures of the other bandwidth-bound stages: whole SLIC (pre-pass 24 + 10 sweeps x 16 +
#: connectivity 16), fused segment statistics, adjacency extraction, final gathers (reference emits segm_soft as f64)
STAGE_BYTES_PER_PX = {'slic (all stages)': 200, 'segment_stats': 16, 'adjacency': 4, 'gather': 4 + 4 + 8 * NB_CLASSES}
SLIC_STAGES = ('slic_prepare', 'slic_assign', 'slic_update', 'slic_finalize', 'slic_connectivity')


def headline_config(n_gpus):
    """the `config` object of the headline line -- identical for both arms (the driver compares them)"""
    return {'workload': WORKLOAD, 'images_per_step_per_gpu': 1, 'sp_size': SP_SIZE, 'sp_regul': SP_REGUL,
            'nb_classes': NB_CLASSES, 'gc_regul': GC_REGUL, 'features': 'color mean', 'class_model': 'StandardScaler + full-covariance GMM (n_init 9, max_iter 99)',
            'parallelism': 'independent images sharded over %d GPU(s) / host processes' % n_gpus,
            'l2': 'no explicit flush: per-step working set (f64 image 100 MB + Lab 100 MB + soft output 100 MB) exceeds the 126 MB L2'}


def probe_reference_libs():
    """BASELINE.md section 3.1: can the real third-party engines of the reference be imported on this box?"""
    out = {}
    for name in ('skimage', 'gco'):
        try:
            mod = __import__(name)
            out[name] = getattr(mod, '__version__', 'present')
        except Exception as exc:  # noqa: BLE001 -- any failure means "not usable here"
            out[name] = 'unavailable (%s)' % type(exc).__name__
    return out


def synth_image(seed, h=H, w=W, n_classes=NB_CLASSES, cell=64):
    rng = np.random.RandomState(seed)
    pts = rng.rand(40, 2) * [h, w]
    cls = rng.randint(0, n_classes, 40)
    gy, gx = np.mgrid[:(h + cell - 1) // cell, :(w + cell - 1) // cell] * cell + cell / 2
    near = ((gy[..., None] - pts[:, 0]) ** 2 + (gx[..., None] - pts[:, 1]) ** 2).argmin(-1)
    cl = np.kron(cls[near], np.ones((cell, cell), dtype=int))[:h, :w]
    means = np.linspace(0.2, 0.8, n_classes)
    img = means[cl][..., None] + np.array([0.0, 0.03, -0.03])
    return np.clip(img + rng.normal(0, 0.05, img.shape), 0, 1)


def synth_texture_image(seed, h=H, w=W, n_classes=4, cell=64):
    """config-3 style image (SURVEY.md section 8d): Voronoi regions of 4 classes, each class with its own mean and a sinusoidal
    texture of period 4 / 8 / 16 / 32 px in a random orientation, gaussian noise"""
    rng = np.random.RandomState(seed)
    pts = rng.rand(40, 2) * [h, w]
    cls = rng.randint(0, n_classes, 40)
    gy, gx = np.mgrid[:(h + cell - 1) // cell, :(w + cell - 1) // cell] * cell + cell / 2
    near = ((gy[..., None] - pts[:, 0]) ** 2 + (gx[..., None] - pts[:, 1]) ** 2).argmin(-1)
    cl = np.kron(cls[near], np.ones((cell, cell), dtype=int))[:h, :w]
    yy, xx = np.mgrid[:h, :w].astype(np.float64)
    img = np.zeros((h, w))
    means = np.linspace(0.3, 0.7, n_classes)
    for c in range(n_classes):
        ang = rng.rand() * np.pi
        period = 4.0 * 2 ** c
        wave = 0.12 * np.sin(2 * np.pi * (np.cos(ang) * xx + np.sin(ang) * yy) / period)
        img = np.where(cl == c, means[c] + wave, img)
    img = img[..., None] + np.array([0.0, 0.03, -0.03])
    return np.clip(img + rng.normal(0, 0.03, img.shape), 0, 1)


def synth_eggs_image(seed, h=640, w=1024, n_eggs=6):
    """config-4 style image (SURVEY.md section 8d; the reference's drosophila ovary slices are 1024 x 647): elliptic 'eggs' of random
    size and orientation, brighter than a noisy background.  Returns (image [H, W, 3], annotation [H, W] with egg i as label i + 1,
    centres)"""
    rng = np.random.RandomState(seed)
    yy, xx = np.mgrid[:h, :w].astype(np.float64)
    annot = np.zeros((h, w), dtype=int)
    centres = []
    cols = np.linspace(0, w, n_eggs // 2 + 2)[1:-1]
    for i in range(n_eggs):
        cy = h * (0.3 if i % 2 == 0 else 0.72) + rng.uniform(-0.04, 0.04) * h
        cx = cols[i // 2] + rng.uniform(-0.03, 0.03) * w
        a, b = rng.uniform(0.10, 0.13) * w * 0.8, rng.uniform(0.14, 0.19) * h * 0.8
        ang = rng.uniform(0, np.pi)
        u = (xx - cx) * np.cos(ang) + (yy - cy) * np.sin(ang)
        v = -(xx - cx) * np.sin(ang) + (yy - cy) * np.cos(ang)
        inside = (u / a) ** 2 + (v / b) ** 2 <= 1.0
        annot[inside & (annot == 0)] = i + 1
        centres.append((int(round(cy)), int(round(cx))))
    img = np.where(annot > 0, 0.7, 0.25)[..., None] + np.array([0.0, 0.03, -0.03])
    return np.clip(img + rng.normal(0, 0.06, img.shape), 0, 1), annot, centres


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def load_tensor_peak():
    """(dense bf16 TFLOP/s, source) -- the tensor-core denominator: MEASURED_PEAKS.json's burst figure, else the profiling guide's"""
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        if 'bf16_tflops' in p:
            return float(p['bf16_tflops']), 'measured (MEASURED_PEAKS.json bf16_tflops, burst)'
    return 1590.0, 'fallback (B200_PROFILING.md 1.59 PFLOP/s)'


TRAFFIC_SOURCE = 'profiles/r02c_assign_traffic.json'


def load_traffic():
    """DRAM bytes per k_assign launch from the committed `ncu --set full` capture (profiles/), or None"""
    path = os.path.join(ROOT, TRAFFIC_SOURCE)
    try:
        with open(path) as f:
            return int(json.load(f)['traffic_bytes_per_launch'])
    except (OSError, KeyError, ValueError):
        return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region"""
    QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm)}


#: pixels of segm_soft that --dump-outputs writes: the whole [H, W, K] float64 array is 100 MB, the sample 25 MB
DUMP_SOFT_PIXELS = 1 << 20


def dump_outputs(out_dir, segm, soft):
    """what the headline path returns, for comparing two builds output for output: the label map whole (float32 holds every label
    exactly) and a fixed, seeded sample of segm_soft's pixels (float64) with their flat pixel indices"""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.RandomState(0).choice(segm.size, DUMP_SOFT_PIXELS, replace=False))
    np.save(os.path.join(out_dir, 'segm.npy'), segm.astype(np.float32))
    np.save(os.path.join(out_dir, 'segm_soft_sample.npy'), soft.reshape(segm.size, -1)[idx].astype(np.float64))
    np.save(os.path.join(out_dir, 'segm_soft_sample_index.npy'), idx.astype(np.float64))


def dist_env():
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    return rank, world, local


# ---------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU path (oracle port; scikit-image and gco are not installable here) on host cores
# ---------------------------------------------------------------------------------------------------------------------

#: images of the bounded sample, generated ONCE in the parent before the pool forks (workers inherit them copy-on-write):
#: image synthesis is not part of the path and is not timed
_REF_IMAGES = []


def _oracle_path(img):
    """the path itself, host ndarray in -> (segm, segm_soft) out; returns (seconds inside the path, checksum)"""
    import oracle
    from sklearn import mixture, pipeline, preprocessing
    t0 = time.perf_counter()
    slic, fts = oracle.compute_color2d_superpixels_features(img, ('mean',), SP_SIZE, SP_REGUL)
    nb_inits = max(1, int(np.sqrt(99)))
    model = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()),
                               ('model', mixture.GaussianMixture(NB_CLASSES, covariance_type='full', n_init=nb_inits, max_iter=99))])
    model.fit(fts)
    proba = model.predict_proba(fts)
    labels = oracle.segment_graph_cut_general(slic, proba, GC_REGUL, 'model')
    segm, soft = labels[slic], proba[slic]
    return time.perf_counter() - t0, int(segm.sum() % 7) + int(soft.shape[2])


def _ref_worker_init():
    """once per worker process, outside every timed region: imports, one BLAS thread, one small pass to warm the code paths"""
    import oracle  # noqa: F401
    import sklearn.mixture  # noqa: F401
    try:  # one BLAS/OpenMP thread per worker process: the pool already uses the cores (no oversubscription)
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except ImportError:
        pass
    _oracle_path(synth_image(7, 160, 160))


def _oracle_one(idx):
    return _oracle_path(_REF_IMAGES[idx])


class ReferencePool(object):
    """the reference's own idiom for many images: a process pool over images (imsegm/utilities/experiments.py:354-410).
    ONE pool for the whole run, workers warmed before the first timed step, images pre-generated."""

    def __init__(self, n_images, workers, first_seed=1000):
        import multiprocessing as mp
        del _REF_IMAGES[:]
        _REF_IMAGES.extend(synth_image(first_seed + i) for i in range(n_images))
        self.n, self.workers = n_images, workers
        if workers > 1:
            self.pool = mp.get_context('fork').Pool(workers, initializer=_ref_worker_init)
            self.pool.map(_noop, range(4 * workers))   # every worker has finished its initializer before anything is timed
        else:
            self.pool = None
            _ref_worker_init()

    def step(self):
        """one bounded sample: every image once.  Returns (wall seconds of the map alone, [seconds inside the path per image])"""
        t0 = time.perf_counter()
        res = self.pool.map(_oracle_one, range(self.n), chunksize=1) if self.pool else [_oracle_one(i) for i in range(self.n)]
        return time.perf_counter() - t0, [r[0] for r in res]

    def close(self):
        if self.pool:
            self.pool.close()
            self.pool.join()


def _noop(_):
    time.sleep(0.05)
    return 0


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # the reference's own rule is NB_WORKERS = 0.6 * cpu_count (pipelines.py:43); on the 128-CPU host of the B200 box the path
    # stops scaling at ~16 processes (measured r01: 1 -> 0.86, 8 -> 7.9, 16 -> 12.0, 32 -> 10.1, 64 -> 6.8 MPix/s; memory bound),
    # so 16 workers is the reference's best case and keeps a step at a few seconds
    workers = args.ref_workers or min(16, max(1, int(0.6 * cores)))
    n_img = workers  # one bounded sample per step: `workers` images through the process pool
    pool = ReferencePool(n_img, workers)
    for _ in range(args.warmup):
        pool.step()
    wall, inner = 0.0, []
    for _ in range(args.steps):
        dt, ins = pool.step()
        wall += dt
        inner += ins
    pool.close()
    value = args.steps * n_img * H * W / 1e6 / wall
    sample = ('%d step(s) x %d pre-generated images of 2048x2048 through ONE warmed %d-process pool (reference idiom: Pool over '
              'images); timed: the pool.map of the path only' % (args.steps, n_img, workers))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'MPix/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': wall / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': headline_config(args.gpus),
        'cpu_baseline': {'value': value, 'unit': 'MPix/s', 'cores': workers, 'kind': 'port', 'sample': sample, 'host_cpus': cores,
                         'note': 'CPU restatement of the reference path (oracle/): scikit-image and gco cannot be installed here',
                         'path_seconds_per_image_mean': float(np.mean(inner)), 'path_seconds_per_image_max': float(np.max(inner)),
                         'ideal_ms_per_step': float(np.sum(inner)) / workers / args.steps * 1e3},
        'e2e': {'value': value, 'unit': 'MPix/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'reference_libs': probe_reference_libs(),
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback)'
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from pyimsegm_b200 import _lib, pipelines
    lib = _lib.lib()

    img = synth_image(2 + rank)
    host_img = torch.from_numpy(img).pin_memory()      # pinned host memory (e2e source)
    host_np = host_img.numpy()
    dev_img = host_img.cuda(non_blocking=True)          # resident copy for the device-timed leg
    torch.cuda.synchronize()

    def step_resident():
        # the default 'GMM' class model is fitted on the device (isb_gmm_fit_predict): no host round trip at all
        return pipelines.segment_resident(dev_img, ('fit', NB_CLASSES, True, 99), FEATURES, SP_SIZE, SP_REGUL, GC_REGUL, 'model')

    def step_e2e():
        return pipelines.pipe_color2d_slic_features_model_graphcut(host_np, NB_CLASSES, FEATURES, sp_size=SP_SIZE, sp_regul=SP_REGUL,
                                                                   gc_regul=GC_REGUL, gc_edge_type='model')

    page_np = np.array(img)   # an ordinary (pageable) array: what a caller of the reference API holds

    def step_page():
        return pipelines.pipe_color2d_slic_features_model_graphcut(page_np, NB_CLASSES, FEATURES, sp_size=SP_SIZE, sp_regul=SP_REGUL,
                                                                   gc_regul=GC_REGUL, gc_edge_type='model')

    def step_batch(n):
        return pipelines.segment_images_batch([host_np] * n, NB_CLASSES, FEATURES, sp_size=SP_SIZE, sp_regul=SP_REGUL, gc_regul=GC_REGUL)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            out = fn()
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device='cuda', dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    keep = None
    for _ in range(max(args.warmup, 3)):
        step_resident()
        keep = step_e2e()   # held across the next call, like `out = fn()` in the timed loop: warms BOTH sets of pinned result buffers
    del keep

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # timed region 1 (the `value`): the device part replayed as one CUDA graph per image (pipelines._run_resident_graph)
    n0 = lib.isb_launch_count()
    ms_res, (d_segm, d_soft) = timed(step_resident, args.steps)
    launches = lib.isb_launch_count() - n0
    # copied now: the passes below refill the same engine buffers
    outputs = (d_segm.cpu().numpy(), d_soft.cpu().numpy()) if args.dump_outputs and rank == 0 else None
    # timed region 2 (same steps, eager launches): per-stage CUDA events on the launching stream -> `stages` and the roofline
    pipelines.USE_CUDA_GRAPHS = False
    step_resident()
    lib.isb_profile_enable(1)
    ms_eager, _ = timed(step_resident, args.steps)
    nstage = lib.isb_profile_stage_count()
    ms_arr, cnt_arr = (C.c_double * nstage)(), (C.c_longlong * nstage)()
    lib.isb_profile_collect(ms_arr, cnt_arr)
    lib.isb_profile_enable(0)
    pipelines.USE_CUDA_GRAPHS = True
    ms_e2e, (segm, soft) = timed(step_e2e, args.steps)
    step_page()
    ms_page, _ = timed(step_page, args.steps)
    # extra (not the headline): a batch of images through the pipelined batch API -- upload / kernels / download of consecutive
    # images overlap on three streams (what the reference's process pool over images becomes on a GPU)
    nbatch = 8

    def batch_once():
        res = step_batch(nbatch)
        del res      # the pinned result buffers go back to torch's host cache before the next call needs them
        return None

    batch_once()
    ms_batch, _ = timed(batch_once, args.steps)
    clocks = sampler.stop() if rank == 0 else None

    stages = {lib.isb_profile_stage_name(i).decode(): {'ms_per_step': ms_arr[i] / args.steps, 'launches_per_step': cnt_arr[i] / args.steps}
              for i in range(nstage)}
    mpix = H * W / 1e6
    value = world * args.steps * mpix / (ms_res / 1e3)
    e2e = world * args.steps * mpix / (ms_e2e / 1e3)
    peak, peak_src = load_peaks()
    a = stages['slic_assign']
    t_assign = a['ms_per_step'] / max(a['launches_per_step'], 1) / 1e3
    achieved = ASSIGN_BYTES_PER_PX * H * W / t_assign / 1e9 if t_assign > 0 else 0.0
    achieved_layout = ASSIGN_LAYOUT_BYTES_PER_PX * H * W / t_assign / 1e9 if t_assign > 0 else 0.0
    # the other bandwidth-bound stages against the same peak, with SURVEY.md section 8(d)'s bytes per pixel
    t_slic = sum(stages[k]['ms_per_step'] for k in stages if k.startswith('slic_')) / 1e3
    stage_roofline = {}
    for name, bpp in STAGE_BYTES_PER_PX.items():
        t = t_slic if name.startswith('slic') else stages[name]['ms_per_step'] / 1e3
        if t > 0:
            gbs = bpp * H * W / t / 1e9
            stage_roofline[name] = {'bytes_per_px': bpp, 'ms_per_step': t * 1e3, 'achieved_gbs': gbs, 'frac': gbs / peak}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        'metric': METRIC, 'value': value, 'unit': 'MPix/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms_res / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': headline_config(world),
        'e2e': {'value': e2e, 'unit': 'MPix/s', 'ms_per_step': ms_e2e / args.steps, 'h2d_bytes_per_step': int(host_np.nbytes),
                'd2h_bytes_per_step': int(segm.nbytes + soft.nbytes), 'source': 'pinned host ndarray'},
        'e2e_pageable': {'value': world * args.steps * mpix / (ms_page / 1e3), 'unit': 'MPix/s', 'ms_per_step': ms_page / args.steps,
                         'source': 'ordinary (pageable) numpy array, as a caller of the reference API would pass it'},
        'e2e_batch': {'value': world * args.steps * nbatch * mpix / (ms_batch / 1e3), 'unit': 'MPix/s', 'images_per_call': nbatch,
                      'note': 'segment_images_batch: same host-in/host-out path, copies of consecutive images overlapped on 3 streams'},
        'gpu_launches': int(launches),
        'roofline': {'kernel': 'k_assign (slic_assign)', 'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                     'frac': achieved / peak, 'traffic': load_traffic(), 'traffic_source': TRAFFIC_SOURCE, 'peak_source': peak_src,
                     'algorithmic_bytes_per_launch': ASSIGN_BYTES_PER_PX * H * W, 'launch_ms': t_assign * 1e3,
                     'bytes_per_px': '16 = SURVEY.md section 8(d) (f32 image 12 + label 4)',
                     'f64_layout': {'bytes_per_px': ASSIGN_LAYOUT_BYTES_PER_PX, 'achieved': achieved_layout, 'frac': achieved_layout / peak,
                                    'note': 'bytes the kernel must move: Lab is held in f64 planes because the k-means is defined in float64'},
                     'stages': stage_roofline},
        'stages': stages,
        'stages_note': 'second timed pass of the same steps with eager launches (%.3f ms per step); `value` replays the same kernels as one CUDA '
                       'graph per image' % (ms_eager / args.steps),
        'clocks': clocks,
        'reference_libs': probe_reference_libs(),
    }
    if world == 1 and not args.no_cpu_baseline:
        pool = ReferencePool(args.cpu_images, 1)
        dt, inner = pool.step()
        v = args.cpu_images * H * W / 1e6 / dt
        line['cpu_baseline'] = {'value': v, 'unit': 'MPix/s', 'cores': 1, 'kind': 'port',
                                'sample': '%d pre-generated image(s) of 2048x2048, single thread (the reference is single-threaded per '
                                          'image), %.1f s inside the path' % (args.cpu_images, dt),
                                'host_cpus': os.cpu_count()}
        # the CPU leg doubles as the parity gate of SURVEY.md section 8(d): the first sample image through both paths
        import oracle
        img0 = _REF_IMAGES[0]
        o_slic, o_fts = oracle.compute_color2d_superpixels_features(img0, ('mean',), SP_SIZE, SP_REGUL)
        d_slic, d_fts = pipelines.compute_color2d_superpixels_features(img0, FEATURES, sp_size=SP_SIZE, sp_regul=SP_REGUL)
        same = bool(np.array_equal(o_slic, d_slic))
        line['parity'] = {'image': 'synth_image(1000), 2048x2048', 'superpixel_label_map_identical': same,
                          'nb_superpixels': int(d_slic.max()) + 1,
                          'features_max_abs_err': float(np.max(np.abs(o_fts - d_fts))) if same and o_fts.shape == d_fts.shape else None}
    if outputs is not None:
        dump_outputs(args.dump_outputs, *outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_tiled(args):
    """extra workload (not the headline line): BASELINE config 5 -- ONE 8192x8192 image banded over the GPUs (strong scaling).
    Host image in, every rank's rows of (segm, segm_soft) out; the time is the max over ranks."""
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback)'
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from pyimsegm_b200 import _lib, pipelines, tiled
    lib = _lib.lib()
    side = args.tiled_side
    host_img = torch.from_numpy(synth_image(5, side, side)).pin_memory()
    host_np = host_img.numpy()
    comm = tiled.default_comm()

    def step():
        return tiled.pipe_color2d_slic_features_model_graphcut_tiled(host_np, NB_CLASSES, FEATURES, sp_size=SP_SIZE, sp_regul=SP_REGUL,
                                                                     gc_regul=GC_REGUL, gc_edge_type='model', comm=comm)

    def whole():
        return pipelines.pipe_color2d_slic_features_model_graphcut(host_np, NB_CLASSES, FEATURES, sp_size=SP_SIZE, sp_regul=SP_REGUL,
                                                                   gc_regul=GC_REGUL, gc_edge_type='model')

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(steps):
            out = fn()
        ev1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device='cuda', dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    keep = None
    for _ in range(max(args.warmup, 3)):
        keep = step()
    del keep
    lib.isb_profile_enable(1)
    n0 = lib.isb_launch_count()
    ms, (segm, soft, (lo, hi)) = timed(step, args.steps)
    launches = lib.isb_launch_count() - n0
    nstage = lib.isb_profile_stage_count()
    ms_arr, cnt_arr = (C.c_double * nstage)(), (C.c_longlong * nstage)()
    lib.isb_profile_collect(ms_arr, cnt_arr)
    lib.isb_profile_enable(0)
    stages = {lib.isb_profile_stage_name(i).decode(): {'ms_per_step': ms_arr[i] / args.steps, 'launches_per_step': cnt_arr[i] / args.steps}
              for i in range(nstage)}
    mono = None
    if world == 1:
        del segm, soft
        for _ in range(2):
            keep = whole()
        del keep
        ms_w, _ = timed(whole, args.steps)
        mono = {'value': args.steps * side * side / 1e6 / (ms_w / 1e3), 'unit': 'MPix/s', 'ms_per_step': ms_w / args.steps,
                'note': 'the same image through the single-GPU API (pipe_color2d_slic_features_model_graphcut)'}
    if rank == 0:
        value = args.steps * side * side / 1e6 / (ms / 1e3)
        line = {'metric': METRIC, 'value': value, 'unit': 'MPix/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
                'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64',
                'data': 'synthetic',
                'config': {'workload': 'config5: ONE %dx%d RGB f64 synthetic image banded over %d GPU(s), sp_size=29, colour-mean, '
                                       '3-class GMM + GraphCut' % (side, side, world),
                           'parallelism': 'row bands; per sweep one all_reduce of 6 int64 per cluster; label map broadcast; graph cut replicated',
                           'timed': 'host image in (pinned), the rank\'s rows of segm + segm_soft out (end to end; there is no resident variant)'},
                'e2e': {'value': value, 'unit': 'MPix/s', 'ms_per_step': ms / args.steps,
                        'h2d_bytes_per_step': int(host_np.nbytes // world), 'd2h_bytes_per_step': int((hi - lo) * side * (4 + 8 * NB_CLASSES))},
                'gpu_launches': int(launches), 'stages': stages, 'whole_image_single_gpu': mono}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_texture(args):
    """extra workload (not the headline line): BASELINE config 3 -- 2048x2048 images with the full Leung-Malik bank + colour
    statistics (D = 189), 4 classes, images sharded over the GPUs (weak scaling; the 64-image batch is steps x GPUs images).
    The class model (D = 189) is fitted on the device by the large-D path of isb_gmm_fit_predict (16 < D <= 232)."""
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback)'
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from pyimsegm_b200 import _lib, pipelines
    lib = _lib.lib()
    fts = {'color': ('mean', 'std', 'energy'), 'tLM': ('mean', 'std', 'energy')}
    host_np = torch.from_numpy(synth_texture_image(3000 + rank)).pin_memory().numpy()

    def features_only():
        return pipelines.compute_color2d_superpixels_features(host_np, fts, sp_size=SP_SIZE, sp_regul=SP_REGUL)

    def step():
        return pipelines.pipe_color2d_slic_features_model_graphcut(host_np, 4, fts, sp_size=SP_SIZE, sp_regul=SP_REGUL,
                                                                   gc_regul=GC_REGUL, gc_edge_type='model')

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(steps):
            out = fn()
        ev1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        ms = torch.tensor([max(ev0.elapsed_time(ev1), wall)], device='cuda', dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for _ in range(max(1, min(args.warmup, 2))):
        features_only()
    step()
    lib.isb_profile_enable(1)
    ms_f, (slic, feats) = timed(features_only, args.steps)
    nstage = lib.isb_profile_stage_count()
    ms_arr, cnt_arr = (C.c_double * nstage)(), (C.c_longlong * nstage)()
    lib.isb_profile_collect(ms_arr, cnt_arr)
    lib.isb_profile_enable(0)
    n0 = lib.isb_launch_count()
    ms, (segm, soft) = timed(step, args.steps)
    launches = lib.isb_launch_count() - n0
    stages = {lib.isb_profile_stage_name(i).decode(): {'ms_per_step': ms_arr[i] / args.steps} for i in range(nstage) if ms_arr[i] > 0}
    # one more pass of the whole step with the stage timers on (class model, graph cut, gathers)
    lib.isb_profile_enable(1)
    step()
    ms_arr2, cnt_arr2 = (C.c_double * nstage)(), (C.c_longlong * nstage)()
    lib.isb_profile_collect(ms_arr2, cnt_arr2)
    lib.isb_profile_enable(0)
    for i in range(nstage):
        name = lib.isb_profile_stage_name(i).decode()
        if ms_arr2[i] > 0 and name not in stages:
            stages[name] = {'ms_per_step': ms_arr2[i]}
    if rank == 0:
        mpix = H * W / 1e6
        lm = stages.get('lm_texture', {}).get('ms_per_step', 0.0)
        line = {'metric': METRIC, 'value': world * args.steps * mpix / (ms / 1e3), 'unit': 'MPix/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f64 (SLIC, statistics), tf32x3 with f32 accumulate (LM bank)', 'data': 'synthetic',
                'config': {'workload': 'config3: 2048x2048 RGB f64 textured synthetic, colour + full LM bank (D=%d), 4-class GMM + GraphCut; '
                                       '1 image per GPU per step' % feats.shape[1],
                           'class_model': 'StandardScaler + full-covariance GMM (n_init 9, max_iter 99) fitted on the device (large-D path)',
                           'timed': 'host image in, (segm, segm_soft) out, max(wall clock, CUDA events)'},
                'e2e': {'value': world * args.steps * mpix / (ms / 1e3), 'unit': 'MPix/s', 'h2d_bytes_per_step': int(host_np.nbytes),
                        'd2h_bytes_per_step': int(segm.nbytes + soft.nbytes)},
                'features_only': {'value': world * args.steps * mpix / (ms_f / 1e3), 'unit': 'MPix/s', 'ms_per_step': ms_f / args.steps,
                                  'note': 'compute_color2d_superpixels_features: SLIC + colour + LM descriptors, host in / host out'},
                'roofline': lm_roofline(lm, H, W),
                'gpu_launches': int(launches), 'stages': stages}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def lm_roofline(lm_ms, H, W):
    """tensor-bound roofline of the Leung-Malik stage: algorithmic flops = one multiply-add per tap (3 channels x 76 kernels x 33^2 x 2
    per pixel, SURVEY 8d); executed = what the tcgen05 contraction issues (76 -> 80 filters, 33 -> 40 taps per kernel row, three TF32
    products per multiply)"""
    if not lm_ms:
        return None
    peak, peak_source = load_tensor_peak()
    algo = 3 * 76 * 33 * 33 * 2 * H * W / (lm_ms / 1e3) / 1e12
    executed = 3 * 80 * 33 * 40 * 2 * 3 * H * W / (lm_ms / 1e3) / 1e12
    return {'kernel': 'k_lm_conv_ts (lm_texture stage: FP64 background blur + tcgen05 contraction + fused statistics)', 'bound': 'tensor',
            'unit': 'TFLOP/s', 'achieved': algo, 'peak': peak, 'frac': algo / peak, 'peak_source': peak_source,
            'executed_tf32': executed, 'executed_frac_of_tf32_peak': executed / (peak / 2),
            'note': 'achieved = algorithmic flops over the WHOLE lm_texture stage time (CUDA events); peak = measured dense bf16 (TF32 runs '
                    'at half of it); the contraction kernel alone and its ncu capture: profiles/r02_lm_tcgen05.md'}


def run_rg2sp(args):
    """extra workload (not the headline line): BASELINE config 4 -- region growing with a shape prior on superpixels (RG2SP) on an
    ovary-like synthetic image (the reference's drosophila slices do not travel to the GPU box): class segmentation by the hot
    path, SLIC superpixels, a shape model from Ray features, then the growing loop whose every step is a device graph cut."""
    import torch
    rank, world, local = dist_env()
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback)'
    torch.cuda.set_device(local)
    if rank != 0:
        return
    from pyimsegm_b200 import _lib, pipelines, region_growing as rg, superpixels
    lib = _lib.lib()
    h, w = 640, 1024
    img, annot, centres = synth_eggs_image(4000, h, w)
    list_rays, _ = rg.compute_object_shapes([(annot == i + 1) for i in range(len(centres))], ray_step=10, interp_order='spline', smooth_coef=1)
    chist = rg.transform_rays_model_cdf_histograms(np.round(list_rays).astype(int), nb_bins=12)
    start = [(c[0] + 5, c[1] - 6) for c in centres]
    times = {'class_segmentation': 0.0, 'superpixels': 0.0, 'region_growing': 0.0}

    def step():
        t0 = time.perf_counter()
        segm, _ = pipelines.pipe_color2d_slic_features_model_graphcut(img, 2, FEATURES, sp_size=25, sp_regul=0.2)
        fg = int(np.bincount(segm[annot > 0]).argmax())            # which of the two unsupervised classes is the eggs
        t1 = time.perf_counter()
        slic = superpixels.segment_slic_img2d(img, sp_size=15, relative_compact=0.3)
        t2 = time.perf_counter()
        prob = rg.compute_segm_prob_fg(slic, (segm == fg).astype(int), [0.1, 0.9])
        history = {}
        labels = rg.region_growing_shape_slic_graphcut(slic, prob, start, (None, chist), 'cdf', coef_shape=2., coef_pairwise=5.,
                                                       prob_label_trans=[0.1, 0.03], nb_iter=150, debug_history=history)
        t3 = time.perf_counter()
        times['class_segmentation'] += t1 - t0; times['superpixels'] += t2 - t1; times['region_growing'] += t3 - t2
        return labels[slic], len(history['criteria'])

    for _ in range(max(args.warmup, 1)):
        step()
    for k in times:
        times[k] = 0.0
    n0 = lib.isb_launch_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        objects, n_steps = step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    jac = []
    for i in range(len(centres)):
        a, b = objects == i + 1, annot == i + 1
        jac.append(float((a & b).sum()) / float((a | b).sum()))
    line = {'metric': METRIC, 'value': h * w / 1e6 / dt, 'unit': 'MPix/s', 'n_gpus': 1, 'steps': args.steps, 'warmup': max(args.warmup, 1),
            'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': 'config4: %dx%d ovary-like synthetic image, 6 eggs; 2-class SLIC+GMM+GraphCut segmentation, SLIC sp_size=15 '
                                   'superpixels, RG2SP region growing with a Ray-feature shape prior (one device graph cut per growing step)' % (h, w),
                       'timed': 'host image in, object label map out, wall clock (the growing loop is host driven)'},
            'e2e': {'value': h * w / 1e6 / dt, 'unit': 'MPix/s', 'h2d_bytes_per_step': int(2 * img.nbytes), 'd2h_bytes_per_step': int(objects.nbytes)},
            'gpu_launches': int(lib.isb_launch_count() - n0), 'growing_steps': int(n_steps),
            'ms_per_stage': {k: v / args.steps * 1e3 for k, v in times.items()}, 'jaccard_per_egg': jac,
            'cpu_baseline': None, 'reference_libs': probe_reference_libs()}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-images', type=int, default=4, help='images in the bounded cpu_baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--ref-workers', type=int, default=0, help='processes of the reference arm (default: min(16, 0.6 * cpus), the measured best)')
    ap.add_argument('--workload', default='config2', choices=['config2', 'config3', 'config4', 'config5'],
                    help='config2 = the headline line (default); config5 = one 8192x8192 image banded over the GPUs (extra)')
    ap.add_argument('--tiled-side', type=int, default=8192)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step of the headline path returned to DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.workload != 'config2'):
        ap.error('--dump-outputs applies to the headline workload (--impl ours --workload config2)')
    if args.impl == 'reference':
        run_reference(args)
    elif args.workload == 'config5':
        run_tiled(args)
    elif args.workload == 'config3':
        run_texture(args)
    elif args.workload == 'config4':
        run_rg2sp(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
