"""Segmenting a sequence of images with ONE shared class model (the reference's experiment_group_gmm,
experiments_segmentation/run_segm_slic_model_graphcut.py:476-514): the model is fitted by estim_model_classes_group over the
images, then every image is segmented with it -- (A) with the fitted scikit-learn model, whose predict_proba runs on the host
(features down, probabilities up, once per image), and (B) with the same model wrapped in graph_cuts.DeviceClassModel, whose
probabilities are computed on the device.  Both through the batch API and through the single-image call.

    python scripts/bench_shared_model.py --workload config2    # 8 x 2048^2, colour means, K = 3, sp_size 29
    python scripts/bench_shared_model.py --workload config3    # 4 x 2048^2, colour + full Leung-Malik statistics (D = 189), K = 4

Prints one JSON line: MPix/s per variant (median, min, max over the repeats; host clock around calls that end in a synchronise),
the share of identical segm pixels and the largest |segm_soft| difference between A and B, and the card it ran on.
Needs a CUDA device; there is no fallback.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'config2': dict(n_images=8, features={'color': ['mean']}, K=3, image='regions'),
    'config3': dict(n_images=4, features={'color': ('mean', 'std', 'energy'), 'tLM': ('mean', 'std', 'energy')}, K=4, image='texture'),
}
SIDE, SP_SIZE, SP_REGUL, GC_REGUL = 2048, 29, 0.2, 1.


def gpu_info():
    """name, power limit and max SM clock of the card, read-only query"""
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in out.split(','))
    return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workload', default='config2', choices=sorted(WORKLOADS))
    ap.add_argument('--repeats', type=int, default=5)
    ap.add_argument('--images', type=int, default=None, help='images in the sequence (default: 8 for config2, 4 for config3)')
    args = ap.parse_args()
    if args.repeats < 5:
        ap.error('--repeats must be at least 5')
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_shared_model.py needs a CUDA device (there is no CPU fallback)')
    torch.cuda.set_device(0)
    import bench
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    wl = WORKLOADS[args.workload]
    n_images = args.images or wl['n_images']
    make = bench.synth_image if wl['image'] == 'regions' else bench.synth_texture_image
    images = [torch.from_numpy(make(5000 + i, SIDE, SIDE)).pin_memory().numpy() for i in range(n_images)]
    feats, K = wl['features'], wl['K']
    t0 = time.perf_counter()
    model, list_fts = pl.estim_model_classes_group(images, K, feats, sp_size=SP_SIZE, sp_regul=SP_REGUL)
    fit_s = time.perf_counter() - t0
    dcm = DeviceClassModel(model)
    kw = dict(dict_features=feats, sp_size=SP_SIZE, sp_regul=SP_REGUL, gc_regul=GC_REGUL)

    variants = {
        'A_batch_host_model': lambda: pl.segment_images_batch(images, model_pipeline=model, **kw),
        'B_batch_device_model': lambda: pl.segment_images_batch(images, model_pipeline=dcm, **kw),
        'A_single_host_model': lambda: [pl.segment_color2d_slic_features_model_graphcut(im, model, **kw) for im in images],
        'B_single_device_model': lambda: [pl.segment_color2d_slic_features_model_graphcut(im, dcm, **kw) for im in images],
    }
    outputs = {}
    for name, fn in variants.items():        # warm-up: every shape, the CUDA graphs (eager, capture, replay)
        for _ in range(3):
            outputs[name] = fn()
    times = {name: [] for name in variants}
    for _ in range(args.repeats):             # alternating, so that drift of the shared machine hits every variant alike
        for name, fn in variants.items():
            torch.cuda.synchronize()
            t = time.perf_counter()
            outputs[name] = fn()              # every call returns host arrays: it ends in a synchronise
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t)
    mpix = n_images * SIDE * SIDE / 1e6
    rates = {name: {'median': mpix / float(np.median(ts)), 'min': mpix / max(ts), 'max': mpix / min(ts),
                    'ms_per_image_median': 1e3 * float(np.median(ts)) / n_images} for name, ts in times.items()}

    def compare(a, b):
        same = sum(int(np.sum(x[0] == y[0])) for x, y in zip(a, b)) / float(sum(x[0].size for x in a))
        soft = max(float(np.abs(x[1] - y[1]).max()) for x, y in zip(a, b))
        return {'identical_segm_fraction': same, 'max_abs_segm_soft_diff': soft}

    line = {
        'metric': 'shared_model_segmentation', 'unit': 'MPix/s', 'higher_is_better': True, 'workload': args.workload,
        'images': n_images, 'side': SIDE, 'features': {k: list(v) for k, v in feats.items()}, 'n_features': int(list_fts[0].shape[1]),
        'K': K, 'sp_size': SP_SIZE, 'superpixels_per_image': [int(len(f)) for f in list_fts], 'repeats': args.repeats,
        'model': repr(model.steps[-1][1]) if hasattr(model, 'steps') else repr(model), 'model_fit_s': fit_s,
        'rates': rates,
        'speedup_batch_median': rates['B_batch_device_model']['median'] / rates['A_batch_host_model']['median'],
        'speedup_single_median': rates['B_single_device_model']['median'] / rates['A_single_host_model']['median'],
        'batch_A_vs_B': compare(outputs['A_batch_host_model'], outputs['B_batch_device_model']),
        'single_A_vs_B': compare(outputs['A_single_host_model'], outputs['B_single_device_model']),
        'gpu': gpu_info(),
        'timed': 'host images in, (segm, segm_soft) of every image out; host clock around calls that end in a synchronise',
    }
    print(json.dumps(line))


if __name__ == '__main__':
    main()
