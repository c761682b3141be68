"""
Generate tests/golden/reference_cython.npz: what the reference's only native module (imsegm/features_cython.pyx, compiled
unchanged into oracle/_ref by `make -C oracle ref`) returns for the inputs of the tests that compare against it:

    tests/test_oracle_goldens.py::test_restatement_equals_reference_cython_module     (colour mean / energy / variance)
    tests/test_gpu_parity.py::test_color_stats_match_oracle_and_reference_module      (colour energy on an oracle SLIC map)
    tests/test_gpu_parity.py::test_remaining_native_functions                         (Ray features, both edge directions)

    python tests/golden/make_cython_goldens.py

The inputs are rebuilt here exactly as those tests build them (same seeds, same draws in the same order); only the module's
outputs are stored, so the tests need neither the reference tree nor oracle/_ref.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))


def main():
    import oracle
    from conftest import synth_regions
    oracle.build()
    fc = oracle.ref_features_cython()
    assert fc is not None, 'oracle/_ref/features_cython is missing: run `make -C oracle ref`'
    out = {}
    # test_restatement_equals_reference_cython_module
    rng = np.random.RandomState(3)
    img = rng.random_sample((60, 70, 3)).astype(np.float32)
    seg = (np.arange(60)[:, None] // 8 * 9 + np.arange(70)[None, :] // 8).astype(np.int32)
    mean = np.array(fc.computeColorImage2dMean(img, seg))
    out.update(blocks_mean=mean, blocks_energy=np.array(fc.computeColorImage2dEnergy(img, seg)),
               blocks_variance=np.array(fc.computeColorImage2dVariance(img, seg, mean.astype(np.float32))))
    # test_color_stats_match_oracle_and_reference_module
    img, _ = synth_regions(300, 400, seed=3)
    seg = oracle.segment_slic_img2d(img, 20, 0.2)
    out.update(slic_energy=np.array(fc.computeColorImage2dEnergy(img.astype(np.float32), seg.astype(np.int32))))
    # test_remaining_native_functions: replay that test's draws from RandomState(0) up to the Ray inputs
    rng = np.random.RandomState(0)
    rng.random_sample((5, 40, 50))
    rng.randint(-1, 6, (64, 80))
    rng.rand(64, 80)
    noise = rng.rand(40, 60) < 0.08
    pos = np.stack([rng.randint(0, 40, 25), rng.randint(0, 60, 25)], 1)
    for edge, e in (('up', 1), ('down', -1)):
        out['rays_' + edge] = np.array([fc.computeRayFeaturesBinary2d(noise.astype(np.int8), np.array(p, dtype=np.int32), 7.5, e)
                                        for p in pos])
    return out


if __name__ == '__main__':
    vectors = main()
    path = os.path.join(HERE, 'reference_cython.npz')
    np.savez_compressed(path, **vectors)
    print('wrote %s: %d arrays, %.0f KB' % (path, len(vectors), os.path.getsize(path) / 1024))
