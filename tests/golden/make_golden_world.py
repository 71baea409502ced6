"""Writes tests/golden/ref_world.npz: what the reference's own PCGVoxelGenerator.next_world (CPU) builds from the
bird's-eye-view files and tree assets of tests/test_gpu_generator.py::test_world_builder_reproduces_next_world.

Needs the reference's Python (staged by oracle/build_ref.py, or SD_REFERENCE_ROOT); no GPU:

    python tests/golden/make_golden_world.py"""
import os
import random
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS):
    if p not in sys.path:
        sys.path.insert(0, p)

import _golden                      # noqa: E402
import test_gpu_generator as tg     # noqa: E402
from oracle import refgen           # noqa: E402


def main():
    refgen.setup('dropin')
    import imaginaire.model_utils.pcg_gen as pcg
    out = {}
    with tempfile.TemporaryDirectory() as d:
        assets = tg.world_builder_inputs(d)
        ref = pcg.PCGVoxelGenerator(tg.WORLD_SIZE)
        random.seed(7)
        ref.next_world('cpu', d, assets)
    out['rng_state'] = np.asarray(random.getstate()[1], dtype=np.int64)
    out['voxel_t_shape'] = np.asarray(ref.voxel_t.shape, dtype=np.int64)
    _golden.record(out, 'voxel_t', ref.voxel_t, seed=1, exact=True)
    _golden.record(out, 'heightmap', ref.heightmap, seed=2, exact=True)
    out['trans_mat'] = ref.trans_mat.numpy()
    _golden.record(out, 'current_height_map', ref.current_height_map, seed=3, exact=True)
    _golden.record(out, 'current_semantic_map', ref.current_semantic_map, seed=4, exact=True)
    dst = os.path.join(HERE, 'ref_world.npz')
    np.savez_compressed(dst, **out)
    print(dst, os.path.getsize(dst) // 1024, 'KiB; voxel_t', tuple(ref.voxel_t.shape), ref.voxel_t.dtype, 'heightmap', ref.heightmap.dtype)


if __name__ == '__main__':
    main()
