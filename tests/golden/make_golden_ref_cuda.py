#!/usr/bin/env python
"""Generates tests/golden/ref_cuda.npz: a seeded sample of the outputs that
tests/test_ref_kernels.py::test_cuda_beside_the_reference_kernels_built_by_nvcc compares with the reference's own
kernels built by nvcc (oracle/_ref/libgf_ref_cuda.so, which needs the reference's source tree to build).  Where that
library is missing the test holds the kernels to this sample instead.

The values are this project's gf_hash_forward and sampler outputs on the test's inputs, written at a commit where the
live comparison found them bit-identical to the nvcc-built reference (hash encodings; per ray: sample counts, first
crossing, t, dist, warp / world positions, anchors).  Regenerate only from kernels that pass that live comparison.

  python tests/golden/make_golden_ref_cuda.py [OUT.npz]       # needs a B200
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests.helpers import load_rig  # noqa: E402
from tests.test_ref_kernels import S, beside_nvcc_inputs, cuda_beside_nvcc  # noqa: E402

N_HASH_ROWS = 2048
N_RAYS = 16


def main():
    rig = load_rig("rig8")
    inp = beside_nvcc_inputs(rig)
    _, got = cuda_beside_nvcc(rig, inp)
    got = {k: v.cpu().numpy() for k, v in got.items()}
    rng = np.random.RandomState(0)
    hash_rows = np.sort(rng.choice(got["hash_out"].shape[0], N_HASH_ROWS, replace=False))
    counts = got["counts"]
    rays = np.sort(rng.choice(np.nonzero(counts > 0)[0], N_RAYS, replace=False))
    m = np.arange(S)[None, :] < counts[rays][:, None]
    fx = dict(hash_rows=hash_rows, hash_out=got["hash_out"][hash_rows], counts=counts,
              first_oct_dis=got["first_oct_dis"], rays=rays)
    for k in ("ts", "dists", "warp_pts", "world_pts", "anchors"):
        fx[k] = got[k][rays][m]
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_cuda.npz")
    np.savez_compressed(path, **fx)
    print("wrote", path, os.path.getsize(path) >> 10, "KiB;", int(m.sum()), "samples of", N_RAYS, "rays")


if __name__ == "__main__":
    main()
