"""Writes tests/golden/reference_kernels.npz: the outputs of the REFERENCE's own CUDA kernels
(index_max / ball_query forward_cuda_shared_mem, compiled unmodified by oracle/build_ref.py into oracle/_ref)
on two seeded inputs at the shipped model's shapes.  tests/test_ops_gpu.py::test_against_reference_kernels
compares the sm_100a kernels with them bit for bit.  Needs a CUDA device and a built oracle/_ref:

    python oracle/build_ref.py && python tests/golden/make_reference_kernels_golden.py [out.npz]

Only the seeds and shapes of the inputs are stored (the test regenerates them with deepi2p_b200.synthetic),
together with a SHA-256 of each input so that a changed generator is reported as such.
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import build_ref  # noqa: E402
from deepi2p_b200 import synthetic as syn  # noqa: E402

IM_SEED, IM_SHAPE = 77, (8, 32, 20480, 128)       # B, C, N, K: shipped model shape, B <= 1024, B*K*4 <= 48 KB
BQ_SEED, BQ_SHAPE = 78, (8, 64, 16384, 64)        # B, M, N, K


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main(out):
    ref_im = build_ref.load("index_max")
    ref_bq = build_ref.load("ball_query")
    data, index = syn.make_index_max_inputs(IM_SEED, *IM_SHAPE)
    im_out = ref_im.forward_cuda_shared_mem(torch.from_numpy(data).cuda(), torch.from_numpy(index).cuda(), IM_SHAPE[3])
    dist, radius = syn.make_ball_query_inputs(BQ_SEED, *BQ_SHAPE)
    bq_out = ref_bq.forward_cuda_shared_mem(torch.from_numpy(dist).cuda(), radius, BQ_SHAPE[3])
    torch.cuda.synchronize()
    np.savez_compressed(out, im_seed=IM_SEED, im_shape=np.array(IM_SHAPE), im_input_sha256=digest(data, index),
                        im_out=im_out.cpu().numpy(), bq_seed=BQ_SEED, bq_shape=np.array(BQ_SHAPE), bq_radius=radius,
                        bq_input_sha256=digest(dist), bq_out=bq_out.cpu().numpy())
    print(out, "index_max", tuple(im_out.shape), "ball_query", tuple(bq_out.shape), "radius", radius)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_kernels.npz"))
