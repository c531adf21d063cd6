"""Writes tests/golden/index_max_*.npz from the REFERENCE's own index_max.forward_cpu
(models/index_max_ext/index_max.cpp:73-112), compiled unmodified from /root/reference by
oracle/build_ref.py.  Run in the build container only (the GPU box has no /root/reference):

    python oracle/build_ref.py && python tests/golden/make_golden.py

ball_query has no CPU implementation in the reference, and the solver needs Ceres, so neither has
a fixture here; tests/golden/make_reference_kernels_golden.py stores the outputs of the reference's
CUDA kernels instead.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import build_ref  # noqa: E402

ref = build_ref.load("index_max")


def save(name, data, index, K):
    out = ref.forward_cpu(torch.from_numpy(data), torch.from_numpy(index), K).numpy()
    out_mt = ref.forward_multi_thread_cpu(torch.from_numpy(data), torch.from_numpy(index), K, 2).numpy()
    assert np.array_equal(out, out_mt)
    np.savez_compressed(os.path.join(HERE, "index_max_%s.npz" % name), data=data, index=index, K=np.int32(K), out=out)
    print(name, data.shape, K, "->", out.shape)


rng = np.random.default_rng(2024)
# 1. random, shipped-model-like proportions (scaled down)
B, C, N, K = 2, 8, 2048, 16
save("random", rng.standard_normal((B, C, N), dtype=np.float32), rng.integers(0, K, (B, N), dtype=np.int32), K)
# 2. ties, floor, NaN, signed zeros, empty segments
B, C, N, K = 1, 8, 512, 12
data = rng.standard_normal((B, C, N), dtype=np.float32)
index = rng.integers(0, K - 3, (B, N), dtype=np.int32)
data[0, 0, :] = 2.0
data[0, 1, :] = -1000.0
data[0, 2, :] = -1500.0
data[0, 3, ::2] = np.nan
data[0, 4, :] = np.nan
data[0, 5, :] = np.where(rng.uniform(size=N) < 0.5, 0.0, -0.0).astype(np.float32)
data[0, 6, :] = rng.integers(0, 2, N).astype(np.float32)
data[0, 7, :] = np.inf
save("adversarial", data, index, K)
# 3. odd sizes (N not a multiple of 4), K > N
B, C, N, K = 3, 3, 37, 50
save("odd", rng.standard_normal((B, C, N), dtype=np.float32), rng.integers(0, K, (B, N), dtype=np.int32), K)
