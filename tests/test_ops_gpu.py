"""GPU parity of index_max / ball_query: bit-exact int32 outputs vs the CPU oracles, the golden
fixtures produced by the reference's own forward_cpu, and the stored outputs of the reference's
own CUDA kernels."""
import glob
import hashlib
import os

import numpy as np
import pytest
import torch

import oracle
from deepi2p_b200 import point_ops, synthetic as syn

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def run_index_max(data, index, K):
    d = torch.from_numpy(np.ascontiguousarray(data)).cuda()
    i = torch.from_numpy(np.ascontiguousarray(index)).cuda()
    return point_ops.index_max_forward(d, i, K).cpu().numpy()


def run_ball_query(dist, radius, K):
    d = torch.from_numpy(np.ascontiguousarray(dist)).cuda()
    return point_ops.ball_query_forward(d, radius, K).cpu().numpy()


@pytest.mark.parametrize("B,C,N,K", [(2, 5, 1000, 16), (3, 32, 20480, 128), (1, 1, 7, 3), (2, 7, 1023, 64),
                                     (1, 3, 4096, 4000), (1, 2, 513, 19000)])
def test_index_max_random(cuda, B, C, N, K):
    data, index = syn.make_index_max_inputs(B * 1000 + C, B, C, N, K)
    np.testing.assert_array_equal(run_index_max(data, index, K), oracle.index_max(data, index, K))


def test_index_max_adversarial(cuda):
    B, C, N, K = 2, 6, 2048, 32
    rng = np.random.default_rng(0)
    data, index = syn.make_index_max_inputs(5, B, C, N, K)
    index[:, :] = rng.integers(0, K - 4, (B, N))          # segments K-4..K-1 empty -> 0
    data[0, 0, :] = 1.5                                    # all ties -> lowest n per segment
    data[0, 1, :] = -2000.0                                # everything <= -1000 -> 0
    data[0, 2, :] = -1000.0                                # exactly the floor never wins (strict >)
    data[0, 3, ::3] = np.nan                               # NaN never wins
    data[0, 4, :] = np.nan                                 # all NaN -> 0
    data[0, 5, :] = np.where(rng.uniform(size=N) < 0.5, 0.0, -0.0)   # -0 == +0: first occurrence
    data[1, 0, :] = np.inf
    data[1, 1, :] = rng.integers(0, 3, N).astype(np.float32)         # many ties
    data[1, 2, 5] = 3e38
    got = run_index_max(data, index, K)
    np.testing.assert_array_equal(got, oracle.index_max(data, index, K))
    assert (got[:, :, K - 4:] == 0).all()


def test_index_max_config3_shape_property(cuda):
    """BASELINE config 3 shape (B=64, C=64, N=16384, K=64): the oracle on a slice, and for the
    whole output the defining property (value at the returned index is the segment max)."""
    B, C, N, K = 64, 64, 16384, 64
    g = torch.Generator(device="cuda").manual_seed(3)
    data = torch.randn((B, C, N), device="cuda", generator=g)
    index = torch.randint(0, K, (B, N), device="cuda", generator=g, dtype=torch.int32)
    out = point_ops.index_max_forward(data, index, K)
    sl = slice(0, 2)
    np.testing.assert_array_equal(out[sl].cpu().numpy(),
                                  oracle.index_max(data[sl].cpu().numpy(), index[sl].cpu().numpy(), K))
    seg_max = torch.full((B, C, K), -float("inf"), device="cuda")
    seg_max.scatter_reduce_(2, index.long()[:, None, :].expand(B, C, N), data, reduce="amax")
    picked = torch.gather(data, 2, out.long())
    assert torch.equal(picked, seg_max)
    assert torch.equal(torch.gather(index.long()[:, None, :].expand(B, C, N), 2, out.long()),
                       torch.arange(K, device="cuda")[None, None, :].expand(B, C, K))


@pytest.mark.parametrize("B,M,N,K", [(2, 8, 1000, 16), (4, 64, 16384, 64), (1, 1, 5, 8), (2, 3, 33, 1), (1, 5, 700, 900)])
def test_ball_query_random(cuda, B, M, N, K):
    dist, radius = syn.make_ball_query_inputs(B + M, B, M, N, min(K, N))
    np.testing.assert_array_equal(run_ball_query(dist, radius, K), oracle.ball_query(dist, radius, K))


def test_ball_query_adversarial(cuda):
    B, M, N, K = 1, 8, 3000, 64
    dist, radius = syn.make_ball_query_inputs(1, B, M, N, K)
    dist[0, 0, :] = radius + 1.0                  # cnt == 0 -> zeros
    dist[0, 1, :] = radius + 1.0; dist[0, 1, 2999] = radius        # single hit at the end, inclusive <=
    dist[0, 2, :] = 0.0                           # everything hits: first K
    dist[0, 3, :] = np.nan                        # NaN never hits
    dist[0, 4, :] = radius + 1.0; dist[0, 4, [5, 17, 2000]] = 0.0  # cnt = 3 < K -> cyclic repeat
    dist[0, 5, :] = radius + 1.0; dist[0, 5, :63] = 0.0            # cnt = K - 1
    got = run_ball_query(dist, radius, K)
    np.testing.assert_array_equal(got, oracle.ball_query(dist, radius, K))
    assert (got[0, 0] == 0).all() and (got[0, 1] == 2999).all() and (got[0, 3] == 0).all()
    np.testing.assert_array_equal(got[0, 4, :6], [5, 17, 2000, 5, 17, 2000])


def test_ball_query_split_path_adversarial(cuda):
    """N >= 4096 takes the row-split kernel: hits only in a late quarter, exactly K hits spread over
    the quarters, more than K in the first quarter, none, cyclic padding across quarter boundaries."""
    B, M, N, K = 1, 8, 6000, 20
    rng = np.random.default_rng(5)
    dist = np.full((B, M, N), 5.0, dtype=np.float32)
    radius = 1.0
    dist[0, 0, [5990, 5995]] = 0.5                               # two hits at the very end -> cyclic repeat
    dist[0, 1, :100] = 0.5                                        # > K hits in the first quarter
    dist[0, 2, [10, 1600, 3100, 4600, 5999]] = 1.0                # one hit per quarter (+1), inclusive <=
    dist[0, 3, rng.choice(N, K, replace=False)] = 0.0             # exactly K hits anywhere
    dist[0, 4, rng.choice(N, 3 * K, replace=False)] = 0.0         # 3K hits anywhere
    dist[0, 5, :] = np.nan
    dist[0, 6, 1499:1503] = 0.1                                   # straddles the first quarter boundary (1504)
    got = run_ball_query(dist, radius, K)
    np.testing.assert_array_equal(got, oracle.ball_query(dist, radius, K))
    np.testing.assert_array_equal(got[0, 0, :4], [5990, 5995, 5990, 5995])


def test_golden_index_max(cuda):
    """Fixtures written by tests/golden/make_golden.py from the REFERENCE's own forward_cpu."""
    files = sorted(glob.glob(os.path.join(GOLDEN, "index_max_*.npz")))
    assert files, "golden fixtures missing"
    for f in files:
        z = np.load(f)
        np.testing.assert_array_equal(run_index_max(z["data"], z["index"], int(z["K"])), z["out"])


def test_index_max_queue_overflow_and_ties(cuda):
    """Ascending data makes EVERY element a new running maximum (the filter passes everything, the per-warp candidate
    queues overflow and the in-place path is taken); constant data makes every element a tie (lowest n must win)."""
    B, C, N, K = 2, 5, 8192, 16
    rng = np.random.default_rng(5)
    index = rng.integers(0, K, (B, N), dtype=np.int32)
    data = np.empty((B, C, N), dtype=np.float32)
    data[:, 0] = np.arange(N, dtype=np.float32)[None]               # ascending: last element of each segment wins
    data[:, 1] = -np.arange(N, dtype=np.float32)[None]              # descending: first element wins
    data[:, 2] = 3.25                                               # all ties: lowest n wins
    data[:, 3] = np.repeat(np.arange(N // 64, dtype=np.float32), 64)[None]   # plateaus of 64 equal values
    data[:, 4] = rng.standard_normal((B, N), dtype=np.float32)
    np.testing.assert_array_equal(run_index_max(data, index, K), oracle.index_max(data, index, K))


def test_index_max_dropin_cpu_entry_points(cuda):
    """forward_cpu / forward_multi_thread_cpu keep the reference's CPU-tensor contract (index_max.cpp:73-112) and
    reproduce the fixtures written by the reference's own forward_cpu."""
    import importlib
    im = importlib.import_module("deepi2p_b200.dropin.index_max")
    for f in sorted(glob.glob(os.path.join(GOLDEN, "index_max_*.npz"))):
        z = np.load(f)
        d, i, K = torch.from_numpy(z["data"]), torch.from_numpy(z["index"]), int(z["K"])
        for out in (im.forward_cpu(d, i, K), im.forward_multi_thread_cpu(d, i, K, 8)):
            assert out.device.type == "cpu" and out.dtype == torch.int32
            np.testing.assert_array_equal(out.numpy(), z["out"])
    with pytest.raises(RuntimeError):
        im.forward_cpu(torch.zeros(1, 1, 4, device="cuda"), torch.zeros(1, 4, dtype=torch.int32, device="cuda"), 2)


def test_ball_query_vector_path_adversarial(cuda):
    """N a multiple of 2048 and an aligned matrix take the 128-bit path (lane l holds elements 4l..4l+3 of a
    128-element block): hits in all four components of one lane, runs across lane / block / step / quarter
    boundaries, every element a hit, K reached in mid-block, K - 1 hits, none, NaN."""
    B, M, N, K = 1, 10, 8192, 24
    dist = np.full((B, M, N), 7.0, dtype=np.float32)
    dist[0, 0, 40:44] = 0.0                                        # the four components of lane 10
    dist[0, 1, 126:131] = 1.0                                      # across a 128-element block boundary, inclusive <=
    dist[0, 2, 509:515] = 0.0                                      # across a 512-element step boundary
    dist[0, 3, 2046:2050] = 0.0                                    # across the first quarter boundary (2048)
    dist[0, 4, :] = 0.0                                            # everything hits: first K
    dist[0, 5, 3:3 + 4 * K:4] = 0.0                                # component 3 of K consecutive lanes
    dist[0, 6, 1000:1000 + K - 1] = 0.0                            # K - 1 hits -> one cyclic repeat
    dist[0, 7, :] = np.nan
    dist[0, 8, 100:110] = 0.0; dist[0, 8, 105] = 7.0; dist[0, 8, 8191] = 0.0   # a gap inside a run; the last element
    rng = np.random.default_rng(9)
    dist[0, 9, rng.choice(N, 5 * K, replace=False)] = 0.0          # 5K hits anywhere: K reached in mid-block
    got = run_ball_query(dist, 1.0, K)
    np.testing.assert_array_equal(got, oracle.ball_query(dist, 1.0, K))
    np.testing.assert_array_equal(got[0, 0, :8], [40, 41, 42, 43, 40, 41, 42, 43])
    # a view that is not 16-byte aligned takes the scalar path: same answer
    d = torch.from_numpy(np.concatenate([np.zeros(1, np.float32), dist.ravel()])).cuda()[1:].view(B, M, N)
    assert d.data_ptr() % 16 != 0
    np.testing.assert_array_equal(point_ops.ball_query_forward(d, 1.0, K).cpu().numpy(), got)


def test_ball_query_later_quarters_stop_early(cuda):
    """Rows whose first quarter already holds K hits: later quarters stop loading once the running counts say so, and
    whatever they had collected must not leak into the output."""
    B, M, N, K = 1, 4, 32768, 32
    dist = np.full((B, M, N), 9.0, dtype=np.float32)
    dist[0, 0, :K] = 0.0; dist[0, 0, N // 2:] = 0.0                 # K hits at once, then half the row hits
    dist[0, 1, 100:100 + 2 * K] = 0.0; dist[0, 1, -5:] = 0.0        # > K early, a few at the very end
    dist[0, 2, ::1024] = 0.0                                        # exactly 32 hits spread over all quarters
    dist[0, 3, N // 4 - 3:N // 4 + 3] = 0.0                         # 6 hits straddling the first boundary
    got = run_ball_query(dist, 1.0, K)
    np.testing.assert_array_equal(got, oracle.ball_query(dist, 1.0, K))


def test_against_reference_kernels(cuda):
    """The reference's own CUDA kernels (forward_cuda_shared_mem of index_max / ball_query, compiled unmodified) as the
    bit-exact checker: their outputs on these inputs are stored in reference_kernels.npz
    (tests/golden/make_reference_kernels_golden.py)."""
    def digest(*arrays):                               # as the fixture's generator computes it
        h = hashlib.sha256()
        for a in arrays:
            h.update(np.ascontiguousarray(a).tobytes())
        return h.hexdigest()

    g = np.load(os.path.join(GOLDEN, "reference_kernels.npz"))
    B, C, N, K = (int(v) for v in g["im_shape"])
    data, index = syn.make_index_max_inputs(int(g["im_seed"]), B, C, N, K)
    assert digest(data, index) == str(g["im_input_sha256"]), "index_max inputs differ from the ones the fixture was made on"
    np.testing.assert_array_equal(run_index_max(data, index, K), g["im_out"])
    B, M, N, K = (int(v) for v in g["bq_shape"])
    dist, radius = syn.make_ball_query_inputs(int(g["bq_seed"]), B, M, N, K)
    assert digest(dist) == str(g["bq_input_sha256"]) and radius == float(g["bq_radius"]), \
        "ball_query inputs differ from the ones the fixture was made on"
    np.testing.assert_array_equal(run_ball_query(dist, radius, K), g["bq_out"])


def test_argument_checks(cuda):
    with pytest.raises(RuntimeError):
        point_ops.index_max_forward(torch.zeros(1, 1, 4), torch.zeros(1, 4, dtype=torch.int32), 2)   # CPU tensor
    d = torch.zeros(2, 2, 8, device="cuda")
    with pytest.raises(RuntimeError):
        point_ops.index_max_forward(d.transpose(1, 2), torch.zeros(2, 2, dtype=torch.int32, device="cuda"), 2)
    with pytest.raises(RuntimeError):
        point_ops.ball_query_forward(torch.zeros(1, 1, 4), 1.0, 2)


@pytest.mark.parametrize("B,M,N,K,cube,radius", [(2, 16, 4096, 32, 20.0, 2.0), (1, 64, 16384, 64, 20.0, 2.0),
                                                 (2, 8, 1000, 16, 5.0, 30.0), (1, 4, 50, 8, 1.0, 0.05),
                                                 (1, 5, 3000, 10, 0.0, 1.0)])
def test_ball_query_xyz_grid_hash(cuda, B, M, N, K, cube, radius):
    """Grid-hash radius search == the float32 restatement (and hence == ball_query on the same distances)."""
    rng = np.random.default_rng(N + K)
    pts = rng.uniform(0, cube, (B, 3, N)).astype(np.float32) if cube > 0 else np.zeros((B, 3, N), np.float32)
    nodes = rng.uniform(-0.1 * cube, 1.1 * cube, (B, 3, M)).astype(np.float32) if cube > 0 else np.zeros((B, 3, M), np.float32)
    if cube > 0:
        nodes[:, :, 0] = pts[:, :, 7]                    # a node exactly on a point (d = 0)
        nodes[0, :, 1] = [1e6, 1e6, 1e6]                 # far outside the bounding box: no hits -> zeros
    got = point_ops.ball_query_xyz_forward(torch.from_numpy(pts).cuda(), torch.from_numpy(nodes).cuda(), radius, K).cpu().numpy()
    want = oracle.ball_query_xyz(pts, nodes, radius, K)
    np.testing.assert_array_equal(got, want)
    if cube > 0:
        assert (got[0, 1] == 0).all()
    # consistency with the dense op on the same float32 squared distances (compare d2 <= r2 via sqrt-free matrix)
    d = pts[:, :, None, :] - nodes[:, :, :, None]
    d2 = ((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]).astype(np.float32)
    dense = run_ball_query(d2, float(np.float32(radius) * np.float32(radius)), K)
    np.testing.assert_array_equal(got, dense)


def _cluster_check(pts, nodes, k):
    got = point_ops.cluster_assign_forward(torch.from_numpy(pts).cuda(), torch.from_numpy(nodes).cuda(), k)
    want = oracle.cluster_assign(pts, nodes, k)
    for name in ("min_k_idx", "min_idx", "count", "cluster_mean", "pc_centers", "pc_decentered"):
        np.testing.assert_array_equal(got[name].cpu().numpy(), want[name], err_msg=name)     # bit-exact, floats too
    return got, want


@pytest.mark.parametrize("B,N,M,k", [(3, 5000, 128, 3), (8, 20480, 128, 3), (2, 1024, 1, 1), (1, 777, 8, 8),
                                     (1, 3000, 2048, 5), (2, 1, 4, 2)])
def test_cluster_assign_matches_oracle(cuda, B, N, M, k):
    """8(f) N4: nearest-node clustering of networks_pc.py:60-85, every output bit-exact against the oracle."""
    rng = np.random.default_rng(B * 1000 + N + M + k)
    pts = rng.uniform(-40, 40, (B, 3, N)).astype(np.float32)
    nodes = rng.uniform(-40, 40, (B, 3, M)).astype(np.float32)
    got, want = _cluster_check(pts, nodes, k)
    assert int(got["count"].sum()) == B * N
    # feeds index_max exactly like the encoder does (:88-90)
    C = 8
    feat = rng.standard_normal((B, C, N)).astype(np.float32)
    idx = point_ops.index_max_forward(torch.from_numpy(feat).cuda(), got["min_idx"], M)
    np.testing.assert_array_equal(idx.cpu().numpy(), oracle.index_max(feat, want["min_idx"], M))


def test_cluster_assign_ties_empty_nodes_and_determinism(cuda):
    rng = np.random.default_rng(5)
    # lattice points and lattice nodes: masses of exact distance ties; duplicated nodes; a node nobody picks
    pts = rng.integers(-4, 5, (2, 3, 4096)).astype(np.float32)
    nodes = rng.integers(-4, 5, (2, 3, 32)).astype(np.float32)
    nodes[:, :, 5] = nodes[:, :, 2]                      # duplicate: the lower index must win every time
    nodes[:, :, 9] = 1e4                                 # empty cluster: count 0, mean 0 (:75, 0 / 1e-5)
    got, want = _cluster_check(pts, nodes, 4)
    assert (got["count"][:, 5] == 0).all() and (got["count"][:, 9] == 0).all()
    assert (got["cluster_mean"][:, :, 9] == 0).all()
    again = point_ops.cluster_assign_forward(torch.from_numpy(pts).cuda(), torch.from_numpy(nodes).cuda(), 4)
    for name in got:
        assert torch.equal(got[name], again[name]), name   # atomics land in any order, the result may not change
    # against the reference's own formulas in torch (float tree sums: tolerance, indices where unambiguous)
    p, nd = torch.from_numpy(pts).cuda(), torch.from_numpy(nodes).cuda()
    diff = torch.norm(p.unsqueeze(3) - nd.unsqueeze(2), dim=1, p=2)
    ref_d = torch.gather(diff, 2, got["min_k_idx"].long())
    top_d, _ = torch.topk(diff, k=4, dim=2, largest=False, sorted=True)
    assert torch.equal(ref_d, top_d)                     # same distances as torch.topk picks (ties may permute ids)
    mask = torch.eq(got["min_idx"].long().unsqueeze(2), torch.arange(32, device="cuda").view(1, 1, 32)).float()
    cm = (p.unsqueeze(3) * mask.unsqueeze(1)).sum(2) / (mask.sum(1).unsqueeze(1) + 1e-5)
    assert (cm - got["cluster_mean"]).abs().max().item() < 1e-4


def test_cluster_assign_argument_checks(cuda):
    p = torch.zeros(1, 3, 16, device="cuda")
    nd = torch.zeros(1, 3, 4, device="cuda")
    from deepi2p_b200 import _native
    with pytest.raises(_native.NativeError):
        point_ops.cluster_assign_forward(p, nd, 5)        # k > M
    with pytest.raises(_native.NativeError):
        point_ops.cluster_assign_forward(p, torch.zeros(1, 3, 16, device="cuda"), 9)    # k > 8
    with pytest.raises(RuntimeError):
        point_ops.cluster_assign_forward(p.cpu(), nd, 1)
    out = point_ops.cluster_assign_forward(torch.zeros(2, 3, 0, device="cuda"), torch.ones(2, 3, 4, device="cuda"), 2)
    assert out["min_k_idx"].shape == (2, 0, 2) and (out["count"] == 0).all() and (out["cluster_mean"] == 0).all()


def test_cluster_assign_committed_golden(cuda):
    g = np.load(os.path.join(GOLDEN, "frustum_small.npz")) if "GOLDEN" in globals() else np.load(
        os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frustum_small.npz"))
    got = point_ops.cluster_assign_forward(torch.from_numpy(g["ca_pc"]).cuda(), torch.from_numpy(g["ca_node"]).cuda(), 3)
    np.testing.assert_array_equal(got["min_k_idx"].cpu().numpy(), g["ca_min_k_idx"])
    np.testing.assert_array_equal(got["count"].cpu().numpy(), g["ca_count"])
    np.testing.assert_array_equal(got["cluster_mean"].cpu().numpy(), g["ca_mean"])
    np.testing.assert_array_equal(got["pc_decentered"].cpu().numpy(), g["ca_decentered"])
