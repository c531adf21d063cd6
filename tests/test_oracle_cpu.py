"""CPU tests of the oracle itself (no GPU): golden vectors from the reference's own code where the
reference can run (index_max), and independent cross-checks where it cannot (solver: PARITY
UNPINNED -- Ceres is not available offline; ball_query: the reference has no CPU path)."""
import glob
import math
import os

import numpy as np
import pytest

import oracle
from deepi2p_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_index_max_oracle_matches_reference_golden():
    files = sorted(glob.glob(os.path.join(GOLDEN, "index_max_*.npz")))
    assert len(files) >= 3
    for f in files:
        z = np.load(f)
        np.testing.assert_array_equal(oracle.index_max(z["data"], z["index"], int(z["K"])), z["out"])


def test_ops_oracles_match_reference_kernel_outputs():
    """tests/golden/reference_kernels.npz holds what the reference's own CUDA kernels returned on two seeded inputs
    (the only reference implementation of ball_query)."""
    g = np.load(os.path.join(GOLDEN, "reference_kernels.npz"))
    B, C, N, K = (int(v) for v in g["im_shape"])
    data, index = syn.make_index_max_inputs(int(g["im_seed"]), B, C, N, K)
    np.testing.assert_array_equal(oracle.index_max(data, index, K), g["im_out"])
    B, M, N, K = (int(v) for v in g["bq_shape"])
    dist, radius = syn.make_ball_query_inputs(int(g["bq_seed"]), B, M, N, K)
    np.testing.assert_array_equal(oracle.ball_query(dist, radius, K), g["bq_out"])


def test_index_max_oracle_vs_independent_restatement():
    data, index = syn.make_index_max_inputs(3, 2, 4, 500, 8)
    got = oracle.index_max(data, index, 8)
    for b in range(2):
        for c in range(4):
            for k in range(8):
                sel = np.where(index[b] == k)[0]
                vals = data[b, c, sel]
                ok = vals > -1000
                want = 0 if not ok.any() else sel[ok][np.argmax(vals[ok])]      # argmax = first maximum
                assert got[b, c, k] == want


def test_index_max_oracle_rejects_out_of_range_index():
    data, index = syn.make_index_max_inputs(3, 1, 1, 16, 4)
    index[0, 3] = 4
    with pytest.raises(ValueError):
        oracle.index_max(data, index, 4)


def test_ball_query_oracle_vs_independent_restatement():
    dist, radius = syn.make_ball_query_inputs(4, 2, 6, 400, 16)
    dist[0, 0, :] = radius + 1
    dist[0, 1, :] = radius + 1
    dist[0, 1, [7, 9]] = radius          # inclusive
    got = oracle.ball_query(dist, radius, 16)
    for b in range(2):
        for m in range(6):
            hits = np.where(dist[b, m] <= radius)[0][:16]
            if len(hits) == 0:
                want = np.zeros(16, dtype=np.int32)
            else:
                want = np.array([hits[i] if i < len(hits) else hits[(i - len(hits)) % len(hits)] for i in range(16)])
            np.testing.assert_array_equal(got[b, m], want)
    np.testing.assert_array_equal(got[0, 1, :4], [7, 9, 7, 9])


def _fd_grad(pts, lab, K, x, H, W, is_2d, h=1e-6):
    g = np.zeros(len(x))
    for j in range(len(x)):
        xp, xm = x.copy(), x.copy()
        xp[j] += h; xm[j] -= h
        g[j] = (oracle.evaluate(pts, lab, K, xp, H, W, is_2d)[0] - oracle.evaluate(pts, lab, K, xm, H, W, is_2d)[0]) / (2 * h)
    return g


@pytest.mark.parametrize("is_2d", [True, False])
def test_solver_oracle_gradient_matches_finite_differences(is_2d):
    smp = syn.make_sample(1, 4000)
    pts = smp["points"].astype(np.float64)
    x = np.array([0.3, -0.4, 0.03, 2.0]) if is_2d else np.array([0.02, 0.3, -0.01, -0.4, 0.03, 2.0])
    c, g, A = oracle.evaluate(pts, smp["pred"], smp["K"], x, smp["H"], smp["W"], is_2d)
    gn = _fd_grad(pts, smp["pred"], smp["K"], x, smp["H"], smp["W"], is_2d)
    np.testing.assert_allclose(g, gn, rtol=2e-4, atol=1e-4 * np.abs(g).max())
    assert np.allclose(A, A.T) and np.all(np.linalg.eigvalsh(A) > -1e-9 * np.abs(A).max())


def test_solver_oracle_cost_matches_numpy_restatement():
    """Independent vectorised numpy evaluation of the same cost (SURVEY.md Appendix A text)."""
    smp = syn.make_sample(2, 3000)
    p = smp["points"].astype(np.float64)
    ry, t = 0.4, np.array([0.5, 0.05, -1.0])
    c, s = math.cos(ry), math.sin(ry)
    X = c * p[0] + s * p[2] + t[0]; Y = p[1] + t[1]; Z = -s * p[0] + c * p[2] + t[2]
    K = smp["K"]; W1 = smp["W"] - 1; H1 = smp["H"] - 1
    u = K[0, 0] * X / Z + K[0, 2]; v = K[1, 1] * Y / Z + K[1, 2]
    lab = smp["pred"]
    xd = W1 / 2 - np.abs(u - W1 / 2); yd = H1 / 2 - np.abs(v - H1 / 2)
    r_out = np.where((Z > 0) & (xd > 0) & (yd > 0), xd + yd, 0.0)
    r0 = np.maximum(-u, 0) + np.maximum(u - W1, 0); r1 = np.maximum(-v, 0) + np.maximum(v - H1, 0)
    r2 = 100 * np.maximum(-Z, 0)
    s_blk = np.where(lab == 1, r0 ** 2 + r1 ** 2 + r2 ** 2, r_out ** 2)
    want = 0.5 * np.sum(np.log1p(s_blk))
    got = oracle.evaluate(p, lab, K, np.array([ry, *t]), smp["H"], smp["W"], True)[0]
    assert abs(got - want) <= 1e-9 * want


@pytest.mark.parametrize("is_2d", [True, False])
def test_solver_oracle_known_answer_and_descent(is_2d):
    smp = syn.make_sample(3, 4096)
    # zero-cost start: exact GT labels, start at GT => the init pose is returned unchanged
    P, cost, res, st, x = oracle.solve(smp["points"], smp["gt"], smp["K"], smp["ry_gt"], smp["t_gt"], smp["H"], smp["W"],
                                       [-100] * 3, [100] * 3, 500, is_2d)
    assert cost == 0.0 and st["iterations"] == 0 and st["termination"] == 0
    np.testing.assert_allclose(P, smp["P_gt"], atol=1e-15)
    assert res.shape[0] == int((smp["gt"] == 0).sum() + 3 * (smp["gt"] == 1).sum()) and not res.any()
    # perturbed start with GT labels: converges back to (near) the GT pose, cost decreases, bounds hold
    P2, cost2, res2, st2, x2 = oracle.solve(smp["points"], smp["gt"], smp["K"], smp["ry_gt"] + 0.05,
                                            smp["t_gt"] + np.array([0.3, 0.0, -0.4]), smp["H"], smp["W"],
                                            [-5, -0.1, -10], [5, 0.1, 10], 500, is_2d)
    x0 = np.array([smp["ry_gt"] + 0.05, *(smp["t_gt"] + np.array([0.3, 0.0, -0.4]))]) if is_2d else \
        np.array([0, smp["ry_gt"] + 0.05, 0, *(smp["t_gt"] + np.array([0.3, 0.0, -0.4]))])
    c0 = oracle.evaluate(smp["points"], smp["gt"], smp["K"], x0, smp["H"], smp["W"], is_2d)[0]
    assert cost2 < 0.5 * c0          # descends (the landscape has local minima; no global claim)
    assert np.isfinite(res2).all()
    t2 = P2[:3, 3]
    assert -5 <= t2[0] <= 5 and -0.1 <= t2[1] <= 0.1 and -10 <= t2[2] <= 10


def test_solver_oracle_infeasible_start_and_ignored_labels():
    smp = syn.make_sample(4, 1000)
    P, cost, res, st, x = oracle.solve(smp["points"], smp["pred"], smp["K"], 0.1, [0, 0.5, 0], smp["H"], smp["W"],
                                       [-5, -0.1, -10], [5, 0.1, 10])
    assert st["termination"] == 6 and x[2] == 0.5
    lab = smp["pred"].copy(); lab[::2] = 7
    c_all = oracle.evaluate(smp["points"][:, 1::2], smp["pred"][1::2], smp["K"], [0.1, 0, 0, 1], smp["H"], smp["W"])[0]
    c_ign = oracle.evaluate(smp["points"], lab, smp["K"], [0.1, 0, 0, 1], smp["H"], smp["W"])[0]
    assert abs(c_all - c_ign) <= 1e-12 * max(1.0, c_all)


def test_solver_oracle_vs_scipy_sanity():
    """Not parity (scipy applies the loss per scalar residual and uses another TR algorithm): with
    exact labels both must land close to the generating pose."""
    from scipy.optimize import least_squares
    smp = syn.make_sample(5, 2048)
    p = smp["points"].astype(np.float64); K = smp["K"]; W1 = smp["W"] - 1; H1 = smp["H"] - 1; lab = smp["gt"]

    def resid(x):
        c, s = math.cos(x[0]), math.sin(x[0])
        X = c * p[0] + s * p[2] + x[1]; Y = p[1] + x[2]; Z = -s * p[0] + c * p[2] + x[3]
        u = K[0, 0] * X / Z + K[0, 2]; v = K[1, 1] * Y / Z + K[1, 2]
        xd = W1 / 2 - np.abs(u - W1 / 2); yd = H1 / 2 - np.abs(v - H1 / 2)
        r_out = np.where((Z > 0) & (xd > 0) & (yd > 0), xd + yd, 0.0)
        r0 = np.maximum(-u, 0) + np.maximum(u - W1, 0); r1 = np.maximum(-v, 0) + np.maximum(v - H1, 0)
        r2 = 100 * np.maximum(-Z, 0)
        return np.concatenate([r_out[lab == 0], r0[lab == 1], r1[lab == 1], r2[lab == 1]])

    x0 = np.array([smp["ry_gt"] + 0.03, smp["t_gt"][0] + 0.2, 0.0, smp["t_gt"][2] - 0.3])
    sol = least_squares(resid, x0, loss="cauchy", bounds=([-10, -5, -0.1, -10], [10, 5, 0.1, 10]))
    P, cost, _, st, x = oracle.solve(p, lab, K, x0[0], x0[1:], smp["H"], smp["W"], [-5, -0.1, -10], [5, 0.1, 10])
    assert abs(x[0] - smp["ry_gt"]) < 0.02 and abs(sol.x[0] - smp["ry_gt"]) < 0.02
    assert np.linalg.norm(x[1:4] - smp["t_gt"]) < 0.5 and np.linalg.norm(sol.x[1:] - smp["t_gt"]) < 0.5


def test_initial_guess_front_filter():
    smp = syn.make_sample(6, 2000)
    iy, pf, lf, mask = oracle.initial_guess(smp["points"], smp["gt"])
    assert abs(oracle.wrap_in_pi(iy - smp["ry_gt"])) < 0.6          # heading of the in-frustum points
    assert pf.shape[1] == mask.sum() == lf.shape[0] and mask.sum() < 2000
    assert oracle.wrap_in_pi(3 * math.pi + 0.1) == pytest.approx(-math.pi + 0.1, abs=1e-12)


def test_cluster_assign_oracle_matches_reference_formulas():
    """oracle.cluster_assign against the reference's own torch formulation (models/networks_pc.py:60-82), on CPU:
    identical indices and counts, means / centres within float tree-sum error."""
    import torch
    rng = np.random.default_rng(11)
    B, N, M, k = 2, 700, 16, 3
    pc = rng.uniform(-40, 40, (B, 3, N)).astype(np.float32)
    node = rng.uniform(-40, 40, (B, 3, M)).astype(np.float32)
    o = oracle.cluster_assign(pc, node, k)
    p, nd = torch.from_numpy(pc), torch.from_numpy(node)
    diff = torch.norm(p.unsqueeze(3).expand(B, 3, N, M) - nd.unsqueeze(2).expand(B, 3, N, M), dim=1, p=2)    # :62
    _, min_k_idx = torch.topk(diff, k=k, dim=2, largest=False, sorted=True)                                    # :63
    min_idx = min_k_idx[:, :, 0]                                                                               # :64
    mask = torch.eq(min_idx.unsqueeze(2).expand(B, N, M), torch.arange(M).view(1, 1, M).expand(B, N, M))       # :65-66
    mask_row_sum = torch.sum(mask.unsqueeze(1).float(), dim=2)                                                 # :70-71
    cluster_mean = torch.sum(p.unsqueeze(3) * mask.unsqueeze(1).float(), dim=2) / (mask_row_sum + 1e-5)        # :74-75
    pc_centers = torch.gather(cluster_mean, index=min_idx.unsqueeze(1).expand(B, 3, N), dim=2)                 # :78-80
    np.testing.assert_array_equal(o["min_k_idx"], min_k_idx.numpy())
    np.testing.assert_array_equal(o["count"], mask_row_sum[:, 0].numpy().astype(np.int32))
    np.testing.assert_allclose(o["cluster_mean"], cluster_mean.numpy(), rtol=0, atol=2e-5)
    np.testing.assert_allclose(o["pc_decentered"], (p - pc_centers).numpy(), rtol=0, atol=2e-5)
    # exact ties (duplicated node): the oracle's documented rule is "lower node index first"
    node[:, :, 7] = node[:, :, 3]
    o = oracle.cluster_assign(pc, node, k)
    assert not (o["min_k_idx"][:, :, 0] == 7).any()
    both = (o["min_k_idx"] == 3).any(axis=2) & (o["min_k_idx"] == 7).any(axis=2)
    pos3 = np.argmax(o["min_k_idx"] == 3, axis=2)
    pos7 = np.argmax(o["min_k_idx"] == 7, axis=2)
    assert (pos3[both] < pos7[both]).all()


def test_oracle_reproduces_committed_golden_vectors():
    """tests/golden/frustum_small.npz (tests/golden/make_frustum_golden.py): the oracle must keep producing the
    vectors the GPU parity tests are also checked against."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frustum_small.npz"))
    S, I, H, W = int(g["S"]), int(g["I"]), float(g["H"]), float(g["W"])
    for s in range(S):
        pts, pred, K = g["points"][s].astype(np.float64), g["pred"][s], g["K"][s]
        for is_2d, x, ev, sol in ((True, g["x4"][s], g["eval4"][s], g["solve4"][s]),
                                  (False, g["x6"][s], g["eval6"][s], g["solve6"][s])):
            P = 4 if is_2d else 6
            c, gr, A = oracle.evaluate(pts, pred, K, x, H, W, is_2d)
            np.testing.assert_allclose(np.concatenate([[c], gr, A.reshape(-1)]), ev, rtol=1e-12, atol=1e-12)
            ms = oracle.solve_multistart(pts, pred, K, g["inits"][s][:, 0], g["inits"][s][:, 1:4], H, W,
                                         (-5.0, -0.1, -10.0), (5.0, 0.1, 10.0), 500, is_2d)
            np.testing.assert_allclose(ms["params"][:, :P], sol[:, :P], rtol=0, atol=1e-9)
            np.testing.assert_allclose(ms["costs"], sol[:, 6], rtol=1e-9)
            for i in range(I):
                st = ms["stats"][i]
                assert [st["iterations"], st["unique_evals"], st["termination"]] == sol[i, 7:10].astype(int).tolist()
    ca = oracle.cluster_assign(g["ca_pc"], g["ca_node"], 3)
    np.testing.assert_array_equal(ca["min_k_idx"], g["ca_min_k_idx"])
    np.testing.assert_array_equal(ca["count"], g["ca_count"])
    np.testing.assert_array_equal(ca["cluster_mean"], g["ca_mean"])
    np.testing.assert_array_equal(ca["pc_decentered"], g["ca_decentered"])


def test_oracle_parity_tooling_options():
    """The oracle's parity-tooling switches (off by default): the Cholesky linear solver lands on the QR solution of a
    well-conditioned solve, the external-evaluation hook fed with the oracle's own sums reproduces the Cholesky run bit
    for bit, and the trace holds one record per evaluation with the decisions the statistics report."""
    smp = syn.make_sample(4300, n_points=1500)
    iy, pf, lf, _ = oracle.initial_guess(smp["points"], smp["pred"])
    ry, t = syn.make_inits(4300, iy, 2)
    args = (pf, lf, smp["K"], ry[0], t[0], smp["H"], smp["W"], syn.T_LB, syn.T_UB, 500, True)
    qr = oracle.solve(*args, want_residuals=False, trace_cap=400)
    ch = oracle.solve(*args, want_residuals=False, linear_solver=1, trace_cap=400)
    assert qr[3]["termination"] in (0, 1, 2) and len(qr[5]) == qr[3]["unique_evals"]
    assert qr[5][0, 10] == 0 and qr[5][-1, 12] == qr[3]["termination"]
    assert np.all(qr[5][:-1, 12] == -1)                       # only the last evaluation ends the solve
    assert int(qr[5][:, 11].sum()) == qr[3]["successful_steps"] + 1   # accepted evaluations = successful steps + the start
    np.testing.assert_allclose(ch[4], qr[4], rtol=0, atol=1e-6)

    def ext(x6):
        return oracle.evaluate(pf, lf, smp["K"], x6[:4], smp["H"], smp["W"], True)

    hy = oracle.solve(*args, linear_solver=1, ext_eval=ext, trace_cap=400)
    assert np.array_equal(hy[4], ch[4]) and hy[3] == ch[3] and np.array_equal(hy[5][:, :13], ch[5][:, :13])
    with pytest.raises(ValueError):
        oracle.solve(*args, ext_eval=ext)                     # the hook has no Jacobian rows: it needs linear_solver=1
