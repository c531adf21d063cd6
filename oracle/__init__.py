"""CPU oracles -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this
package.  The product path (deepi2p_b200/) never does; it fails loudly when its CUDA
library is missing instead of falling back to anything here.

PARITY UNPINNED for the solver: the reference's solvePGivenK delegates to Ceres, which is
not available offline, and the reference has no golden vectors (SURVEY.md 8c).  See the
header of frustum_oracle.cpp for what is restated and from where.
"""
import ctypes
import math
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))
_libs = {}
_libs_lock = threading.Lock()        # the first callers may be worker threads: one of them builds

STAT_FIELDS = ("iterations", "successful_steps", "unique_evals", "cost_evals", "jac_evals",
               "line_search_steps", "termination", "reserved")


def _lib(name):
    with _libs_lock:
        if name not in _libs:
            out = _build.build()
            _libs[name] = ctypes.CDLL(os.path.join(out, name))
        return _libs[name]


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


def _prep_points(points):
    pts = np.ascontiguousarray(np.asarray(points, dtype=np.float64))
    if pts.ndim != 2 or pts.shape[0] != 3:
        raise ValueError("points must be 3xN")
    return pts


EXT_EVAL = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.POINTER(ctypes.c_double),
                            ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                            ctypes.POINTER(ctypes.c_double))


def solve(points, labels, K, init_y_angle, init_T, H, W, t_lb, t_ub, max_iter=500, is_2d=True,
          want_residuals=True, linear_solver=0, ext_eval=None, trace_cap=0):
    """Oracle for FrustumRegistration.solvePGivenK (registration.cpp:9-186).

    Returns (P 4x4, final_cost, residuals, stats dict, params[6]) (+ trace [n,16] as a sixth element when
    trace_cap > 0).  Parity-tooling options (defaults = the reference behaviour): linear_solver=1 solves the damped
    normal equations by Cholesky (the CUDA kernel's arithmetic) instead of Householder QR; ext_eval(x6) -> (cost,
    g[P], JtJ[P,P]) replaces the dual-number evaluation (needs linear_solver=1; residuals are then not returned).
    """
    lib = _lib("libfrustum_oracle.so")
    pts = _prep_points(points)
    n = pts.shape[1]
    lab = np.ascontiguousarray(np.asarray(labels).astype(np.int32))
    K9 = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(9))
    T = np.ascontiguousarray(np.asarray(init_T, dtype=np.float64).reshape(3))
    lb = np.ascontiguousarray(np.asarray(t_lb, dtype=np.float64).reshape(3))
    ub = np.ascontiguousarray(np.asarray(t_ub, dtype=np.float64).reshape(3))
    P16 = np.zeros(16)
    cost = ctypes.c_double(0.0)
    lib.frustum_oracle_num_residuals.restype = ctypes.c_int64
    rows = lib.frustum_oracle_num_residuals(_p(lab, ctypes.c_int32), ctypes.c_int64(n))
    want_residuals = want_residuals and ext_eval is None
    res = np.zeros(rows) if want_residuals else None
    stats = np.zeros(8, dtype=np.int32)
    params = np.zeros(6)
    Pn = 4 if is_2d else 6
    cb = None
    if ext_eval is not None:
        def _cb(_user, x6, c_out, g_out, A_out):
            c, g, A = ext_eval(np.array([x6[j] for j in range(6)]))
            c_out[0] = float(c)
            for j in range(Pn):
                g_out[j] = float(g[j])
                for k in range(Pn):
                    A_out[j * Pn + k] = float(A[j][k])
            return 0
        cb = EXT_EVAL(_cb)
    trace = np.zeros((max(int(trace_cap), 1), 16)) if trace_cap > 0 else None
    rc = lib.frustum_oracle_solve_ex(
        _p(pts, ctypes.c_double), _p(lab, ctypes.c_int32), ctypes.c_int64(n), _p(K9, ctypes.c_double),
        ctypes.c_double(float(init_y_angle)), _p(T, ctypes.c_double), ctypes.c_double(float(H)),
        ctypes.c_double(float(W)), _p(lb, ctypes.c_double), _p(ub, ctypes.c_double),
        ctypes.c_int(int(max_iter)), ctypes.c_int(1 if is_2d else 0), _p(P16, ctypes.c_double),
        ctypes.byref(cost), _p(res, ctypes.c_double) if want_residuals else None,
        _p(stats, ctypes.c_int32), _p(params, ctypes.c_double), ctypes.c_int(int(linear_solver)),
        cb if cb is not None else ctypes.cast(None, EXT_EVAL), None,
        _p(trace, ctypes.c_double) if trace is not None else None, ctypes.c_int(int(trace_cap)))
    if rc != 0:
        raise ValueError("frustum_oracle_solve_ex: ext_eval needs linear_solver=1")
    out = (P16.reshape(4, 4), cost.value, res, dict(zip(STAT_FIELDS, stats.tolist())), params)
    if trace is not None:
        out = out + (trace[trace[:, 15] > 0],)
    return out


def evaluate(points, labels, K, x, H, W, is_2d=True):
    """cost, g = J^T r, JtJ at parameter vector x (dual-number evaluation)."""
    lib = _lib("libfrustum_oracle.so")
    pts = _prep_points(points)
    n = pts.shape[1]
    lab = np.ascontiguousarray(np.asarray(labels).astype(np.int32))
    K9 = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(9))
    P = 4 if is_2d else 6
    xx = np.zeros(6)
    xx[:P] = np.asarray(x, dtype=np.float64)[:P]
    cost = ctypes.c_double(0.0)
    g = np.zeros(P)
    JtJ = np.zeros((P, P))
    lib.frustum_oracle_evaluate(
        _p(pts, ctypes.c_double), _p(lab, ctypes.c_int32), ctypes.c_int64(n), _p(K9, ctypes.c_double),
        _p(xx, ctypes.c_double), ctypes.c_double(float(H)), ctypes.c_double(float(W)),
        ctypes.c_int(1 if is_2d else 0), ctypes.byref(cost), _p(g, ctypes.c_double),
        _p(JtJ, ctypes.c_double), None)
    return cost.value, g, JtJ


def residuals(points, labels, K, x, H, W, is_2d=True):
    """Loss-corrected residual vector at parameter vector x (what Problem::Evaluate returns,
    registration.cpp:150-155)."""
    lib = _lib("libfrustum_oracle.so")
    pts = _prep_points(points)
    n = pts.shape[1]
    lab = np.ascontiguousarray(np.asarray(labels).astype(np.int32))
    K9 = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(9))
    P = 4 if is_2d else 6
    xx = np.zeros(6)
    xx[:P] = np.asarray(x, dtype=np.float64)[:P]
    lib.frustum_oracle_num_residuals.restype = ctypes.c_int64
    rows = lib.frustum_oracle_num_residuals(_p(lab, ctypes.c_int32), ctypes.c_int64(n))
    res = np.zeros(rows)
    cost = ctypes.c_double(0.0)
    g = np.zeros(P)
    JtJ = np.zeros((P, P))
    lib.frustum_oracle_evaluate(
        _p(pts, ctypes.c_double), _p(lab, ctypes.c_int32), ctypes.c_int64(n), _p(K9, ctypes.c_double),
        _p(xx, ctypes.c_double), ctypes.c_double(float(H)), ctypes.c_double(float(W)),
        ctypes.c_int(1 if is_2d else 0), ctypes.byref(cost), _p(g, ctypes.c_double),
        _p(JtJ, ctypes.c_double), _p(res, ctypes.c_double))
    return res, cost.value


def wrap_in_pi(x):
    """registration_lsq.py:189-193."""
    x = math.fmod(x + math.pi, math.pi * 2)
    if x < 0:
        x += math.pi * 2
    return x - math.pi


def ry_matrix(a):
    """Rotation about +y (data/augmentation.py:18-20 convention)."""
    c, s = math.cos(a), math.sin(a)
    return np.array([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])


def initial_guess(points, pred):
    """get_initial_guess (registration_lsq.py:196-220): heading of the mean predicted-inside
    point, and the 'front' filter.  Returns (init_y_angle, points_front, pred_front, mask)."""
    pts = np.asarray(points, dtype=np.float64)
    pred = np.asarray(pred)
    inside = pred == 1
    mean = pts[:, inside].mean(axis=1)
    init_y = wrap_in_pi(math.atan2(mean[2], mean[0]) - math.pi / 2)
    R1 = ry_matrix(init_y)
    rp = R1 @ pts
    zmin = rp[2, inside].min()
    mask = rp[2, :] > zmin - 10
    return init_y, pts[:, mask], pred[mask], mask


def solve_multistart(points, labels, K, init_ry, init_t, H, W, t_lb, t_ub, max_iter=500, is_2d=True,
                     threads=1, linear_solver=0):
    """Multi-start driver (registration_lsq.py:142-186) over MATERIALISED inits
    init_ry [I], init_t [I,3].  Deterministic arg-min (lowest index wins ties; the reference's
    winner is racy).  Returns dict(P, cost, best, costs[I], params[I,6], stats[list])."""
    init_ry = np.asarray(init_ry, dtype=np.float64)
    init_t = np.asarray(init_t, dtype=np.float64)
    I = init_ry.shape[0]

    def one(i):
        return solve(points, labels, K, init_ry[i], init_t[i], H, W, t_lb, t_ub, max_iter, is_2d,
                     want_residuals=False, linear_solver=linear_solver)

    if threads > 1:
        with ThreadPoolExecutor(threads) as ex:
            outs = list(ex.map(one, range(I)))
    else:
        outs = [one(i) for i in range(I)]
    costs = np.array([o[1] for o in outs])
    best = int(np.argmin(costs))       # first minimum
    return dict(P=outs[best][0], cost=float(costs[best]), best=best, costs=costs,
                params=np.stack([o[4] for o in outs]), stats=[o[3] for o in outs],
                poses=np.stack([o[0] for o in outs]))


def inside_img_mask(pc, P, K, H, W):
    """get_inside_img_mask (evaluation/registration_lsq.py:67-84), restated line by line."""
    pc = np.asarray(pc, dtype=np.float64)
    P = np.asarray(P, dtype=np.float64)
    K = np.asarray(K, dtype=np.float64)
    homo = np.concatenate((pc, np.ones((1, pc.shape[1]), dtype=pc.dtype)), axis=0)
    P_points = np.dot(P, homo)[0:3, :]
    K_pc = np.dot(K, P_points)
    with np.errstate(divide="ignore", invalid="ignore"):
        pxpy = K_pc[0:2, :] / K_pc[2:3, :]
    x_in = np.logical_and(pxpy[0:1, :] >= 0, pxpy[0:1, :] <= W - 1)
    y_in = np.logical_and(pxpy[1:2, :] >= 0, pxpy[1:2, :] <= H - 1)
    z_in = P_points[2:3, :] > 0.1
    return np.logical_and(np.logical_and(x_in, y_in), z_in)[0]


def pose_diff(P_pred, P_gt):
    """get_P_diff (evaluation/registration_lsq.py:87-95): (t_diff, angles_diff in degrees)."""
    from scipy.spatial.transform import Rotation
    P_diff = np.dot(np.linalg.inv(P_pred), P_gt)
    t_diff = np.linalg.norm(P_diff[0:3, 3])
    angles = np.sum(np.abs(Rotation.from_matrix(P_diff[0:3, 0:3]).as_euler('xzy', degrees=True)))
    return t_diff, angles


def index_max(data, index, K):
    """Oracle for index_max.forward_* (index_max.cpp:73-112)."""
    lib = _lib("libops_oracle.so")
    data = np.ascontiguousarray(np.asarray(data, dtype=np.float32))
    index = np.ascontiguousarray(np.asarray(index, dtype=np.int32))
    B, C, N = data.shape
    out = np.zeros((B, C, K), dtype=np.int32)
    scratch = np.zeros((B, C, K), dtype=np.float32)
    rc = lib.index_max_oracle(_p(data, ctypes.c_float), _p(index, ctypes.c_int32), _p(out, ctypes.c_int32),
                              ctypes.c_int64(B), ctypes.c_int64(C), ctypes.c_int64(N), ctypes.c_int64(K),
                              _p(scratch, ctypes.c_float))
    if rc != 0:
        raise ValueError("index out of [0,K)")
    return out


def ball_query(dist, radius, K):
    """Oracle for ball_query.forward_cuda_shared_mem (ball_query_cuda.cu:11-50)."""
    lib = _lib("libops_oracle.so")
    dist = np.ascontiguousarray(np.asarray(dist, dtype=np.float32))
    B, M, N = dist.shape
    out = np.zeros((B, M, K), dtype=np.int32)
    lib.ball_query_oracle(_p(dist, ctypes.c_float), ctypes.c_float(float(radius)), _p(out, ctypes.c_int32),
                          ctypes.c_int64(B), ctypes.c_int64(M), ctypes.c_int64(N), ctypes.c_int64(K))
    return out


def ball_query_xyz(points, nodes, radius, K):
    """Oracle for the coordinate-based radius search: float32 distance ((dx*dx + dy*dy) + dz*dz) <= r*r, then
    the ball_query rule (ball_query_cuda.cu:11-50).  points [B,3,N], nodes [B,3,M]."""
    p = np.asarray(points, dtype=np.float32)
    q = np.asarray(nodes, dtype=np.float32)
    d = p[:, :, None, :] - q[:, :, :, None]                     # [B,3,M,N], point - node as in the kernel
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    r2 = np.float32(radius) * np.float32(radius)
    B, M, N = d2.shape
    out = np.zeros((B, M, K), dtype=np.int32)
    for b in range(B):
        for m in range(M):
            hits = np.nonzero(d2[b, m] <= r2)[0][:K]
            if len(hits):
                out[b, m] = [hits[i] if i < len(hits) else hits[(i - len(hits)) % len(hits)] for i in range(K)]
    return out


def cluster_assign(pc, node, k):
    """Oracle for cluster_assign_forward: the clustering front-end of models/networks_pc.py:60-85.

    pc [B,3,N], node [B,3,M].  Ordering key = float32 ((dx*dx + dy*dy) + dz*dz) (numpy float32 arithmetic has no
    fma), stable sort => ties go to the lower node index (torch.topk leaves them unspecified; sqrt is monotone).
    Sums are exact fixed point (rint(x * 2^24) in int64), mean = float32(sum * 2^-24) / (float32(count) + 1e-5f)."""
    p = np.asarray(pc, dtype=np.float32)
    q = np.asarray(node, dtype=np.float32)
    B, _, N = p.shape
    M = q.shape[2]
    d = p[:, :, :, None] - q[:, :, None, :]                      # [B,3,N,M], point - node
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    order = np.argsort(d2, axis=2, kind="stable")[:, :, :k].astype(np.int32)
    min_idx = order[:, :, 0]
    count = np.zeros((B, M), dtype=np.int32)
    sums = np.zeros((B, 3, M), dtype=np.int64)
    finite = np.isfinite(p).all(axis=1)                           # non-finite points join no count / sum
    fixed = np.rint(np.where(finite[:, None, :], p, 0).astype(np.float64) * 16777216.0).astype(np.int64)
    for b in range(B):
        np.add.at(count[b], min_idx[b][finite[b]], 1)
        for a in range(3):
            np.add.at(sums[b, a], min_idx[b][finite[b]], fixed[b, a][finite[b]])
    num = (sums.astype(np.float64) * (1.0 / 16777216.0)).astype(np.float32)
    mean = num / (count.astype(np.float32)[:, None, :] + np.float32(1e-5))
    centers = np.take_along_axis(mean, np.broadcast_to(min_idx[:, None, :].astype(np.int64), (B, 3, N)), axis=2)
    return dict(min_k_idx=order, min_idx=min_idx.copy(), count=count, cluster_mean=mean.astype(np.float32),
                pc_centers=centers.astype(np.float32), pc_decentered=(p - centers).astype(np.float32))
