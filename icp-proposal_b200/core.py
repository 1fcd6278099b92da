"""Thin numpy-facing wrappers of the libicpcuda.so handles (one class per C-ABI handle type).

Everything here is argument marshalling; all arithmetic happens in the CUDA library. There is no CPU
fallback: constructing a Context without a CUDA device raises IcpCudaError.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, dptr, f64, i32, iptr

THETA0 = 10  # theta = [s, t3, rot3, c3, alpha_K]


class Context:
    def __init__(self, device=0):
        self.lib = _lib.load()
        self.h = C.c_void_p()
        check(self.lib.icp_ctx_create(int(device), C.byref(self.h)))
        self.device = int(device)

    def version(self):
        buf = C.create_string_buffer(256)
        self.lib.icp_version(self.h, buf, 256)
        return buf.value.decode()

    def synchronize(self):
        check(self.lib.icp_ctx_synchronize(self.h), self.h)

    def fp64_peak(self):
        out = np.zeros(2)
        check(self.lib.icp_debug_fp64_peak(self.h, dptr(out)), self.h)
        return {"dfma_tflops": float(out[0]), "dmma_tflops": float(out[1])}

    def i8_peak(self, ctas=296, iters=400):
        """INT8 tensor-core TOP/s of the rank update's MMA tile (tcgen05.mma kind::i8, 128 x 112 x 32, operands in shared
        memory, accumulator in TMEM), `ctas` CTAs each running `iters` passes over a 608-row image (icp_debug_i8_gram)."""
        a = np.ones((608, 128), np.int8)
        ms = C.c_double(0)
        check(self.lib.icp_debug_i8_gram(self.h, 608, a.ctypes.data, None, int(iters), int(ctas), C.byref(ms)), self.h)
        return 2.0 * 128 * 112 * 608 * iters * ctas / (ms.value * 1e-3) / 1e12

    def l2_bandwidth(self, working_set_bytes=32 << 20):
        """GB/s of L2 -> SM reads over an L2-resident working set (icp_debug_l2_bandwidth)."""
        out = C.c_double(0)
        check(self.lib.icp_debug_l2_bandwidth(self.h, int(working_set_bytes), C.byref(out)), self.h)
        return out.value

    def factor(self, M, b, theta_post=None, theta_other=None, step=1.0, ymean=False):
        """Cholesky factorisation of C posterior matrices M (C x K x K) with right-hand sides b on the device path the
        posterior pipeline takes at rank K (icp_debug_factor): L, the mean slot (mu, or y = L^-1 b when ymean), the
        backward-form |L^T (w - mu)|^2 of theta_post -> theta_other (None without thetas) and the status words."""
        M = f64(M); c, K = M.shape[0], M.shape[1]
        b = f64(b).reshape(c, K)
        L = np.zeros((c, K, K)); mean = np.empty((c, K)); st = np.empty(c, np.int32)
        q = np.empty(c) if theta_post is not None else None
        tp = None if q is None else f64(theta_post).reshape(c, K + THETA0)
        to = None if q is None else f64(theta_other).reshape(c, K + THETA0)
        check(self.lib.icp_debug_factor(self.h, c, K, dptr(M), dptr(b), None if tp is None else dptr(tp), None if to is None else dptr(to),
                                        float(step), int(bool(ymean)), dptr(L), dptr(mean), None if q is None else dptr(q), iptr(st)), self.h)
        return L, mean, q, st

    def philox(self, seed, chain, step, block):
        out = (C.c_uint32 * 4)()
        check(self.lib.icp_debug_philox(self.h, seed, chain, step, block, out), self.h)
        return np.array(list(out), dtype=np.uint32)

    def close(self):
        if self.h:
            self.lib.icp_ctx_destroy(self.h)
            self.h = None


class Model:
    """StatisticalMeshModel: reference mesh + low-rank GP (mean deformation, basis U, variances)."""

    def __init__(self, ctx: Context, ref, cells, basis, variance, mean_def=None):
        self.ctx, self.lib = ctx, ctx.lib
        self.ref = f64(ref).reshape(-1, 3)
        self.cells = i32(cells).reshape(-1, 3)
        self.variance = f64(variance).reshape(-1)
        self.N, self.T, self.K = len(self.ref), len(self.cells), len(self.variance)
        self.basis = f64(basis)
        if self.basis.shape != (3 * self.N, self.K):
            raise ValueError(f"basis must be (3N, K) = {(3 * self.N, self.K)}, got {self.basis.shape}")
        self.mean_def = None if mean_def is None else f64(mean_def).reshape(-1)
        self.h = C.c_void_p()
        check(self.lib.icp_model_create(ctx.h, self.N, self.T, self.K, dptr(self.ref),
                                        None if self.mean_def is None else dptr(self.mean_def), dptr(self.basis),
                                        dptr(self.variance), iptr(self.cells), C.byref(self.h)), ctx.h)

    @property
    def rank(self):
        return self.K

    def theta(self, alpha=None, translation=(0, 0, 0), rotation=(0, 0, 0), center=None, scale=1.0):
        """Packs ModelFittingParameters.allParameters (ModelFittingParameters.scala:64)."""
        th = np.zeros(self.K + THETA0)
        th[0] = scale
        th[1:4] = translation
        th[4:7] = rotation
        th[7:10] = self.ref.mean(0) if center is None else center
        if alpha is not None:
            th[10:] = alpha
        return th

    def _theta(self, theta):
        th = f64(theta).reshape(-1, self.K + THETA0)
        return th, len(th)

    def reconstruct(self, theta):
        th, c = self._theta(theta)
        out = np.empty((c, self.N, 3))
        check(self.lib.icp_reconstruct(self.h, c, dptr(th), dptr(out)), self.ctx.h)
        return out

    def vertex_normals(self, theta):
        th, c = self._theta(theta)
        out = np.empty((c, self.N, 3))
        check(self.lib.icp_vertex_normals(self.h, c, dptr(th), dptr(out)), self.ctx.h)
        return out

    def closest_point_surface(self, theta, q):
        th, c = self._theta(theta)
        q = f64(q).reshape(-1, 3)
        n = len(q)
        tri = np.empty((c, n), np.int32); feat = np.empty((c, n), np.int32); cp = np.empty((c, n, 3)); d2 = np.empty((c, n))
        check(self.lib.icp_model_closest_point_surface(self.h, c, dptr(th), n, dptr(q), iptr(tri), iptr(feat), dptr(cp),
                                                       dptr(d2)), self.ctx.h)
        return tri, feat, cp, d2

    def closest_vertex(self, theta, q):
        th, c = self._theta(theta)
        q = f64(q).reshape(-1, 3)
        n = len(q)
        ids = np.empty((c, n), np.int32); d2 = np.empty((c, n))
        check(self.lib.icp_model_closest_vertex(self.h, c, dptr(th), n, dptr(q), iptr(ids), dptr(d2)), self.ctx.h)
        return ids, d2

    def boundary_flags(self):
        f = np.zeros(self.N, np.uint8)
        check(self.lib.icp_model_boundary_flags(self.h, f.ctypes.data_as(_lib._bp)))
        return f.astype(bool)

    def prior(self, theta):
        th, c = self._theta(theta)
        out = np.empty(c)
        check(self.lib.icp_eval_prior(self.h, c, dptr(th), dptr(out)), self.ctx.h)
        return out

    def close(self):
        if self.h:
            self.lib.icp_model_destroy(self.h)
            self.h = None


class Target:
    """TriangleMesh3D with its device query structures."""

    def __init__(self, ctx: Context, verts, cells):
        self.ctx, self.lib = ctx, ctx.lib
        self.verts = f64(verts).reshape(-1, 3)
        self.cells = i32(cells).reshape(-1, 3)
        self.h = C.c_void_p()
        check(self.lib.icp_target_create(ctx.h, len(self.verts), len(self.cells), dptr(self.verts), iptr(self.cells),
                                         C.byref(self.h)), ctx.h)

    def closest_point_surface(self, q):
        q = f64(q).reshape(-1, 3)
        n = len(q)
        tri = np.empty(n, np.int32); feat = np.empty(n, np.int32); cp = np.empty((n, 3)); d2 = np.empty(n)
        check(self.lib.icp_closest_point_surface(self.h, n, dptr(q), iptr(tri), iptr(feat), dptr(cp), dptr(d2)), self.ctx.h)
        return tri, feat, cp, d2

    def closest_vertex(self, q):
        q = f64(q).reshape(-1, 3)
        n = len(q)
        ids = np.empty(n, np.int32); d2 = np.empty(n)
        check(self.lib.icp_closest_vertex(self.h, n, dptr(q), iptr(ids), dptr(d2)), self.ctx.h)
        return ids, d2

    def boundary_flags(self):
        f = np.zeros(len(self.verts), np.uint8)
        check(self.lib.icp_target_boundary_flags(self.h, f.ctypes.data_as(_lib._bp)))
        return f.astype(bool)

    def close(self):
        if self.h:
            self.lib.icp_target_destroy(self.h)
            self.h = None


class IcpProposal:
    """Device side of NonRigidIcpProposal (api/sampling/proposals/NonRigidIcpProposal.scala)."""

    def __init__(self, model: Model, target: Target, step_length, tangential_noise, noise_along_normal, direction,
                 boundary_aware, model_point_ids, target_points, factor=_lib.FACTOR_CHOLESKY,
                 rank_update=_lib.RANK_UPDATE_FP64):
        self.model, self.target, self.lib, self.ctx = model, target, model.lib, model.ctx
        self.ids = i32(np.asarray(model_point_ids).reshape(-1))
        self.tp = f64(np.asarray(target_points, dtype=np.float64).reshape(-1, 3))
        self.params = _lib.ProposalParams(step_length, tangential_noise, noise_along_normal, int(direction), int(boundary_aware),
                                          int(factor), int(rank_update))
        self.h = C.c_void_p()
        check(self.lib.icp_proposal_create(model.h, target.h, C.byref(self.params), iptr(self.ids), len(self.ids),
                                           dptr(self.tp), len(self.tp), C.byref(self.h)), self.ctx.h)

    def posterior(self, theta, want_M=True):
        th, c = self.model._theta(theta)
        K = self.model.K
        mu = np.empty((c, K)); M = np.empty((c, K, K)) if want_M else None; n = np.empty(c, np.int32)
        check(self.lib.icp_posterior(self.h, c, dptr(th), dptr(mu), None if M is None else dptr(M), iptr(n)), self.ctx.h)
        return mu, M, n

    def propose(self, theta, z):
        th, c = self.model._theta(theta)
        z = f64(z).reshape(c, self.model.K)
        out = np.empty_like(th)
        check(self.lib.icp_propose(self.h, c, dptr(th), dptr(z), dptr(out)), self.ctx.h)
        return out

    def log_transition(self, frm, to):
        f, c = self.model._theta(frm)
        t, c2 = self.model._theta(to)
        assert c == c2
        out = np.empty(c)
        check(self.lib.icp_log_transition(self.h, c, dptr(f), dptr(t), dptr(out)), self.ctx.h)
        return out

    def clear_cache(self):
        check(self.lib.icp_proposal_clear_cache(self.h), self.ctx.h)

    def close(self):
        if self.h:
            self.lib.icp_proposal_destroy(self.h)
            self.h = None


def std_icp_iteration(model: Model, target: Target, direction, model_point_ids, target_points, sigma2, step_length, alpha):
    ids = i32(np.asarray(model_point_ids).reshape(-1))
    tp = f64(np.asarray(target_points, dtype=np.float64).reshape(-1, 3))
    a = f64(alpha).reshape(-1, model.K)
    out = np.empty_like(a)
    check(model.lib.icp_std_icp_iteration(model.h, target.h, int(direction), iptr(ids), len(ids), dptr(tp), len(tp),
                                          float(sigma2), float(step_length), len(a), dptr(a), dptr(out)), model.ctx.h)
    return out


def std_icp_iteration_theta(model: Model, target: Target, direction, model_point_ids, target_points, sigma2, step_length, theta):
    """icp_std_icp_iteration_theta: one deterministic ICP iteration under the rigid transform carried by theta -> alpha_out."""
    ids = i32(np.asarray(model_point_ids).reshape(-1))
    tp = f64(np.asarray(target_points, dtype=np.float64).reshape(-1, 3))
    th, c = model._theta(theta)
    out = np.empty((c, model.K))
    check(model.lib.icp_std_icp_iteration_theta(model.h, target.h, int(direction), iptr(ids), len(ids), dptr(tp), len(tp),
                                                float(sigma2), float(step_length), c, dptr(th), dptr(out)), model.ctx.h)
    return out


class StdIcp:
    """Device-resident IcpBasedSurfaceFitting.runfitting for batches of independent fits (icp_std_icp_*)."""

    def __init__(self, model: Model, target: Target, model_point_ids, target_points, step_length=1.0,
                 direction=_lib.MODEL_SAMPLING, max_fits=1):
        self.model, self.target, self.lib, self.ctx = model, target, model.lib, model.ctx
        self.ids = i32(np.asarray(model_point_ids).reshape(-1))
        self.tp = f64(np.asarray(target_points, dtype=np.float64).reshape(-1, 3))
        self.max_fits = int(max_fits)
        self.h = C.c_void_p()
        check(self.lib.icp_std_icp_create(model.h, target.h, iptr(self.ids), len(self.ids), dptr(self.tp), len(self.tp),
                                          float(step_length), int(direction), self.max_fits, C.byref(self.h)), self.ctx.h)

    def run(self, theta0, sigma2, num_iterations, directions=None, seed=1024, fit_id_offset=0, log=True):
        """theta0 (C, K + 10); sigma2: iterationSeq; directions (iters, C) or None. Returns dict(alpha_final (C, K), status (C,),
        iterations_done (C,), and with log=True log_alpha (iters, C, K) and log_direction (iters, C))."""
        th, c = self.model._theta(theta0)
        s2 = f64(np.atleast_1d(sigma2))
        K, iters = self.model.K, len(s2) * (int(num_iterations) + 1)
        io = _lib.StdIcpIO()
        io.seed, io.fit_id_offset = int(seed), int(fit_id_offset)
        d = None
        if directions is not None:
            d = i32(directions).reshape(iters, c)
            io.directions = d.ctypes.data
        out = dict(alpha_final=np.empty((c, K)), status=np.zeros(c, np.int32), iterations_done=np.zeros(c, np.int32))
        io.alpha_final, io.status, io.iterations_done = (out[k].ctypes.data for k in ("alpha_final", "status", "iterations_done"))
        if log:
            out["log_alpha"], out["log_direction"] = np.empty((iters, c, K)), np.empty((iters, c), np.int32)
            io.log_alpha, io.log_direction = out["log_alpha"].ctypes.data, out["log_direction"].ctypes.data
        check(self.lib.icp_std_icp_run(self.h, c, dptr(th), len(s2), dptr(s2), int(num_iterations), C.byref(io)), self.ctx.h)
        return out

    def run_device(self, C_, theta0_ptr, sigma2, num_iterations, directions=0, seed=1024, fit_id_offset=0, alpha_final=0,
                   log_alpha=0, log_direction=0, status=0, iterations_done=0, async_=False):
        """All pointers are raw device addresses (e.g. torch.Tensor.data_ptr()); sigma2 is a host sequence."""
        s2 = f64(np.atleast_1d(sigma2))
        io = _lib.StdIcpIO()
        io.seed, io.fit_id_offset, io.directions = int(seed), int(fit_id_offset), directions or None
        io.alpha_final, io.log_alpha, io.log_direction = alpha_final or None, log_alpha or None, log_direction or None
        io.status, io.iterations_done = status or None, iterations_done or None
        check(self.lib.icp_std_icp_run_device(self.h, int(C_), theta0_ptr, len(s2), dptr(s2), int(num_iterations), C.byref(io),
                                              int(async_)), self.ctx.h)

    def last_run_stats(self):
        """(device milliseconds, kernel launches) of the last run."""
        ms = C.c_double(0); n = C.c_int64(0)
        check(self.lib.icp_std_icp_last_run_stats(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def close(self):
        if self.h:
            self.lib.icp_std_icp_destroy(self.h)
            self.h = None


class Evaluator:
    """Device side of the DistributionEvaluators (api/sampling/evaluators/*.scala)."""

    def __init__(self, model: Model, target: Target, kind, mode=_lib.MODEL_TO_TARGET, use_prior=True, p0=0.0, p1=1.0,
                 p2=1.0, model_point_ids=(), target_points=()):
        self.model, self.target, self.lib, self.ctx = model, target, model.lib, model.ctx
        self.ids = i32(np.asarray(model_point_ids).reshape(-1))
        self.tp = f64(np.asarray(target_points, dtype=np.float64).reshape(-1, 3))
        self.params = _lib.EvaluatorParams(int(kind), int(mode), int(bool(use_prior)), 0, p0, p1, p2)
        self.h = C.c_void_p()
        check(self.lib.icp_evaluator_create(model.h, target.h, C.byref(self.params), iptr(self.ids), len(self.ids),
                                            dptr(self.tp), len(self.tp), C.byref(self.h)), self.ctx.h)

    def log_value(self, theta, with_status=False):
        """-> (C, 3) array of {product, prior, distance} log-values."""
        th, c = self.model._theta(theta)
        out = np.empty((c, 3)); st = np.zeros(c, np.int32)
        check(self.lib.icp_eval_log_value(self.h, c, dptr(th), dptr(out), iptr(st)), self.ctx.h)
        return (out, st) if with_status else out

    def close(self):
        if self.h:
            self.lib.icp_evaluator_destroy(self.h)
            self.h = None


def registration_metrics(model: Model, target: Target, theta):
    th, c = model._theta(theta)
    out = np.empty((c, 4))
    check(model.lib.icp_registration_metrics(model.h, target.h, c, dptr(th), dptr(out)), model.ctx.h)
    return out


def dice_coefficient(model: Model, target: Target, theta, unit_samples=None, n_samples=10000, seed=0):
    """icp_dice_coefficient: MeshMetrics.diceCoefficient(transformedMesh(theta), target) per parameter vector."""
    th, c = model._theta(theta)
    out = np.empty(c)
    us = None
    if unit_samples is not None:
        us = f64(unit_samples).reshape(-1, 3)
        n_samples = len(us)
    check(model.lib.icp_dice_coefficient(model.h, target.h, c, dptr(th), int(n_samples), dptr(us) if us is not None else None,
                                         int(seed), dptr(out)), model.ctx.h)
    return out


def _kernel_terms(terms):
    """terms: iterable of (scale, sigma, A) with A a 3 x 3 matrix or None (identity)."""
    arr = (_lib.KernelTerm * len(terms))()
    for t, (scale, sigma, a) in zip(arr, terms):
        t.scale, t.sigma = float(scale), float(sigma)
        t.A[:] = list(np.asarray(np.eye(3) if a is None else a, float).reshape(9))
    return arr


def gpmm_kernel_matrix(ctx: "Context", x, y, terms):
    """icp_gpmm_kernel_matrix: (3 nx) x (3 ny) matrix of the Gaussian-mixture matrix-valued kernel."""
    x, y = f64(x).reshape(-1, 3), f64(y).reshape(-1, 3)
    out = np.empty((3 * len(x), 3 * len(y)))
    arr = _kernel_terms(terms)
    check(ctx.lib.icp_gpmm_kernel_matrix(ctx.h, len(x), dptr(x), len(y), dptr(y), arr, len(arr), dptr(out)), ctx.h)
    return out


def gpmm_eigen_psd(ctx: "Context", A, n_top):
    """icp_gpmm_eigen_psd: (w descending, V n x n_top) of a symmetric positive semi-definite matrix, on the device."""
    A = f64(A)
    n = len(A)
    if A.shape != (n, n):
        raise ValueError("A must be square")
    w, V = np.empty(n_top), np.empty((n, n_top))
    check(ctx.lib.icp_gpmm_eigen_psd(ctx.h, n, dptr(A), int(n_top), dptr(w), dptr(V)), ctx.h)
    return w, V


def gpmm_nystrom_extend(ctx: "Context", pts, nys_pts, terms, V, w):
    """icp_gpmm_nystrom_extend: (basis 3N x rank, variance rank) from the leading eigenpairs (V, w) of the Nystrom kernel matrix."""
    pts, nys = f64(pts).reshape(-1, 3), f64(nys_pts).reshape(-1, 3)
    V, w = f64(V), f64(w)
    rank = len(w)
    if V.shape != (3 * len(nys), rank):
        raise ValueError("V must be (3 m) x rank")
    basis, var = np.empty((3 * len(pts), rank)), np.empty(rank)
    arr = _kernel_terms(terms)
    check(ctx.lib.icp_gpmm_nystrom_extend(ctx.h, len(pts), dptr(pts), len(nys), dptr(nys), arr, len(arr), rank, dptr(V), dptr(w),
                                          dptr(basis), dptr(var)), ctx.h)
    return basis, var


def _face_kernel(levels, scales, symmetric_weight, plain_weight):
    fk = _lib.FaceKernel()
    fk.n_levels = len(levels)
    for i, (l, sc) in enumerate(zip(levels, scales)):
        fk.level[i], fk.scale[i] = int(l), float(sc)
    fk.symmetric_weight, fk.plain_weight = float(symmetric_weight), float(plain_weight)
    return fk


def _opt_weights(w, n_levels, n):
    if w is None:
        return None, None
    w = f64(w)
    if w.shape != (n_levels, n):
        raise ValueError("region weights must be n_levels x n_points")
    return w, dptr(w)


def gpmm_face_kernel_matrix(ctx: "Context", x, y, levels, scales, symmetric_weight=0.7, plain_weight=0.3, wx=None, wy=None, wy_mirror=None):
    """icp_gpmm_face_kernel_matrix: (3 nx) x (3 ny) matrix of the symmetrised multiscale B-spline kernel (apps/bfm/FaceKernel.scala)."""
    x, y = f64(x).reshape(-1, 3), f64(y).reshape(-1, 3)
    out = np.empty((3 * len(x), 3 * len(y)))
    fk = _face_kernel(levels, scales, symmetric_weight, plain_weight)
    (a, pa), (b, pb), (c, pc) = _opt_weights(wx, len(levels), len(x)), _opt_weights(wy, len(levels), len(y)), _opt_weights(wy_mirror, len(levels), len(y))
    check(ctx.lib.icp_gpmm_face_kernel_matrix(ctx.h, len(x), dptr(x), pa, len(y), dptr(y), pb, pc, C.byref(fk), dptr(out)), ctx.h)
    return out


def gpmm_face_nystrom_extend(ctx: "Context", pts, nys_pts, levels, scales, V, w, symmetric_weight=0.7, plain_weight=0.3, w_pts=None,
                             w_nys=None, w_nys_mirror=None):
    """icp_gpmm_face_nystrom_extend: (basis 3N x rank, variance rank) for the face kernel."""
    pts, nys = f64(pts).reshape(-1, 3), f64(nys_pts).reshape(-1, 3)
    V, w = f64(V), f64(w)
    rank = len(w)
    if V.shape != (3 * len(nys), rank):
        raise ValueError("V must be (3 m) x rank")
    basis, var = np.empty((3 * len(pts), rank)), np.empty(rank)
    fk = _face_kernel(levels, scales, symmetric_weight, plain_weight)
    (a, pa), (b, pb), (c, pc) = _opt_weights(w_pts, len(levels), len(pts)), _opt_weights(w_nys, len(levels), len(nys)), _opt_weights(w_nys_mirror, len(levels), len(nys))
    check(ctx.lib.icp_gpmm_face_nystrom_extend(ctx.h, len(pts), dptr(pts), pa, len(nys), dptr(nys), pb, pc, C.byref(fk), rank, dptr(V), dptr(w),
                                               dptr(basis), dptr(var)), ctx.h)
    return basis, var


def posterior_variability(model: Model, thetas, sum_normals=True, theta_ref=None):
    """icp_posterior_variability: dict(mean N x 3, cov N x 3 x 3, total_variance N, normal_variance N)."""
    th, s = model._theta(thetas)
    n = model.N
    mean, cov, tot, nrm = np.empty((n, 3)), np.empty((n, 3, 3)), np.empty(n), np.empty(n)
    ref = None
    if theta_ref is not None:
        ref, one = model._theta(theta_ref)
        if one != 1:
            raise ValueError("theta_ref must be a single parameter vector")
    check(model.lib.icp_posterior_variability(model.h, s, dptr(th), 1 if sum_normals else 0, dptr(ref) if ref is not None else None,
                                              dptr(mean), dptr(cov), dptr(tot), dptr(nrm)), model.ctx.h)
    return dict(mean=mean, cov=cov, total_variance=tot, normal_variance=nrm)


class JsonLog:
    """Streaming writer of the reference's chain-log file (icp_jsonlog_*; JSONAcceptRejectLogger.scala:93-122)."""

    def __init__(self, path, K, component_names, value_keys=("product", "prior", "distance")):
        self.lib = _lib.load()
        names = (C.c_char_p * len(component_names))(*[str(n).encode() for n in component_names])
        keys = (C.c_char_p * 3)(*[str(k).encode() for k in value_keys])
        self.h = C.c_void_p()
        check(self.lib.icp_jsonlog_open(str(path).encode(), int(K), names, len(component_names), keys, C.byref(self.h)))

    def append(self, run, chain=0):
        """run: the dict Chain.run returned (log arrays [n_steps][C])."""
        comp = i32(run["component"]); acc = np.ascontiguousarray(run["accepted"], dtype=np.uint8)
        vals, th = f64(run["values"]), f64(run["theta"])
        n, c = comp.shape
        check(self.lib.icp_jsonlog_append(self.h, n, c, int(chain), iptr(comp), acc.ctypes.data_as(_lib._bp), dptr(vals), dptr(th)))

    def close(self):
        if self.h:
            self.lib.icp_jsonlog_close(self.h)
            self.h = None


def jsonlog_load(path, K):
    """icp_jsonlog_load -> dict(index, status, values [n, 3], value_keys, theta [n, K + 10] (NaN rows for rejected records), names)."""
    lib = _lib.load()
    n = C.c_int64(0)
    check(lib.icp_jsonlog_load(str(path).encode(), int(K), 0, C.byref(n), None, None, None, None, None, None))
    cnt = n.value
    index = np.zeros(cnt, np.int64); status = np.zeros(cnt, np.uint8); values = np.zeros((cnt, 3)); theta = np.zeros((cnt, K + THETA0))
    names = C.create_string_buffer(64 * max(cnt, 1)); keys = C.create_string_buffer(64 * 3)
    check(lib.icp_jsonlog_load(str(path).encode(), int(K), cnt, C.byref(n), index.ctypes.data_as(_lib._lp), status.ctypes.data_as(_lib._bp),
                               dptr(values), dptr(theta), names, keys))
    nm = [names.raw[64 * i: 64 * i + 64].split(b"\0")[0].decode() for i in range(cnt)]
    ks = [keys.raw[64 * i: 64 * i + 64].split(b"\0")[0].decode() for i in range(3)]
    return dict(index=index, status=status.astype(bool), values=values, value_keys=ks, theta=theta, names=nm)


def chainlog_sample_indices(status, take_every_n=50, total=100, burn_in=0):
    """icp_chainlog_sample_indices: LogHelper.samplesFromLog's indices (closest accepted record at or before each pick)."""
    lib = _lib.load()
    st = np.ascontiguousarray(status, dtype=np.uint8)
    n = C.c_int64(0)
    check(lib.icp_chainlog_sample_indices(len(st), st.ctypes.data_as(_lib._bp), int(take_every_n), int(total), int(burn_in), 0, C.byref(n), None))
    out = np.zeros(n.value, np.int64)
    check(lib.icp_chainlog_sample_indices(len(st), st.ctypes.data_as(_lib._bp), int(take_every_n), int(total), int(burn_in), len(out),
                                          C.byref(n), out.ctypes.data_as(_lib._lp)))
    return out


class Comm:
    """NCCL communicator of the library (icp_comm_*): end-of-run gather of chain logs and reduction of posterior statistics.
    Rank 0 calls Comm.unique_id(ctx) and ships the 128 bytes to the other ranks through any channel it likes."""

    def __init__(self, ctx: Context, rank, world, unique_id):
        self.ctx, self.lib = ctx, ctx.lib
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        assert uid.size == 128
        self.h = C.c_void_p()
        check(self.lib.icp_comm_init(ctx.h, int(rank), int(world), uid.ctypes.data_as(_lib._bp), C.byref(self.h)), ctx.h)
        self.rank, self.world = int(rank), int(world)

    @staticmethod
    def unique_id(ctx: Context):
        uid = np.zeros(128, np.uint8)
        check(ctx.lib.icp_comm_unique_id(ctx.h, uid.ctypes.data_as(_lib._bp)), ctx.h)
        return uid

    def nccl_version(self):
        v = C.c_int32(0)
        check(self.lib.icp_comm_info(self.h, None, None, C.byref(v)))
        return v.value

    def chainlog_gather(self, n_steps, C_, K, local: "_lib.ChainIO", gathered: "_lib.ChainIO"):
        """local / gathered: ChainIO structures holding raw DEVICE addresses. Returns (device ms, bytes received)."""
        ms = C.c_double(0); nb = C.c_int64(0)
        check(self.lib.icp_chainlog_gather(self.h, int(n_steps), int(C_), int(K), C.byref(local), C.byref(gathered), C.byref(ms),
                                           C.byref(nb)), self.ctx.h)
        return ms.value, nb.value

    def variability_allreduce(self, model: Model, thetas, sum_normals=True, theta_ref=None):
        th = f64(thetas).reshape(-1, model.K + THETA0)
        s = len(th)
        n = model.N
        mean, cov, tot, nrm = np.empty((n, 3)), np.empty((n, 3, 3)), np.empty(n), np.empty(n)
        ref = None if theta_ref is None else f64(theta_ref).reshape(-1)
        total = C.c_int64(0)
        check(self.lib.icp_variability_allreduce(self.h, model.h, s, dptr(th) if s else None, 1 if sum_normals else 0,
                                                 dptr(ref) if ref is not None else None, dptr(mean), dptr(cov), dptr(tot), dptr(nrm),
                                                 C.byref(total)), self.ctx.h)
        return dict(n=total.value, mean=mean, cov=cov, total_variance=tot, normal_variance=nrm)

    def close(self):
        if self.h:
            self.lib.icp_comm_destroy(self.h)
            self.h = None


class Chain:
    """Fused Metropolis-Hastings runner (Scalismo MetropolisHastings + MixtureProposal on the device)."""

    def __init__(self, model: Model, target: Target = None, components=None, evaluator: Evaluator = None, max_chains=1,
                 targets=None):
        """components: list of dict(kind, weight, proposal=IcpProposal|None, sd=0, axis=0, name=...).
        targets: instead of (target, components, evaluator), a list of such triples, one per target of the handle
        (icp_chain_create_targets); run() then needs target_index."""
        self.lib, self.ctx, self.model = model.lib, model.ctx, model
        if targets is None:
            targets = [(target, components, evaluator)]
        elif target is not None or components is not None or evaluator is not None:
            raise ValueError("pass either target, components and evaluator or targets")
        self.targets = [(t, list(cs), e) for t, cs, e in targets]
        self.target, self.components, self.evaluator = self.targets[0]
        self.n_targets = len(self.targets)
        self._arrs = []
        for _, cs, _ in self.targets:
            arr = (_lib.Component * len(cs))()
            for i, c in enumerate(cs):
                arr[i].kind = int(c["kind"]); arr[i].axis = int(c.get("axis", 0)); arr[i].weight = float(c["weight"])
                arr[i].sd = float(c.get("sd", 0.0))
                arr[i].proposal = c["proposal"].h if c.get("proposal") is not None else None
            self._arrs.append(arr)
        self._arr = self._arrs[0]
        self.max_chains = int(max_chains)
        self.h = C.c_void_p()
        if len(self.targets) == 1:
            check(self.lib.icp_chain_create(model.h, self.target.h, self._arr, len(self.components), self.evaluator.h,
                                            self.max_chains, C.byref(self.h)), self.ctx.h)
        else:
            ents = (_lib.ChainTarget * len(self.targets))()
            for g, (t, cs, e) in enumerate(self.targets):
                ents[g].target, ents[g].components, ents[g].evaluator = t.h, self._arrs[g], e.h
            check(self.lib.icp_chain_create_targets(model.h, len(self.targets), ents, len(self.components), self.max_chains,
                                                    C.byref(self.h)), self.ctx.h)

    def set_target_index(self, target_index):
        """icp_chain_set_target_index: chain c of the next run from theta0 runs on targets[target_index[c]]."""
        ti = np.ascontiguousarray(target_index, dtype=np.int32).reshape(-1)
        check(self.lib.icp_chain_set_target_index(self.h, len(ti), ti.ctypes.data_as(_lib._ip)), self.ctx.h)

    def run(self, theta0, n_steps, seed=1024, chain_id_offset=0, u_comp=None, z=None, u_acc=None, log_theta=True,
            raise_on_status=True, metrics_interval=0, target_index=None):
        """raise_on_status=False: a per-chain status failure (empty set / not positive definite / NaN, the cases in which the
        reference throws) does not raise; the result carries `status` (per-chain words) and `status_code` (the return code).
        target_index: [C] target of every chain (set_target_index before the run)."""
        if target_index is not None:
            self.set_target_index(target_index)
        th, c = self.model._theta(theta0)
        K, L = self.model.K, self.model.K + THETA0
        io = _lib.ChainIO()
        io.seed, io.chain_id_offset = int(seed), int(chain_id_offset)
        keep = []
        if u_comp is not None:
            uc = f64(u_comp).reshape(n_steps, c); zz = f64(z).reshape(n_steps, c, K); ua = f64(u_acc).reshape(n_steps, c)
            keep += [uc, zz, ua]
            io.u_comp, io.z, io.u_acc = uc.ctypes.data, zz.ctypes.data, ua.ctypes.data
        comp = np.empty((n_steps, c), np.int32); acc = np.empty((n_steps, c), np.uint8)
        vals = np.empty((n_steps, c, 3)); final = np.empty((c, L)); nacc = np.zeros(c, np.int64)
        io.log_component, io.log_accepted, io.log_values = comp.ctypes.data, acc.ctypes.data, vals.ctypes.data
        thl = None
        if log_theta:
            thl = np.empty((n_steps, c, L))
            io.log_theta = thl.ctypes.data
        io.theta_final, io.n_accepted = final.ctypes.data, nacc.ctypes.data
        status = np.zeros(c, np.int32)
        io.status = status.ctypes.data
        best, vbest = np.empty((c, L)), np.empty(c)
        io.theta_best, io.value_best = best.ctypes.data, vbest.ctypes.data
        metrics = None
        if metrics_interval > 0:
            metrics = np.empty((n_steps // metrics_interval, c, 4))
            io.metrics_interval, io.log_metrics = int(metrics_interval), metrics.ctypes.data
        rc = self.lib.icp_chain_run(self.h, c, int(n_steps), dptr(th), C.byref(io))
        if rc != _lib.OK and (raise_on_status or rc not in (_lib.ERR_EMPTY_SET, _lib.ERR_NOT_POSITIVE_DEFINITE, _lib.ERR_NAN)):
            check(rc, self.ctx.h)
        return dict(component=comp, accepted=acc.astype(bool), values=vals, theta=thl, theta_final=final, n_accepted=nacc,
                    status=status, status_code=rc, theta_best=best, value_best=vbest, metrics=metrics)

    def run_device(self, C_, n_steps, theta0_ptr, seed=1024, chain_id_offset=0, log_component=0, log_accepted=0,
                   log_values=0, log_theta=0, theta_final=0, n_accepted=0, async_=False, target_index=None):
        """All pointers are raw device addresses (e.g. torch.Tensor.data_ptr()); target_index is a host array as for run()."""
        if target_index is not None:
            self.set_target_index(target_index)
        io = _lib.ChainIO()
        io.seed, io.chain_id_offset = int(seed), int(chain_id_offset)
        io.log_component, io.log_accepted, io.log_values = log_component or None, log_accepted or None, log_values or None
        io.log_theta, io.theta_final, io.n_accepted = log_theta or None, theta_final or None, n_accepted or None
        check(self.lib.icp_chain_run_device(self.h, int(C_), int(n_steps), theta0_ptr, C.byref(io), int(async_)), self.ctx.h)

    def last_run_stats(self):
        ms = C.c_double(0); n = C.c_int64(0)
        check(self.lib.icp_chain_last_run_stats(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def set_lookahead(self, width):
        """icp_chain_set_lookahead: -1 automatic, 0 off, 2..32 lanes per chain."""
        check(self.lib.icp_chain_set_lookahead(self.h, int(width)), self.ctx.h)

    def last_run_rounds(self):
        n = C.c_int64(0)
        check(self.lib.icp_chain_last_run_rounds(self.h, C.byref(n)))
        return n.value

    def set_statistics(self, burn_in, take_every_n=1, end=0, normals=True):
        """icp_chain_set_statistics: accumulate the posterior variability maps of the records burn_in, burn_in + take_every_n, ...
        below `end` (<= 0: no limit) inside the run, from the next run from theta0 on. burn_in=None switches them off."""
        if burn_in is None:
            check(self.lib.icp_chain_set_statistics(self.h, None), self.ctx.h)
            return
        p = _lib.ChainStatsParams(int(burn_in), int(take_every_n), int(end), 1 if normals else 0, 0)
        check(self.lib.icp_chain_set_statistics(self.h, C.byref(p)), self.ctx.h)

    def statistics(self, chain=-1, sum_normals=True, theta_ref=None):
        """icp_chain_statistics: the maps of chain `chain` of the resident run, or pooled over its chains (-1): the dict of
        posterior_variability plus n, the number of samples."""
        n = self.model.N
        mean, cov, tot, nrm = np.empty((n, 3)), np.empty((n, 3, 3)), np.empty(n), np.empty(n)
        ref = None
        if theta_ref is not None:
            ref, one = self.model._theta(theta_ref)
            if one != 1:
                raise ValueError("theta_ref must be a single parameter vector")
        s = C.c_int64(0)
        check(self.lib.icp_chain_statistics(self.h, int(chain), 1 if sum_normals else 0, dptr(ref) if ref is not None else None,
                                            C.byref(s), dptr(mean), dptr(cov), dptr(tot), dptr(nrm)), self.ctx.h)
        return dict(mean=mean, cov=cov, total_variance=tot, normal_variance=nrm, n=int(s.value))

    def profile(self, theta0, n_steps, seed=1024):
        th, c = self.model._theta(theta0)
        ms = np.zeros(_lib.N_STAGES); n = np.zeros(_lib.N_STAGES, np.int64)
        check(self.lib.icp_chain_profile(self.h, c, int(n_steps), dptr(th), int(seed), dptr(ms), n.ctypes.data_as(_lib._lp)),
              self.ctx.h)
        names = [self.lib.icp_stage_name(i).decode() for i in range(_lib.N_STAGES)]
        return {nm: {"ms": float(a), "launches": int(b)} for nm, a, b in zip(names, ms, n)}

    def close(self):
        if self.h:
            self.lib.icp_chain_destroy(self.h)
            self.h = None
