// metrics.cu - registration quality measures between transformedMesh(theta) and the target, batched over chains.
//
// Replaces (paths relative to src/main/scala of the reference):
//   api/other/RegistrationComparison.scala:24-49   MeshMetrics.avgDistance / hausdorffDistance and the boundary-aware
//                                                   average + maximum, printed every acceptInfoPrintInterval steps for the
//                                                   best sample so far (api/sampling/SamplingRegistration.scala:75-82)
//   apps/femur/StdIcpVsChainICPrandomInitComparisonAll.scala:43-47   MeshMetrics.diceCoefficient(best, target)
// All of them are the closest-point / nearest-vertex queries of the hot path over every vertex (or over sample points).
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "icp_device.cuh"
#include "icp_internal.h"

using namespace icp;

namespace icp {

// per chain: {avg, hausdorff, avg_boundary_aware, max_boundary_aware}
__global__ void __launch_bounds__(128) k_metrics(int N, int Nt, const double *__restrict__ d2_m2t,
                                                 const uint8_t *__restrict__ skip, const double *__restrict__ d2_t2m,
                                                 double *__restrict__ out) {
    __shared__ double red[4][128];
    int c = blockIdx.x;
    double s = 0, mx = 0, sb = 0, cb = 0, mb = -INFINITY, mt = 0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        double d = sqrt(d2_m2t[(size_t)c * N + i]);
        s += d; mx = fmax(mx, d);
        if (!(skip && skip[(size_t)c * N + i])) { sb += d; cb += 1; mb = fmax(mb, d); }
    }
    for (int i = threadIdx.x; i < Nt; i += blockDim.x) mt = fmax(mt, sqrt(d2_t2m[(size_t)c * Nt + i]));
    red[0][threadIdx.x] = s; red[1][threadIdx.x] = fmax(mx, mt); red[2][threadIdx.x] = sb; red[3][threadIdx.x] = cb;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            red[0][threadIdx.x] += red[0][threadIdx.x + o];
            red[1][threadIdx.x] = fmax(red[1][threadIdx.x], red[1][threadIdx.x + o]);
            red[2][threadIdx.x] += red[2][threadIdx.x + o];
            red[3][threadIdx.x] += red[3][threadIdx.x + o];
        }
        __syncthreads();
    }
    // an empty filtered list: the reference's `filteredDists.sum / size` is NaN and `.max` throws (:42); both NaN here
    double avg = red[0][0] / N, hd = red[1][0], avgb = red[2][0] / red[3][0];
    const bool empty = red[3][0] == 0.0;
    __syncthreads();
    red[0][threadIdx.x] = mb;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[0][threadIdx.x] = fmax(red[0][threadIdx.x], red[0][threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[4 * c] = avg; out[4 * c + 1] = hd; out[4 * c + 2] = avgb; out[4 * c + 3] = empty ? NAN : red[0][0]; }
}

// row c of dst [C][nt][3]: the vertices of target tidx[c], its last vertex repeated up to nt entries. Only the maximum of the
// target -> model distances is read (k_metrics), and a repeat does not change it.
__global__ void k_gather_target_verts(long long total, int nt, const TargetGeom *__restrict__ geom, const int *__restrict__ tidx,
                                      double *__restrict__ dst) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const TargetGeom &g = geom[tidx[i / nt]];
    const int v = min((int)(i % nt), g.Nt - 1);
#pragma unroll
    for (int d = 0; d < 3; d++) dst[3 * i + d] = g.verts[3 * v + d];
}

void registration_metrics_device(icp_model m, icp_target t, int C, const double *d_theta, double *d_out, MetricsWork &w,
                                 cudaStream_t s, const MetricsTargets *ts) {
    if (C <= 0) return;
    const int N = m->N, Nt = ts ? ts->max_nt : t->Nt;
    const bool has_boundary = ts ? ts->has_boundary : t->has_boundary;
    // a target set writes closest points only for the boundary filter
    const bool want_cp = !ts || has_boundary;
    w.X.ensure((size_t)C * N * 3); w.d2a.ensure((size_t)C * N); w.d2b.ensure((size_t)C * Nt);
    if (want_cp) w.cpa.ensure((size_t)C * N * 3);
    launch_reconstruct(m->dev(), C, d_theta, w.X.p, s);
    // every model vertex against the target surface
    NearestArgs a;
    a.bvh = &t->tri_bvh; a.prim_data = t->tri_data.p; a.wide = t->wide(); a.sm_count = t->ctx->sm_count; a.C = C; a.nq = N; a.q = w.X.p; a.q_per_chain = 1;
    a.out_d2 = w.d2a.p; a.out_cp = want_cp ? w.cpa.p : nullptr;
    if (ts) { a.mt_rec = ts->rec; a.mt_idx = ts->tidx; }   // row c walks the BVH of its own target
    launch_nearest(a, s);
    const uint8_t *skip_p = nullptr;
    if (has_boundary) {
        // :35-37 nearest target vertex of the closest point, dropped when it lies on the target's boundary
        w.prim.ensure((size_t)C * N); w.skip.ensure((size_t)C * N);
        NearestArgs v;
        v.bvh = &t->vert_bvh; v.prim_data = t->vert_data.p; v.C = C; v.nq = N; v.q = w.cpa.p; v.q_per_chain = 1; v.out_prim = w.prim.p;
        if (ts) { v.mt_rec = ts->rec; v.mt_idx = ts->tidx; }
        launch_nearest(v, s);
        // a closed target of a set has an all-zero table: its rows sum as with no filter, in the same order
        if (ts) launch_lookup_flags((int64_t)C * N, w.prim.p, t->boundary.p, Nt, w.skip.p, s, ts->rec, ts->tidx, N);
        else launch_lookup_flags((int64_t)C * N, w.prim.p, t->boundary.p, Nt, w.skip.p, s);
        skip_p = w.skip.p;
    }
    // every target vertex against the model surfaces (second half of hausdorffDistance)
    const double *tq = t->verts.p;
    if (ts) {
        w.tq.ensure((size_t)C * Nt * 3);
        const long long total = (long long)C * Nt;
        k_gather_target_verts<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(total, Nt, ts->geom, ts->tidx, w.tq.p);
        ICP_CUDA(cudaGetLastError());
        tq = w.tq.p;
    }
    bvh_refit(m->tri_bvh, C, w.X.p, N, m->tris.p, s);
    NearestArgs b;
    b.bvh = &m->tri_bvh; b.X = w.X.p; b.tris = m->tris.p; b.N = N; b.C = C; b.nq = Nt; b.q = tq; b.q_per_chain = ts ? 1 : 0;
    b.out_d2 = w.d2b.p;
    launch_nearest(b, s);
    k_metrics<<<C, 128, 0, s>>>(N, Nt, w.d2a.p, skip_p, w.d2b.p, d_out);
    ICP_CUDA(cudaGetLastError());
}

// ---- Dice coefficient ------------------------------------------------------------------------------------------------
// Scalismo MeshMetrics.diceCoefficient [S-recall]: n uniform samples in the union of the two bounding boxes; a sample is
// inside a mesh when  vertexNormal(v) . (v - p) > 0  for the mesh vertex v nearest to p (toBinaryImage);
// dice = 2 |A and B| / (|A| + |B|). The reference draws the samples from an unseeded global RNG (10 000 of them), so the
// caller supplies unit-cube samples (or a Philox seed) and they are scaled into each chain's evaluation region here.
// MT: row c's target box is geom[tidx[c]]'s instead of (tlx .. thz).
template <bool MT>
__global__ void __launch_bounds__(256) k_dice_points(int N, const double *__restrict__ X, double tlx, double tly, double tlz,
                                                     double thx, double thy, double thz, int n,
                                                     const double *__restrict__ unit, unsigned long long seed,
                                                     double *__restrict__ pts, const TargetGeom *__restrict__ geom,
                                                     const int *__restrict__ tidx) {
    __shared__ double red[6][256];
    const int c = blockIdx.x, tid = threadIdx.x;
    if (MT) {
        const TargetGeom &g = geom[tidx[c]];
        tlx = g.lo[0]; tly = g.lo[1]; tlz = g.lo[2]; thx = g.hi[0]; thy = g.hi[1]; thz = g.hi[2];
    }
    const double *Xc = X + (size_t)c * N * 3;
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int v = tid; v < N; v += blockDim.x)
#pragma unroll
        for (int d = 0; d < 3; d++) { const double x = Xc[3 * v + d]; lo[d] = fmin(lo[d], x); hi[d] = fmax(hi[d], x); }
#pragma unroll
    for (int d = 0; d < 3; d++) { red[d][tid] = lo[d]; red[3 + d][tid] = hi[d]; }
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o)
#pragma unroll
            for (int d = 0; d < 3; d++) {
                red[d][tid] = fmin(red[d][tid], red[d][tid + o]);
                red[3 + d][tid] = fmax(red[3 + d][tid], red[3 + d][tid + o]);
            }
        __syncthreads();
    }
    const double l0 = fmin(red[0][0], tlx), l1 = fmin(red[1][0], tly), l2 = fmin(red[2][0], tlz);
    const double e0 = fmax(red[3][0], thx) - l0, e1 = fmax(red[4][0], thy) - l1, e2 = fmax(red[5][0], thz) - l2;
    for (int i = tid; i < n; i += blockDim.x) {
        double u0, u1, u2;
        if (unit) { u0 = unit[3 * i]; u1 = unit[3 * i + 1]; u2 = unit[3 * i + 2]; }
        else {
            // the same sample set for every chain (keyed by the sample index only): chains are compared on equal terms
            const uint4 r0 = chain_philox(seed, (unsigned long long)i, 0u, 0u), r1 = chain_philox(seed, (unsigned long long)i, 0u, 1u);
            u0 = u53(r0.x, r0.y); u1 = u53(r0.z, r0.w); u2 = u53(r1.x, r1.y);
        }
        double *p = pts + ((size_t)c * n + i) * 3;
        p[0] = l0 + u0 * e0; p[1] = l1 + u1 * e1; p[2] = l2 + u2 * e2;
    }
}

// MT: row c reads the vertices and vertex normals of target geom[tidx[c]] instead of (tverts, tnormals)
template <bool MT>
__global__ void __launch_bounds__(128) k_dice_count(ModelDev m, const double *__restrict__ X, int n,
                                                    const double *__restrict__ pts, const int *__restrict__ vid_model,
                                                    const int *__restrict__ vid_target, const double *__restrict__ tverts,
                                                    const double *__restrict__ tnormals, double *__restrict__ out,
                                                    const TargetGeom *__restrict__ geom, const int *__restrict__ tidx) {
    __shared__ double red[40];
    const int c = blockIdx.x;
    if (MT) {
        const TargetGeom &g = geom[tidx[c]];
        tverts = g.verts; tnormals = g.vnormals;
    }
    const double *Xc = X + (size_t)c * m.N * 3;
    double na = 0.0, nb = 0.0, nab = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double *p = pts + ((size_t)c * n + i) * 3;
        const int va = vid_model[(size_t)c * n + i], vb = vid_target[(size_t)c * n + i];
        double nx, ny, nz;
        vertex_normal_dev(m, Xc, va, nx, ny, nz);
        const bool ina = nx * (Xc[3 * va] - p[0]) + ny * (Xc[3 * va + 1] - p[1]) + nz * (Xc[3 * va + 2] - p[2]) > 0.0;
        const bool inb = tnormals[3 * vb] * (tverts[3 * vb] - p[0]) + tnormals[3 * vb + 1] * (tverts[3 * vb + 1] - p[1]) +
                         tnormals[3 * vb + 2] * (tverts[3 * vb + 2] - p[2]) > 0.0;
        na += ina ? 1.0 : 0.0; nb += inb ? 1.0 : 0.0; nab += (ina && inb) ? 1.0 : 0.0;
    }
    na = block_sum(na, red);
    __syncthreads();
    nb = block_sum(nb, red);
    __syncthreads();
    nab = block_sum(nab, red);
    if (threadIdx.x == 0) out[c] = 2.0 * nab / (na + nb);
}

void dice_device(icp_model m, icp_target t, int C, const double *d_theta, int n, const double *d_unit, uint64_t seed,
                 double *d_out, DiceWork &w, cudaStream_t s, const MetricsTargets *ts) {
    if (C <= 0) return;
    const int N = m->N;
    w.X.ensure((size_t)C * N * 3); w.pts.ensure((size_t)C * n * 3);
    w.va.ensure((size_t)C * n); w.vb.ensure((size_t)C * n);
    launch_reconstruct(m->dev(), C, d_theta, w.X.p, s);
    const TargetGeom *geom = ts ? ts->geom : nullptr;
    const int *tidx = ts ? ts->tidx : nullptr;
    if (ts) k_dice_points<true><<<C, 256, 0, s>>>(N, w.X.p, 0, 0, 0, 0, 0, 0, n, d_unit, seed, w.pts.p, geom, tidx);
    else k_dice_points<false><<<C, 256, 0, s>>>(N, w.X.p, t->lo[0], t->lo[1], t->lo[2], t->hi[0], t->hi[1], t->hi[2], n, d_unit, seed,
                                                w.pts.p, nullptr, nullptr);
    ICP_CUDA(cudaGetLastError());
    nearest_model_vertex(m, C, w.X.p, n, w.pts.p, 1, nullptr, w.va.p, s);
    NearestArgs v;
    v.bvh = &t->vert_bvh; v.prim_data = t->vert_data.p; v.C = C; v.nq = n; v.q = w.pts.p; v.q_per_chain = 1; v.out_prim = w.vb.p;
    if (ts) { v.mt_rec = ts->rec; v.mt_idx = ts->tidx; }
    launch_nearest(v, s);
    if (ts) k_dice_count<true><<<C, 128, 0, s>>>(m->dev(), w.X.p, n, w.pts.p, w.va.p, w.vb.p, nullptr, nullptr, d_out, geom, tidx);
    else k_dice_count<false><<<C, 128, 0, s>>>(m->dev(), w.X.p, n, w.pts.p, w.va.p, w.vb.p, t->verts.p, t->vnormals.p, d_out,
                                                nullptr, nullptr);
    ICP_CUDA(cudaGetLastError());
}

// ---- target sets -----------------------------------------------------------------------------------------------------
// The target-set calls process their rows in chunks, so that their scratch stays within a fixed budget whatever C is. Every
// row depends on its own data only, so the results do not depend on the chunking. Metrics: model vertices + padded target
// vertices of a row (each model vertex also carries its share of the refitted model BVH, about 300 bytes in all);
// Dice: sample points of a row (32 bytes each).
constexpr int64_t kMetricsChunkPoints = int64_t(1) << 23;
constexpr int64_t kDiceChunkPoints = int64_t(1) << 25;

int chunk_rows(int64_t budget, int64_t points_per_row, int C) {
    return (int)std::max<int64_t>(1, std::min<int64_t>(C, budget / std::max<int64_t>(points_per_row, 1)));
}

void upload_unit_samples(const double *h, int n, DevBuf<double> &d, cudaStream_t s) {
    for (size_t i = 0; i < (size_t)3 * n; i++) ICP_REQUIRE(h[i] >= 0.0 && h[i] <= 1.0, "unit_samples must lie in [0, 1]");
    d.upload(h, (size_t)3 * n, s);
}

// every entry non-null and of the model's context
void check_target_list(icp_model m, int G, const icp_target *targets) {
    ICP_REQUIRE(G >= 1 && targets != nullptr, "n_targets must be >= 1 and targets non-null");
    for (int g = 0; g < G; g++) {
        ICP_REQUIRE(targets[g] != nullptr, "targets[" + std::to_string(g) + "] is null");
        ICP_REQUIRE(targets[g]->ctx == m->ctx, "targets[" + std::to_string(g) + "] belongs to another context than the model");
    }
}

// A target set of one call on the device (nothing outlives the call)
struct TargetSetUpload {
    DevBuf<TargetRec> rec;
    DevBuf<TargetGeom> geom;
    DevBuf<int> tidx;
    MetricsTargets ts{};
};

void upload_metrics_targets(int G, const icp_target *targets, int C, const int32_t *target_index, TargetSetUpload &u,
                            cudaStream_t s) {
    for (int c = 0; c < C; c++)
        ICP_REQUIRE(target_index[c] >= 0 && target_index[c] < G, "target_index[" + std::to_string(c) + "] = " +
                    std::to_string(target_index[c]) + " is outside [0, n_targets)");
    std::vector<icp_target> list(targets, targets + G);
    std::vector<TargetGeom> geom(G);
    bool has_boundary = false;
    int max_nt = 0;
    for (int g = 0; g < G; g++) {
        const icp_target t = targets[g];
        geom[g] = TargetGeom{t->verts.p, t->vnormals.p, t->Nt, {t->lo[0], t->lo[1], t->lo[2]}, {t->hi[0], t->hi[1], t->hi[2]}};
        has_boundary = has_boundary || t->has_boundary;
        max_nt = std::max(max_nt, t->Nt);
    }
    upload_target_table(list, u.rec, s);
    u.geom.upload(geom.data(), geom.size(), s);
    u.tidx.upload(target_index, C, s);
    u.ts = MetricsTargets{u.rec.p, u.geom.p, u.tidx.p, has_boundary, max_nt};
}

}  // namespace icp

extern "C" int32_t icp_registration_metrics(icp_model m, icp_target t, int32_t C, const double *theta, double *out) {
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        CtxLock lock(_ctx);
        ICP_REQUIRE(t && t->ctx == m->ctx, "bad target");
        if (C == 0) return ICP_OK;
        ICP_REQUIRE(C > 0 && theta != nullptr && out != nullptr, "bad arguments");
        cudaStream_t s = _ctx->stream;
        m->s_theta.upload(theta, (size_t)C * (m->K + kTheta0), s);
        MetricsWork w;
        DevBuf<double> dout;
        dout.alloc((size_t)4 * C);
        registration_metrics_device(m, t, C, m->s_theta.p, dout.p, w, s);
        ICP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * 4 * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_dice_coefficient(icp_model m, icp_target t, int32_t C, const double *theta, int32_t n_samples,
                                        const double *unit_samples, uint64_t seed, double *out) {
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        CtxLock lock(_ctx);
        ICP_REQUIRE(t && t->ctx == m->ctx, "bad target");
        if (C == 0) return ICP_OK;
        ICP_REQUIRE(C > 0 && theta != nullptr && out != nullptr && n_samples >= 1, "bad arguments");
        cudaStream_t s = _ctx->stream;
        m->s_theta.upload(theta, (size_t)C * (m->K + kTheta0), s);
        DevBuf<double> unit, dout;
        DiceWork w;
        dout.alloc(C);
        if (unit_samples) upload_unit_samples(unit_samples, n_samples, unit, s);
        dice_device(m, t, C, m->s_theta.p, n_samples, unit_samples ? unit.p : nullptr, seed, dout.p, w, s);
        ICP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_registration_metrics_targets(icp_model m, int32_t n_targets, const icp_target *targets, int32_t C,
                                                    const double *theta, const int32_t *target_index, double *out) {
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        check_target_list(m, n_targets, targets);
        if (n_targets == 1 && target_index == nullptr) return icp_registration_metrics(m, targets[0], C, theta, out);
        ICP_REQUIRE(target_index != nullptr || C == 0, "target_index is required when n_targets > 1");
        CtxLock lock(_ctx);
        if (C == 0) return ICP_OK;
        ICP_REQUIRE(C > 0 && theta != nullptr && out != nullptr, "bad arguments");
        cudaStream_t s = _ctx->stream;
        TargetSetUpload u;
        upload_metrics_targets(n_targets, targets, C, target_index, u, s);
        const size_t Lt = (size_t)m->K + kTheta0;
        DevBuf<double> dth, dout;
        dth.upload(theta, (size_t)C * Lt, s);
        dout.alloc((size_t)4 * C);
        MetricsWork w;
        const int rows = chunk_rows(kMetricsChunkPoints, (int64_t)m->N + u.ts.max_nt, C);
        for (int c0 = 0; c0 < C; c0 += rows) {
            MetricsTargets ts = u.ts;
            ts.tidx += c0;
            registration_metrics_device(m, targets[0], std::min(rows, C - c0), dth.p + c0 * Lt, dout.p + (size_t)4 * c0, w, s, &ts);
        }
        ICP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * 4 * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_dice_coefficient_targets(icp_model m, int32_t n_targets, const icp_target *targets, int32_t C,
                                                const double *theta, const int32_t *target_index, int32_t n_samples,
                                                const double *unit_samples, uint64_t seed, double *out) {
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        check_target_list(m, n_targets, targets);
        if (n_targets == 1 && target_index == nullptr)
            return icp_dice_coefficient(m, targets[0], C, theta, n_samples, unit_samples, seed, out);
        ICP_REQUIRE(target_index != nullptr || C == 0, "target_index is required when n_targets > 1");
        CtxLock lock(_ctx);
        if (C == 0) return ICP_OK;
        ICP_REQUIRE(C > 0 && theta != nullptr && out != nullptr && n_samples >= 1, "bad arguments");
        cudaStream_t s = _ctx->stream;
        TargetSetUpload u;
        upload_metrics_targets(n_targets, targets, C, target_index, u, s);
        const size_t Lt = (size_t)m->K + kTheta0;
        DevBuf<double> dth, unit, dout;
        if (unit_samples) upload_unit_samples(unit_samples, n_samples, unit, s);
        dth.upload(theta, (size_t)C * Lt, s);
        dout.alloc(C);
        DiceWork w;
        const int rows = chunk_rows(kDiceChunkPoints, n_samples, C);
        for (int c0 = 0; c0 < C; c0 += rows) {
            MetricsTargets ts = u.ts;
            ts.tidx += c0;
            dice_device(m, targets[0], std::min(rows, C - c0), dth.p + c0 * Lt, n_samples, unit_samples ? unit.p : nullptr, seed,
                        dout.p + c0, w, s, &ts);
        }
        ICP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}
