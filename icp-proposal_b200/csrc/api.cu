// api.cu - C ABI entry points of libicpcuda.so (include/icpcuda.h): contexts, handles, primitives,
// the batched proposal / evaluator calls and the pipelines they share with the chain runner.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "icp_internal.h"

using namespace icp;

// ---------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_thread_err;

namespace icp {

uint64_t next_alloc_id() {
    static std::atomic<uint64_t> counter{0};
    return ++counter;
}

void set_error(icp_ctx ctx, const std::string &msg) {
    g_thread_err = msg;
    if (ctx) {
        std::lock_guard<std::mutex> g(ctx->err_mu);
        ctx->err = msg;
    }
}

CtxLock::CtxLock(icp_ctx c) : lk(c->mu) {
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) throw CudaError{e, __FILE__, __LINE__};
}

int32_t translate_exception(icp_ctx ctx) {
    try {
        throw;
    } catch (const ArgError &e) {
        set_error(ctx, "invalid argument: " + e.msg);
        return ICP_ERR_INVALID_ARGUMENT;
    } catch (const StatusError &e) {
        set_error(ctx, e.msg);
        return e.code;
    } catch (const CudaError &e) {
        set_error(ctx, std::string("CUDA error: ") + cudaGetErrorString(e.e) + " at " + e.file + ":" + std::to_string(e.line));
        cudaGetLastError();
        return e.e == cudaErrorMemoryAllocation ? ICP_ERR_OUT_OF_MEMORY : ICP_ERR_CUDA;
    } catch (const std::bad_alloc &) {
        set_error(ctx, "host allocation failed");
        return ICP_ERR_OUT_OF_MEMORY;
    } catch (const std::exception &e) {
        set_error(ctx, std::string("internal error: ") + e.what());
        return ICP_ERR_INVALID_ARGUMENT;
    } catch (...) {
        set_error(ctx, "unknown internal error");
        return ICP_ERR_INVALID_ARGUMENT;
    }
}

}  // namespace icp

#define ICP_API_BEGIN(ctxexpr)      \
    icp_ctx _ctx = (ctxexpr);       \
    try {                           \
        ICP_REQUIRE(_ctx != nullptr, "null handle"); \
        CtxLock _lock(_ctx);
// per-call entry point on a proposal / evaluator: `cs` is the leased call slot (scratch), `s` the stream the call runs on
// and synchronises
#define ICP_API_BEGIN_HANDLE(HandleT, h, self_contained)                   \
    icp_ctx _ctx = (h) ? (h)->model->ctx : nullptr;                        \
    try {                                                                  \
        ICP_REQUIRE(_ctx != nullptr, "null handle");                       \
        CallLease<HandleT> _lease(_ctx, (h), (self_contained));            \
        HandleT::Call &cs = *_lease.call;                                  \
        cudaStream_t s = _lease.stream;
#define ICP_API_END                         \
        return ICP_OK;                      \
    } catch (...) {                         \
        return translate_exception(_ctx);   \
    }

static void sync_stream(icp_ctx ctx) { ICP_CUDA(cudaStreamSynchronize(ctx->stream)); }

template <class T>
static void download(T *h, const T *d, size_t n, cudaStream_t s) {
    if (n && h) ICP_CUDA(cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, s));
}

// ---------------------------------------------------------------------------------------------------
// (1) context
// ---------------------------------------------------------------------------------------------------
extern "C" int32_t icp_ctx_create(int32_t device, icp_ctx *out) {
    icp_ctx ctx = nullptr;
    try {
        ICP_REQUIRE(out != nullptr, "out is null");
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess) throw CudaError{e, __FILE__, __LINE__};
        ICP_REQUIRE(device >= 0 && device < count, "no such CUDA device (libicpcuda has no CPU fallback)");
        ICP_CUDA(cudaSetDevice(device));
        ctx = new icp_ctx_s();
        ctx->device = device;
        cudaDeviceProp prop;
        ICP_CUDA(cudaGetDeviceProperties(&prop, device));
        ctx->sm_count = prop.multiProcessorCount;
        ctx->device_name = prop.name;
        ICP_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        for (int i = 0; i < icp_ctx_s::kAux; i++) {
            ICP_CUDA(cudaStreamCreateWithFlags(&ctx->aux[i], cudaStreamNonBlocking));
            ICP_CUDA(cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming));
        }
        ICP_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        *out = ctx;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(nullptr);
        delete ctx;
        return rc;
    }
}

extern "C" int32_t icp_ctx_destroy(icp_ctx ctx) {
    if (!ctx) return ICP_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
        for (int i = 0; i < icp_ctx_s::kAux; i++) {
            if (ctx->aux[i]) { cudaStreamSynchronize(ctx->aux[i]); cudaStreamDestroy(ctx->aux[i]); }
            if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
        }
        if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    }
    delete ctx;
    return ICP_OK;
}

extern "C" int32_t icp_last_error(icp_ctx ctx, char *buf, size_t n) {
    if (!buf || n == 0) return ICP_ERR_INVALID_ARGUMENT;
    std::string s = g_thread_err;
    if (ctx) {
        std::lock_guard<std::mutex> g(ctx->err_mu);
        s = ctx->err;
    }
    size_t k = std::min(n - 1, s.size());
    memcpy(buf, s.data(), k);
    buf[k] = 0;
    return ICP_OK;
}

extern "C" int32_t icp_version(icp_ctx ctx, char *buf, size_t n) {
    if (!buf || n == 0) return ICP_ERR_INVALID_ARGUMENT;
    std::string s = "icpcuda 0.1 sm_100a";
    if (ctx) s += " " + ctx->device_name + " (" + std::to_string(ctx->sm_count) + " SMs)";
    size_t k = std::min(n - 1, s.size());
    memcpy(buf, s.data(), k);
    buf[k] = 0;
    return ICP_OK;
}

extern "C" int32_t icp_ctx_synchronize(icp_ctx ctx) {
    ICP_API_BEGIN(ctx)
    sync_stream(ctx);
    ICP_API_END
}

// ---------------------------------------------------------------------------------------------------
// host-side mesh tables (construction time only)
// ---------------------------------------------------------------------------------------------------
// Scalismo pointIsOnBoundary (SURVEY Appendix A12): vertex on an edge with exactly one incident triangle
static std::vector<uint8_t> boundary_table(int nv, int nt, const int32_t *tris) {
    std::vector<uint64_t> ek((size_t)3 * nt);
    for (int t = 0; t < nt; t++)
        for (int k = 0; k < 3; k++) {
            uint64_t a = (uint64_t)tris[3 * t + k], b = (uint64_t)tris[3 * t + (k + 1) % 3];
            ek[(size_t)3 * t + k] = a < b ? (a << 32) | b : (b << 32) | a;
        }
    std::sort(ek.begin(), ek.end());
    std::vector<uint8_t> f((size_t)std::max(nv, 1), 0);
    for (size_t i = 0; i < ek.size();) {
        size_t j = i;
        while (j < ek.size() && ek[j] == ek[i]) j++;
        if (j - i == 1) {
            f[ek[i] >> 32] = 1;
            f[ek[i] & 0xffffffffu] = 1;
        }
        i = j;
    }
    return f;
}

static void check_mesh(int nv, int nt, const double *xyz, const int32_t *tris) {
    ICP_REQUIRE(nv >= 1 && nt >= 1, "mesh needs at least one vertex and one triangle");
    ICP_REQUIRE(xyz != nullptr && tris != nullptr, "mesh arrays are null");
    for (size_t i = 0; i < (size_t)3 * nt; i++) ICP_REQUIRE(tris[i] >= 0 && tris[i] < nv, "triangle index out of range");
    for (size_t i = 0; i < (size_t)3 * nv; i++) ICP_REQUIRE(std::isfinite(xyz[i]), "non-finite vertex coordinate");
}

static double max_abs(const double *x, size_t n) {
    double m = 0;
    for (size_t i = 0; i < n; i++) m = std::max(m, std::fabs(x[i]));
    return m;
}

// ---------------------------------------------------------------------------------------------------
// (2) model
// ---------------------------------------------------------------------------------------------------
extern "C" int32_t icp_model_create(icp_ctx ctx, int32_t N, int32_t T, int32_t K, const double *ref_xyz,
                                    const double *mean_def, const double *basis, const double *variance,
                                    const int32_t *tris, icp_model *out) {
    icp_model m = nullptr;
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx != nullptr && out != nullptr, "null handle");
        CtxLock lock(ctx);
        ICP_REQUIRE(K >= 1 && K <= 224, "rank K must be in [1, 224]");
        ICP_REQUIRE(basis != nullptr && variance != nullptr, "basis / variance are null");
        check_mesh(N, T, ref_xyz, tris);
        for (int j = 0; j < K; j++) ICP_REQUIRE(variance[j] >= 0 && std::isfinite(variance[j]), "variance must be finite and >= 0");
        cudaStream_t s = ctx->stream;
        m = new icp_model_s();
        m->ctx = ctx; m->N = N; m->T = T; m->K = K; m->Kp = pad8(K);
        const int Kp = m->Kp;
        size_t n3 = (size_t)3 * N;
        m->ref.upload(ref_xyz, n3, s);
        m->h_ref.assign(ref_xyz, ref_xyz + n3);
        std::vector<double> mean(n3, 0.0);
        if (mean_def) std::copy(mean_def, mean_def + n3, mean.begin());
        m->mean.upload(mean.data(), n3, s);
        m->tris.upload(tris, (size_t)3 * T, s);
        // adjacency (ascending triangle id per vertex) and boundary table
        std::vector<int> off(N + 1, 0), adj((size_t)3 * T), fill(N, 0);
        for (size_t i = 0; i < (size_t)3 * T; i++) off[tris[i] + 1]++;
        for (int v = 0; v < N; v++) off[v + 1] += off[v];
        for (int t = 0; t < T; t++)
            for (int k = 0; k < 3; k++) { int v = tris[3 * t + k]; adj[off[v] + fill[v]++] = t; }
        m->adj_off.upload(off.data(), off.size(), s);
        m->adj.upload(adj.data(), adj.size(), s);
        m->h_boundary = boundary_table(N, T, tris);
        m->has_boundary = std::any_of(m->h_boundary.begin(), m->h_boundary.end(), [](uint8_t b) { return b != 0; });
        m->boundary.upload(m->h_boundary.data(), m->h_boundary.size(), s);
        // scaled basis
        DevBuf<double> dU, dvar;
        dU.upload(basis, n3 * K, s);
        dvar.upload(variance, K, s);
        m->h_var.assign(variance, variance + K);
        m->h_col_norm.assign(m->Kp, 0.0);
        for (int v = 0; v < N; v++)
            for (int j = 0; j < K; j++) {
                double s2 = 0.0;
                for (int e = 0; e < 3; e++) { const double u = basis[((size_t)3 * v + e) * K + j]; s2 += u * u; }
                m->h_col_norm[j] = std::max(m->h_col_norm[j], std::sqrt(s2 * variance[j]));
            }
        {
            std::vector<double> sv(Kp, 1.0);
            for (int j = 0; j < K; j++) sv[j] = std::sqrt(variance[j]);
            m->sqrt_var.upload(sv.data(), sv.size(), s);
            sync_stream(ctx);
        }
        m->Q.alloc(n3 * Kp);
        m->QT.alloc(n3 * Kp);
        launch_scale_basis((int)n3, K, Kp, dU.p, dvar.p, m->Q.p, m->QT.p, s);
        m->col_norm.upload(m->h_col_norm.data(), m->h_col_norm.size(), s);
        m->Qhat.alloc(n3 * Kp);
        launch_unit_basis((int)n3, Kp, m->Q.p, m->col_norm.p, m->Qhat.p, s);
        // S = (G/eps + I)^-1 G/eps, eps = 1e-5 (model.coefficients, SURVEY Appendix A5): G on the device,
        // the one-off K x K solve on the host
        m->S.alloc((size_t)Kp * Kp);
        DevBuf<double> dG;
        dG.alloc((size_t)Kp * Kp);
        ModelDev md = m->dev();
        launch_gram(md, dG.p, s);
        std::vector<double> G((size_t)Kp * Kp), A((size_t)K * K), S((size_t)Kp * Kp, 0.0);
        download(G.data(), dG.p, G.size(), s);
        sync_stream(ctx);
        const double eps = 1e-5;
        for (int i = 0; i < K; i++)
            for (int j = 0; j < K; j++) A[(size_t)i * K + j] = G[(size_t)i * Kp + j] / eps + (i == j ? 1.0 : 0.0);
        // Cholesky A = L L^T (host, double)
        for (int j = 0; j < K; j++) {
            double d = A[(size_t)j * K + j];
            for (int k = 0; k < j; k++) d -= A[(size_t)j * K + k] * A[(size_t)j * K + k];
            ICP_REQUIRE(d > 0.0, "Gram matrix of the basis is not positive definite");
            d = std::sqrt(d);
            A[(size_t)j * K + j] = d;
            for (int i = j + 1; i < K; i++) {
                double t = A[(size_t)i * K + j];
                for (int k = 0; k < j; k++) t -= A[(size_t)i * K + k] * A[(size_t)j * K + k];
                A[(size_t)i * K + j] = t / d;
            }
        }
        std::vector<double> col(K);
        for (int c = 0; c < K; c++) {  // solve A s = G[:, c] / eps
            for (int i = 0; i < K; i++) {
                double t = G[(size_t)i * Kp + c] / eps;
                for (int k = 0; k < i; k++) t -= A[(size_t)i * K + k] * col[k];
                col[i] = t / A[(size_t)i * K + i];
            }
            for (int i = K - 1; i >= 0; i--) {
                double t = col[i];
                for (int k = i + 1; k < K; k++) t -= A[(size_t)k * K + i] * col[k];
                col[i] = t / A[(size_t)i * K + i];
            }
            for (int i = 0; i < K; i++) S[(size_t)i * Kp + c] = col[i];
        }
        for (int i = 0; i < K; i++)  // symmetrise the rounding noise (S is symmetric in exact arithmetic)
            for (int j = 0; j < i; j++) {
                double a = 0.5 * (S[(size_t)i * Kp + j] + S[(size_t)j * Kp + i]);
                S[(size_t)i * Kp + j] = S[(size_t)j * Kp + i] = a;
            }
        for (int i = K; i < Kp; i++) S[(size_t)i * Kp + i] = 1.0;
        m->S.upload(S.data(), S.size(), s);
        // query structures over the model mesh: topology from the reference, boxes refit per sample
        m->scale = std::max(max_abs(ref_xyz, n3) * 2.0, 1e-3);
        bvh_build(m->tri_bvh, 0, T, m->ref.p, m->tris.p, m->scale, s);
        bvh_build(m->vert_bvh, 1, N, m->ref.p, nullptr, m->scale, s);
        sync_stream(ctx);
        *out = m;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete m;
        return rc;
    }
}

extern "C" int32_t icp_model_destroy(icp_model m) {
    if (!m) return ICP_OK;
    icp_ctx _ctx = m->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_REQUIRE(m->refs == 0, "model is still referenced by " + std::to_string(m->refs) + " proposal / evaluator / chain handle(s): destroy those first");
        sync_stream(_ctx);
        delete m;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_model_rank(icp_model m, int32_t *K) {
    if (!m || !K) return ICP_ERR_INVALID_ARGUMENT;
    *K = m->K;
    return ICP_OK;
}

// ---------------------------------------------------------------------------------------------------
// (3) target
// ---------------------------------------------------------------------------------------------------
__global__ void k_gather_tri_data(int n, const int *__restrict__ prim, const double *__restrict__ verts,
                                  const int *__restrict__ tris, double *__restrict__ out) {
    int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    int p = prim[slot];
    for (int k = 0; k < 3; k++)
        for (int d = 0; d < 3; d++) out[(size_t)slot * 10 + 3 * k + d] = verts[3 * tris[3 * p + k] + d];
    out[(size_t)slot * 10 + 9] = 0.0;
}
__global__ void k_gather_vert_data(int n, const int *__restrict__ prim, const double *__restrict__ verts,
                                   double *__restrict__ out) {
    int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    int p = prim[slot];
    out[(size_t)slot * 4] = verts[3 * p]; out[(size_t)slot * 4 + 1] = verts[3 * p + 1];
    out[(size_t)slot * 4 + 2] = verts[3 * p + 2]; out[(size_t)slot * 4 + 3] = 0.0;
}

extern "C" int32_t icp_target_create(icp_ctx ctx, int32_t Nt, int32_t Tt, const double *xyz, const int32_t *tris,
                                     icp_target *out) {
    icp_target t = nullptr;
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx != nullptr && out != nullptr, "null handle");
        CtxLock lock(ctx);
        check_mesh(Nt, Tt, xyz, tris);
        cudaStream_t s = ctx->stream;
        t = new icp_target_s();
        t->ctx = ctx; t->Nt = Nt; t->Tt = Tt;
        t->verts.upload(xyz, (size_t)3 * Nt, s);
        t->tris.upload(tris, (size_t)3 * Tt, s);
        t->h_boundary = boundary_table(Nt, Tt, tris);
        t->has_boundary = std::any_of(t->h_boundary.begin(), t->h_boundary.end(), [](uint8_t b) { return b != 0; });
        t->boundary.upload(t->h_boundary.data(), t->h_boundary.size(), s);
        {   // Scalismo vertexNormals (SURVEY Appendix A13): normalised unweighted mean of the adjacent unit cell normals
            std::vector<double> acc((size_t)3 * Nt, 0.0);
            std::vector<int> cnt(Nt, 0);
            for (int k = 0; k < Tt; k++) {
                const double *a = xyz + 3 * (size_t)tris[3 * k], *b = xyz + 3 * (size_t)tris[3 * k + 1], *c = xyz + 3 * (size_t)tris[3 * k + 2];
                const double u[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, v[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
                double n[3] = {u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0]};
                const double nrm = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
                for (int e = 0; e < 3; e++) {
                    const int vtx = tris[3 * k + e];
                    for (int d = 0; d < 3; d++) acc[(size_t)3 * vtx + d] += n[d] / nrm;
                    cnt[vtx]++;
                }
            }
            for (int vtx = 0; vtx < Nt; vtx++) {
                double n[3];
                for (int d = 0; d < 3; d++) n[d] = acc[(size_t)3 * vtx + d] / (double)cnt[vtx];
                const double nrm = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
                for (int d = 0; d < 3; d++) acc[(size_t)3 * vtx + d] = n[d] / nrm;
            }
            t->vnormals.upload(acc.data(), acc.size(), s);
            sync_stream(ctx);
        }
        double scale = std::max(max_abs(xyz, (size_t)3 * Nt), 1e-3);
        for (int d = 0; d < 3; d++) { t->lo[d] = 1e300; t->hi[d] = -1e300; }
        for (int v = 0; v < Nt; v++)
            for (int d = 0; d < 3; d++) { t->lo[d] = std::min(t->lo[d], xyz[3 * v + d]); t->hi[d] = std::max(t->hi[d], xyz[3 * v + d]); }
        bvh_build(t->tri_bvh, 0, Tt, t->verts.p, t->tris.p, scale, s);
        bvh_build(t->vert_bvh, 1, Nt, t->verts.p, nullptr, scale, s);
        {   // warp-cooperative closest point: L-ary collapse of the triangle LBVH (ICPCUDA_WIDE = 4 | 8). Off by default:
            // measured on B200 it runs at 0.41 (L = 4) / 0.30 (L = 8) of the per-thread binary walk (profiles/r2_traversal.md)
            const char *env = getenv("ICPCUDA_WIDE");
            const int L = env ? atoi(env) : 0;
            if (L == 4 || L == 8) wide_build(t->tri_bvh, t->tri_wide, L, s);
        }
        t->tri_data.alloc((size_t)t->tri_bvh.n * 10);
        t->vert_data.alloc((size_t)t->vert_bvh.n * 4);
        k_gather_tri_data<<<(t->tri_bvh.n + 127) / 128, 128, 0, s>>>(t->tri_bvh.n, t->tri_bvh.prim.p, t->verts.p, t->tris.p, t->tri_data.p);
        ICP_CUDA(cudaGetLastError());
        k_gather_vert_data<<<(t->vert_bvh.n + 127) / 128, 128, 0, s>>>(t->vert_bvh.n, t->vert_bvh.prim.p, t->verts.p, t->vert_data.p);
        ICP_CUDA(cudaGetLastError());
        sync_stream(ctx);
        *out = t;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete t;
        return rc;
    }
}

extern "C" int32_t icp_target_destroy(icp_target t) {
    if (!t) return ICP_OK;
    icp_ctx _ctx = t->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_REQUIRE(t->refs == 0, "target is still referenced by " + std::to_string(t->refs) + " proposal / evaluator / chain handle(s): destroy those first");
        sync_stream(_ctx);
        delete t;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

// ---------------------------------------------------------------------------------------------------
// (4) primitives
// ---------------------------------------------------------------------------------------------------
static NearestArgs target_tri_args(icp_target t) {
    NearestArgs a;
    a.bvh = &t->tri_bvh;
    a.prim_data = t->tri_data.p;
    a.wide = t->wide();
    a.sm_count = t->ctx->sm_count;
    return a;
}
static NearestArgs target_vert_args(icp_target t) {
    NearestArgs a;
    a.bvh = &t->vert_bvh;
    a.prim_data = t->vert_data.p;
    return a;
}

extern "C" int32_t icp_closest_point_surface(icp_target t, int64_t nq, const double *q, int32_t *tri, int32_t *feature,
                                             double *cp, double *d2) {
    ICP_API_BEGIN(t ? t->ctx : nullptr)
    ICP_REQUIRE(nq >= 0 && (nq == 0 || q != nullptr), "bad query array");
    if (nq == 0) return ICP_OK;
    cudaStream_t s = _ctx->stream;
    t->s_q.upload(q, (size_t)3 * nq, s);
    t->s_d.ensure((size_t)4 * nq);
    t->s_i.ensure((size_t)2 * nq);
    NearestArgs a = target_tri_args(t);
    a.nq = nq; a.q = t->s_q.p;
    a.out_prim = t->s_i.p; a.out_feat = t->s_i.p + nq; a.out_cp = t->s_d.p; a.out_d2 = t->s_d.p + 3 * nq;
    launch_nearest_sorted(a, t->qsort, t->lo, t->hi, s);
    download(tri, t->s_i.p, nq, s);
    download(feature, t->s_i.p + nq, nq, s);
    download(cp, t->s_d.p, 3 * nq, s);
    download(d2, t->s_d.p + 3 * nq, nq, s);
    sync_stream(_ctx);
    ICP_API_END
}

extern "C" int32_t icp_closest_point_surface_device(icp_target t, int64_t nq, const double *q_dev, int32_t *tri_dev,
                                                    double *cp_dev, double *d2_dev) {
    ICP_API_BEGIN(t ? t->ctx : nullptr)
    ICP_REQUIRE(nq >= 0 && (nq == 0 || q_dev != nullptr), "bad query array");
    if (nq == 0) return ICP_OK;
    NearestArgs a = target_tri_args(t);
    a.nq = nq; a.q = q_dev; a.out_prim = tri_dev; a.out_cp = cp_dev; a.out_d2 = d2_dev;
    launch_nearest_sorted(a, t->qsort, t->lo, t->hi, _ctx->stream);
    sync_stream(_ctx);
    ICP_API_END
}

extern "C" int32_t icp_closest_vertex(icp_target t, int64_t nq, const double *q, int32_t *id, double *d2) {
    ICP_API_BEGIN(t ? t->ctx : nullptr)
    ICP_REQUIRE(nq >= 0 && (nq == 0 || q != nullptr), "bad query array");
    if (nq == 0) return ICP_OK;
    cudaStream_t s = _ctx->stream;
    t->s_q.upload(q, (size_t)3 * nq, s);
    t->s_d.ensure((size_t)nq);
    t->s_i.ensure((size_t)nq);
    NearestArgs a = target_vert_args(t);
    a.nq = nq; a.q = t->s_q.p; a.out_prim = t->s_i.p; a.out_d2 = t->s_d.p;
    launch_nearest(a, s);
    download(id, t->s_i.p, nq, s);
    download(d2, t->s_d.p, nq, s);
    sync_stream(_ctx);
    ICP_API_END
}

extern "C" int32_t icp_target_boundary_flags(icp_target t, uint8_t *flags) {
    if (!t || !flags) return ICP_ERR_INVALID_ARGUMENT;
    memcpy(flags, t->h_boundary.data(), (size_t)t->Nt);
    return ICP_OK;
}

extern "C" int32_t icp_model_boundary_flags(icp_model m, uint8_t *flags) {
    if (!m || !flags) return ICP_ERR_INVALID_ARGUMENT;
    memcpy(flags, m->h_boundary.data(), (size_t)m->N);
    return ICP_OK;
}

static void upload_theta(icp_model m, int C, const double *theta, DevBuf<double> &buf, cudaStream_t s) {
    ICP_REQUIRE(C >= 0 && (C == 0 || theta != nullptr), "bad theta array");
    buf.upload(theta, (size_t)C * (m->K + kTheta0), s);
}

extern "C" int32_t icp_reconstruct(icp_model m, int32_t C, const double *theta, double *xyz) {
    ICP_API_BEGIN(m ? m->ctx : nullptr)
    if (C == 0) return ICP_OK;
    ICP_REQUIRE(xyz != nullptr, "xyz is null");
    cudaStream_t s = _ctx->stream;
    upload_theta(m, C, theta, m->s_theta, s);
    m->s_X.ensure((size_t)C * m->N * 3);
    launch_reconstruct(m->dev(), C, m->s_theta.p, m->s_X.p, s);
    download(xyz, m->s_X.p, (size_t)C * m->N * 3, s);
    sync_stream(_ctx);
    ICP_API_END
}

extern "C" int32_t icp_vertex_normals(icp_model m, int32_t C, const double *theta, double *normals) {
    ICP_API_BEGIN(m ? m->ctx : nullptr)
    if (C == 0) return ICP_OK;
    ICP_REQUIRE(normals != nullptr, "normals is null");
    cudaStream_t s = _ctx->stream;
    upload_theta(m, C, theta, m->s_theta, s);
    size_t n = (size_t)C * m->N * 3;
    m->s_X.ensure(n);
    m->s_d.ensure(n);
    launch_reconstruct(m->dev(), C, m->s_theta.p, m->s_X.p, s);
    launch_vertex_normals(m->dev(), C, m->s_X.p, m->s_d.p, s);
    download(normals, m->s_d.p, n, s);
    sync_stream(_ctx);
    ICP_API_END
}

extern "C" int32_t icp_model_closest_point_surface(icp_model m, int32_t C, const double *theta, int64_t nq,
                                                   const double *q, int32_t *tri, int32_t *feature, double *cp,
                                                   double *d2) {
    ICP_API_BEGIN(m ? m->ctx : nullptr)
    ICP_REQUIRE(nq >= 0 && (nq == 0 || q != nullptr), "bad query array");
    if (C == 0 || nq == 0) return ICP_OK;
    cudaStream_t s = _ctx->stream;
    upload_theta(m, C, theta, m->s_theta, s);
    size_t tot = (size_t)C * nq;
    m->s_X.ensure((size_t)C * m->N * 3);
    m->s_q.upload(q, (size_t)3 * nq, s);
    m->s_d.ensure(4 * tot);
    m->s_i.ensure(2 * tot);
    launch_reconstruct(m->dev(), C, m->s_theta.p, m->s_X.p, s);
    bvh_refit(m->tri_bvh, C, m->s_X.p, m->N, m->tris.p, s);
    NearestArgs a;
    a.bvh = &m->tri_bvh; a.X = m->s_X.p; a.tris = m->tris.p; a.N = m->N;
    a.C = C; a.nq = nq; a.q = m->s_q.p;
    a.out_prim = m->s_i.p; a.out_feat = m->s_i.p + tot; a.out_cp = m->s_d.p; a.out_d2 = m->s_d.p + 3 * tot;
    launch_nearest(a, s);
    download(tri, m->s_i.p, tot, s);
    download(feature, m->s_i.p + tot, tot, s);
    download(cp, m->s_d.p, 3 * tot, s);
    download(d2, m->s_d.p + 3 * tot, tot, s);
    sync_stream(_ctx);
    ICP_API_END
}

extern "C" int32_t icp_model_closest_vertex(icp_model m, int32_t C, const double *theta, int64_t nq, const double *q,
                                            int32_t *id, double *d2) {
    ICP_API_BEGIN(m ? m->ctx : nullptr)
    ICP_REQUIRE(nq >= 0 && (nq == 0 || q != nullptr), "bad query array");
    if (C == 0 || nq == 0) return ICP_OK;
    cudaStream_t s = _ctx->stream;
    upload_theta(m, C, theta, m->s_theta, s);
    size_t tot = (size_t)C * nq;
    m->s_X.ensure((size_t)C * m->N * 3);
    m->s_q.upload(q, (size_t)3 * nq, s);
    m->s_d.ensure(tot);
    m->s_i.ensure(tot);
    launch_reconstruct(m->dev(), C, m->s_theta.p, m->s_X.p, s);
    bvh_refit(m->vert_bvh, C, m->s_X.p, m->N, nullptr, s);
    NearestArgs a;
    a.bvh = &m->vert_bvh; a.X = m->s_X.p; a.N = m->N;
    a.C = C; a.nq = nq; a.q = m->s_q.p; a.out_prim = m->s_i.p; a.out_d2 = m->s_d.p;
    launch_nearest(a, s);
    download(id, m->s_i.p, tot, s);
    download(d2, m->s_d.p, tot, s);
    sync_stream(_ctx);
    ICP_API_END
}

// ---------------------------------------------------------------------------------------------------
// (5) ICP proposal
// ---------------------------------------------------------------------------------------------------
// Order in which the closest-point kernel walks a list of model points: Morton order of their reference positions,
// so that the 32 queries of a warp stay close together in the target tree (results keep the caller's order).
static std::vector<int> morton_perm(const std::vector<double> &ref, const int32_t *ids, int n) {
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int i = 0; i < n; i++)
        for (int d = 0; d < 3; d++) { double x = ref[(size_t)3 * ids[i] + d]; lo[d] = std::min(lo[d], x); hi[d] = std::max(hi[d], x); }
    std::vector<std::pair<uint32_t, int>> key(n);
    for (int i = 0; i < n; i++) {
        uint32_t code = 0;
        uint32_t q[3];
        for (int d = 0; d < 3; d++) {
            double f = hi[d] > lo[d] ? (ref[(size_t)3 * ids[i] + d] - lo[d]) / (hi[d] - lo[d]) : 0.0;
            q[d] = (uint32_t)(std::min(std::max(f, 0.0), 1.0) * 1023.0);
        }
        for (int b = 9; b >= 0; b--)
            for (int d = 0; d < 3; d++) code = (code << 1) | ((q[d] >> b) & 1u);
        key[i] = {code, i};
    }
    std::sort(key.begin(), key.end());
    std::vector<int> perm(n);
    for (int i = 0; i < n; i++) perm[i] = key[i].second;
    return perm;
}

static void check_ids(int N, const int32_t *ids, int n) {
    ICP_REQUIRE(n >= 0 && (n == 0 || ids != nullptr), "bad id list");
    for (int i = 0; i < n; i++) ICP_REQUIRE(ids[i] >= 0 && ids[i] < N, "model point id out of range");
}

extern "C" int32_t icp_proposal_create(icp_model m, icp_target t, const icp_proposal_params *params,
                                       const int32_t *model_point_ids, int32_t n_ids, const double *target_points,
                                       int32_t n_tp, icp_proposal *out) {
    icp_proposal p = nullptr;
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(m && t && params && out, "null argument");
        ICP_REQUIRE(m->ctx == t->ctx, "model and target belong to different contexts");
        CtxLock lock(_ctx);
        ICP_REQUIRE(params->direction == ICP_MODEL_SAMPLING || params->direction == ICP_TARGET_SAMPLING, "bad direction");
        ICP_REQUIRE(params->step_length != 0.0 && std::isfinite(params->step_length), "step_length must be finite and non-zero");
        ICP_REQUIRE(params->tangential_noise > 0 && params->noise_along_normal > 0, "noise std-devs must be > 0");
        ICP_REQUIRE(params->factor == ICP_FACTOR_CHOLESKY || params->factor == ICP_FACTOR_SVD, "bad covariance factor");
        ICP_REQUIRE(params->rank_update == ICP_RANK_UPDATE_FP64 || params->rank_update == ICP_RANK_UPDATE_INT8, "bad rank_update mode");
        if (params->factor == ICP_FACTOR_SVD)
            for (double v : m->h_var) ICP_REQUIRE(v > 0.0, "ICP_FACTOR_SVD needs strictly positive variances");
        check_ids(m->N, model_point_ids, n_ids);
        ICP_REQUIRE(n_tp >= 0 && (n_tp == 0 || target_points != nullptr), "bad target point list");
        p = new icp_proposal_s();
        p->model = m; p->target = t; p->prm = *params; p->n_ids = n_ids; p->n_tp = n_tp;
        p->ids.upload(model_point_ids, n_ids, _ctx->stream);
        if (n_ids > 0) { std::vector<int> pm = morton_perm(m->h_ref, model_point_ids, n_ids); p->qperm.upload(pm.data(), pm.size(), _ctx->stream); sync_stream(_ctx); }
        p->tp.upload(target_points, (size_t)3 * n_tp, _ctx->stream);
        // constant-Gram fast path: model sampling, anisotropic noise with sd_n <= sd_t (kappa >= 0)
        {
            const char *env = getenv("ICPCUDA_NO_GRAM_FAST");
            if (params->direction == ICP_MODEL_SAMPLING && n_ids > 0 && params->noise_along_normal <= params->tangential_noise &&
                !(env && env[0] == '1')) {
                p->Gs.alloc((size_t)m->Kp * m->Kp);
                launch_gram_rows(m->dev(), n_ids, p->ids.p, p->Gs.p, _ctx->stream);
                p->gram_fast = true;
                p->Qsub.alloc((size_t)n_ids * (3 * m->Kp + 2));
                launch_pack_obs_rows(n_ids, m->Kp, p->ids.p, m->Qhat.p, p->Qsub.p, _ctx->stream);
            }
        }
        sync_stream(_ctx);
        m->refs++; t->refs++;
        { std::lock_guard<std::mutex> g(m->props_mu); m->proposals.push_back(p); }
        *out = p;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete p;
        return rc;
    }
}

extern "C" int32_t icp_proposal_destroy(icp_proposal p) {
    if (!p) return ICP_OK;
    icp_ctx _ctx = p->model->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_REQUIRE(p->refs == 0, "proposal is still used by a chain: destroy the chain first");
        {
            std::lock_guard<std::mutex> g(p->model->props_mu);
            auto &v = p->model->proposals;
            v.erase(std::remove(v.begin(), v.end(), p), v.end());
        }
        drain_calls(p);
        {
            std::lock_guard<std::mutex> g(p->bg_mu);
            if (p->bg_busy) { cudaEventSynchronize(p->bg_ev); p->bg_busy = false; }
        }
        sync_stream(_ctx);
        p->model->refs--; p->target->refs--;
        delete p;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

namespace icp {

// currentMesh.pointSet.findClosestPoint for C chains: the vertex BVH refitted and walked in shared memory (default), the
// FP32-screened brute force when the tree does not fit, the global-memory refit + traversal as the last resort.
// ICPCUDA_NEAREST_VERTEX = tree | brute | bvh forces one of them (all three return the same answers).
static const std::string &nearest_vertex_mode() {
    static const std::string mode = getenv("ICPCUDA_NEAREST_VERTEX") ? getenv("ICPCUDA_NEAREST_VERTEX") : "";
    return mode;
}

// true when nearest_model_vertex never falls through to the refit of the model's own vertex BVH (scratch shared by every
// user of the model): the shared-memory tree or the brute-force kernel takes every call
static bool nearest_model_vertex_self_contained(icp_model m) {
    const std::string &mode = nearest_vertex_mode();
    if ((mode.empty() || mode == "tree") && nearest_vertex_tree_fits(m->vert_bvh, m->N)) return true;
    return mode != "bvh" && nearest_vertex_brute_fits(m->N);
}

// a per-call pipeline that only reads its model and target and writes the handle's own work buffers
static bool proposal_self_contained(icp_proposal p) {
    return p->prm.direction != ICP_TARGET_SAMPLING || nearest_model_vertex_self_contained(p->model);
}
static bool evaluator_self_contained(icp_evaluator e) {
    // target -> model distances refit the model's triangle BVH (and the collective evaluator its vertex BVH)
    return e->prm.kind == ICP_EVAL_ACCEPT_ALL || (e->prm.kind != ICP_EVAL_HAUSDORFF && e->prm.mode == ICP_MODEL_TO_TARGET);
}

void nearest_model_vertex(icp_model m, int C, const double *d_X, int64_t nq, const double *d_q, int q_per_chain, int *d_seed,
                          int *d_prim, cudaStream_t s) {
    const std::string &mode = nearest_vertex_mode();
    if ((mode.empty() || mode == "tree") &&
        launch_nearest_vertex_tree(m->vert_bvh, m->N, C, d_X, nq, d_q, q_per_chain, d_seed, d_prim, nullptr, s))
        return;
    if (mode != "bvh" && launch_nearest_vertex_brute(m->N, C, d_X, nq, d_q, q_per_chain, m->scale, d_prim, nullptr, s)) return;
    bvh_refit(m->vert_bvh, C, d_X, m->N, nullptr, s);
    NearestArgs a;
    a.bvh = &m->vert_bvh; a.X = d_X; a.N = m->N; a.C = C; a.nq = nq; a.q = d_q; a.q_per_chain = q_per_chain;
    a.out_prim = d_prim; a.seed_slot = d_seed;
    launch_nearest(a, s);
}

void posterior_pipeline(icp_proposal p, int C, const double *d_theta, const double *d_X, PosteriorWork &w, double *d_L,
                        double *d_mu, const int *d_out_slot, cudaStream_t s, const SharedCp *shared, double *d_W,
                        const QuadArgs *qa, bool ymean, const TargetSet *ts) {
    if (C <= 0) return;
    icp_model m = p->model;
    icp_target t = p->target;
    const bool has_boundary = ts ? ts->has_boundary : t->has_boundary;
    const int Kp = m->Kp;
    ModelDev md = m->dev();
    if (!d_X) {
        w.X.ensure((size_t)C * m->N * 3);
        launch_reconstruct(md, C, d_theta, w.X.p, s);
        d_X = w.X.p;
    }
    const bool tsamp = p->prm.direction == ICP_TARGET_SAMPLING;
    int n = tsamp ? p->n_tp : p->n_ids;
    size_t tot = (size_t)C * std::max(n, 1);
    w.vid.ensure(tot); w.F.ensure(9 * tot); w.y.ensure(3 * tot); w.nobs.ensure(2 * (size_t)C);
    w.M.ensure((size_t)C * Kp * Kp); w.b.ensure((size_t)C * Kp); w.status.ensure(C);
    ObsArgs oa{};
    oa.m = md; oa.prm = p->prm; oa.C = C; oa.theta = d_theta; oa.X = d_X;
    if (tsamp) {
        // :118 currentMesh.pointSet.findClosestPoint(targetPoint): vertex BVH refit to the current meshes
        w.prim.ensure(tot);
        if (w.seed.n < tot) { w.seed.ensure(tot); ICP_CUDA(cudaMemsetAsync(w.seed.p, 0xFF, sizeof(int) * tot, s)); }
        const double *tp = ts ? ts->tp : p->tp.p;
        nearest_model_vertex(m, C, d_X, n, tp, ts ? 1 : 0, w.seed.p, w.prim.p, s);
        oa.tp = tp; oa.tp_per_chain = ts ? 1 : 0; oa.near_vid = w.prim.p;
    } else {
        // :97 target.operations.closestPointOnSurface(currentMeshPoint)
        const bool need_flags = p->prm.boundary_aware && has_boundary;
        if (shared && !need_flags) {
            oa.cp = shared->cp; oa.cp_stride = shared->stride; oa.cp_map = shared->map;
        } else {
            w.cp.ensure(3 * tot);
            NearestArgs a;
            a.bvh = &t->tri_bvh; a.prim_data = t->tri_data.p; a.wide = t->wide(); a.sm_count = t->ctx->sm_count; a.C = C; a.nq = n;
            a.Xq = d_X; a.q_ids = p->ids.p; a.Nq = m->N; a.out_cp = w.cp.p; a.perm = p->qperm.p;
            if (ts) { a.mt_rec = ts->rec; a.mt_idx = ts->tidx; }
            if (w.seed.n < tot) { w.seed.ensure(tot); ICP_CUDA(cudaMemsetAsync(w.seed.p, 0xFF, sizeof(int) * tot, s)); }
            a.seed_slot = w.seed.p;
            launch_nearest(a, s);
            oa.cp = w.cp.p; oa.cp_stride = n; oa.cp_map = nullptr;
        }
        oa.ids = p->ids.p; oa.cp_on_boundary = nullptr;
        if (need_flags) {
            // :98-99 target.pointSet.findClosestPoint(targetPoint).id -> pointIsOnBoundary
            w.prim.ensure(tot); w.flags.ensure(tot);
            NearestArgs v;
            v.bvh = &t->vert_bvh; v.prim_data = t->vert_data.p; v.C = C; v.nq = n; v.q = w.cp.p; v.q_per_chain = 1;
            v.out_prim = w.prim.p;
            if (ts) { v.mt_rec = ts->rec; v.mt_idx = ts->tidx; }
            launch_nearest(v, s);
            launch_lookup_flags((int64_t)C * n, w.prim.p, t->boundary.p, t->Nt, w.flags.p, s, ts ? ts->rec : nullptr,
                                ts ? ts->tidx : nullptr, n);
            oa.cp_on_boundary = w.flags.p;
        }
    }
    ObsDev od{n, w.vid.p, w.F.p, w.y.p, w.nobs.p};
    od.nrows = w.nobs.p + C;
    launch_observations(oa, od, s);
    // every observation is kept (no boundary filtering possible) -> the Gram part of M is the proposal's constant
    const bool all_kept = !tsamp && !(p->prm.boundary_aware && has_boundary);
    GramFast gf{p->Gs.p, 1.0 / (p->prm.tangential_noise * p->prm.tangential_noise),
                std::sqrt(std::max(0.0, 1.0 - (p->prm.noise_along_normal * p->prm.noise_along_normal) /
                                                  (p->prm.tangential_noise * p->prm.tangential_noise)))};
    const GramFast *gfp = (p->gram_fast && all_kept) ? &gf : nullptr;
    w.Mp.ensure((size_t)C * (Kp / 8) * (Kp / 8 + 1) / 2 * 64);
    bool quad_done = false;
    // ICPCUDA_RANK_UPDATE=int8: the rank update on the tcgen05 INT8 tensor cores (split-integer emulation of the FP64 product,
    // 1e-8 on the posterior mean; tc_i8.cu) instead of the FP64 tensor pipe. Not for grouped observations (their rows are
    // scaled by sqrt(multiplicity), outside the column bound).
    static const std::string ru_env = getenv("ICPCUDA_RANK_UPDATE") ? getenv("ICPCUDA_RANK_UPDATE") : "";
    const bool want_i8 = ru_env == "int8" || (ru_env != "fp64" && p->prm.rank_update == ICP_RANK_UPDATE_INT8);
    const bool grouped = tsamp && 2 * (long long)n >= m->N;
    I8Scale sc{0.0, 0.0, 0.0};
    if (want_i8 && !grouped) {
        // whitened rows |F_d . Qhat_v[:, j]| <= max(1 / sd_n, 1 / sd_t) resp. sqrt(kappa) (constant-Gram rows): scaled to 2^30
        const double top = 1073741824.0 * (1.0 - 1e-6);
        if (gfp) {
            const double kr = gf.row_scale / p->prm.noise_along_normal;
            if (kr > 0.0) { const double fs = top / kr; sc = I8Scale{gf.row_scale * fs, 16777216.0 / (fs * fs), 1.0}; }
        } else {
            const double fs = top / std::max(1.0 / p->prm.noise_along_normal, 1.0 / p->prm.tangential_noise);
            sc = I8Scale{fs, 16777216.0 / (fs * fs), 1.0 / fs};
        }
    }
    if (want_i8 && !grouped &&
        launch_rank_update_i8(md, C, od, gfp, I8Model{m->Qhat.p, m->col_norm.p, p->Qsub.p}, sc, w.Mp.p, w.b.p, m->ctx->sm_count, s)) {
        launch_cholesky_packed(C, Kp, w.Mp.p, w.b.p, w.want_M ? w.M.p : nullptr, d_L, d_mu, d_out_slot, w.status.p, qa, ymean, s);
        quad_done = qa != nullptr;
    } else
    if (!launch_posterior_fused(md, C, od, gfp, w.want_M ? w.M.p : nullptr, d_L, d_mu, d_out_slot, w.status.p, w.Mp.p, w.b.p, s, qa,
                                &quad_done, ymean)) {
        launch_posterior_build(md, C, od, w.M.p, w.b.p, s, gfp);
        launch_cholesky_solve(C, m->K, Kp, w.M.p, w.b.p, d_L, d_mu, d_out_slot, w.status.p, s, w.Mp.p, qa, &quad_done, ymean);
    }
    if (qa && !quad_done) launch_quad_form(C, Kp, d_L, d_mu, d_out_slot, *qa, ymean, s);
    if (d_W) launch_svd_factor(C, m->K, Kp, d_L, m->sqrt_var.p, d_out_slot, d_W, w.svd_scratch, s);
}

}  // namespace icp

static void strip_pad_vec(const std::vector<double> &src, int C, int K, int Kp, double *dst) {
    for (int c = 0; c < C; c++)
        for (int j = 0; j < K; j++) dst[(size_t)c * K + j] = src[(size_t)c * Kp + j];
}

extern "C" int32_t icp_posterior(icp_proposal p, int32_t C, const double *theta, double *mu, double *M, int32_t *n_obs) {
    ICP_API_BEGIN_HANDLE(icp_proposal_s, p, p && proposal_self_contained(p))
    if (C == 0) return ICP_OK;
    icp_model m = p->model;
    const int K = m->K, Kp = m->Kp;
    upload_theta(m, C, theta, cs.s_theta, s);
    DevBuf<double> &dL = cs.s_L, &dmu = cs.s_mu;   // kept on the call slot: cudaFree would synchronise the whole device
    dL.ensure((size_t)C * Kp * Kp);
    dmu.ensure((size_t)C * Kp);
    cs.work.want_M = M != nullptr;
    posterior_pipeline(p, C, cs.s_theta.p, nullptr, cs.work, dL.p, dmu.p, nullptr, s);
    cs.work.want_M = false;
    std::vector<double> hmu((size_t)C * Kp), hM;
    std::vector<int> hn(C), hst(C);
    download(hmu.data(), dmu.p, hmu.size(), s);
    if (M) { hM.resize((size_t)C * Kp * Kp); download(hM.data(), cs.work.M.p, hM.size(), s); }
    download(hn.data(), cs.work.nobs.p, C, s);
    download(hst.data(), cs.work.status.p, C, s);
    ICP_CUDA(cudaStreamSynchronize(s));
    if (mu) strip_pad_vec(hmu, C, K, Kp, mu);
    if (M)
        for (int c = 0; c < C; c++)
            for (int i = 0; i < K; i++)
                for (int j = 0; j < K; j++) M[((size_t)c * K + i) * K + j] = hM[((size_t)c * Kp + i) * Kp + j];
    if (n_obs) std::copy(hn.begin(), hn.end(), n_obs);
    ICP_API_END
}

// ---- per-call entries as replayed graphs (run_call_graph) ----------------------------------------------------------
static bool call_graphs_enabled() {
    // ICPCUDA_CALL_GRAPH=0: launch the kernels of a per-call entry directly. Also under Nsight Compute (it sets
    // NV_COMPUTE_PROFILER_PERFWORKS_DIR in the target process): stream capture from several host threads aborts inside the
    // profiler's injection library (ncu 2025.2.1, measured: profiles/r2_session3.md section 1), and a profile wants the
    // kernels one by one anyway.
    static const bool on = !(getenv("ICPCUDA_CALL_GRAPH") && getenv("ICPCUDA_CALL_GRAPH")[0] == '0') &&
                           !getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR");
    return on;
}
enum CallKind : uint64_t { CALL_POSTERIOR = 1, CALL_PROPOSE, CALL_LOG_TRANSITION, CALL_EVAL };
static uint64_t call_key(CallKind kind, int C) { return ((uint64_t)kind << 56) | (uint64_t)(uint32_t)C; }
// every allocation a captured proposal call bakes in (DevBuf / PinnedBuf ids)
static std::vector<uint64_t> proposal_call_ptrs(icp_proposal p, icp_proposal_s::Call &cs) {
    const PosteriorWork &w = cs.work;
    return {w.X.id, w.cp.id, w.d2.id, w.prim.id, w.seed.id, w.flags.id, w.vid.id, w.F.id, w.y.id, w.nobs.id, w.M.id, w.b.id, w.Mp.id,
            w.status.id, w.svd_scratch.id, cs.s_theta.id, cs.s_theta2.id, cs.s_z.id, cs.s_out.id, cs.s_slot.id, cs.s_qslot.id,
            cs.h_in.id, cs.h_out.id, cs.h_aux.id, p->cache_L.id, p->cache_mu.id, p->cache_W.id};
}
static std::vector<uint64_t> evaluator_call_ptrs(icp_evaluator_s::Call &cs) {
    const EvalWork &w = cs.work;
    return {w.X.id, w.cp_m2t.id, w.d2_m2t.id, w.cp_t2m.id, w.d2_t2m.id, w.prim.id, w.seed_m2t.id, w.seed_t2m.id, w.skip_m2t.id,
            w.skip_t2m.id, w.hd_max.id, cs.s_theta.id, cs.s_values.id, cs.s_status.id, cs.h_in.id, cs.h_out.id};
}
static void h2d(void *d, const void *h, size_t bytes, cudaStream_t s) {
    if (bytes) ICP_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s));
}
static void d2h(void *h, const void *d, size_t bytes, cudaStream_t s) {
    if (bytes) ICP_CUDA(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s));
}

// Memoize(icpPosterior, 20) (NonRigidIcpProposal.scala:49): per-handle cache keyed by the bytes of theta, shared by the
// concurrent calls on the handle (Scalismo's Memoize is shared between the fitting threads the same way).
// PosteriorLease holds the cache slot of every chain of one call: slots are pinned (never evicted) until it goes out of
// scope; posteriors that are missing are computed in one batch on the call's stream, and a call that hits a slot another
// call is still computing waits for it.
namespace {
// waits for the background posterior of q (bg_mu held) and publishes its cache slots
void bg_finalize_locked(icp_proposal q) {
    if (!q->bg_busy) return;
    const cudaError_t e = cudaEventSynchronize(q->bg_ev);
    {
        std::lock_guard<std::mutex> g(q->cache_lock);
        for (size_t i = 0; i < q->bg_slots.size(); i++) {
            const int sl = q->bg_slots[i];
            if (e != cudaSuccess) { q->cache_map.erase(q->bg_keys[i]); q->slot_key[sl].clear(); }   // waiters fail on the key check
            q->slot_ready[sl] = 1;
            q->slot_bg[sl] = 0;
            q->slot_pin[sl]--;
        }
    }
    if (e != cudaSuccess) cudaGetLastError();
    q->bg_slots.clear();
    q->bg_keys.clear();
    q->bg_busy = false;
    q->cache_cv.notify_all();
}

bool prefetch_enabled() {
    static const bool on = !(getenv("ICPCUDA_PREFETCH") && getenv("ICPCUDA_PREFETCH")[0] == '0');
    return on;
}
}  // namespace


// starts the posteriors of C states on q in the background (see icp_proposal_s::bg_call); never blocks, never throws: a
// prefetch that cannot start right away (another one in flight, cache being resized, no free slot) simply does not happen
static void prefetch_posterior(icp_proposal q, int C, const double *theta_host) noexcept {
    try {
        if (!prefetch_enabled() || C > 64 || !proposal_self_contained(q)) return;
        std::unique_lock<std::mutex> bg(q->bg_mu, std::try_to_lock);
        if (!bg.owns_lock()) return;
        if (q->bg_busy) {
            if (cudaEventQuery(q->bg_ev) != cudaSuccess) { cudaGetLastError(); return; }
            bg_finalize_locked(q);
        }
        std::shared_lock<std::shared_mutex> rd(q->cache_rw, std::try_to_lock);
        if (!rd.owns_lock() || q->cache_slots < 32 + 6 * C) return;
        icp_model m = q->model;
        const int Lt = m->K + kTheta0;
        std::vector<std::string> key(C);
        for (int c = 0; c < C; c++) key[c].assign((const char *)(theta_host + (size_t)c * Lt), sizeof(double) * Lt);
        std::vector<int> miss, slots;
        {
            std::lock_guard<std::mutex> g(q->cache_lock);
            if (q->slot_bg.size() != (size_t)q->cache_slots) q->slot_bg.assign(q->cache_slots, 0);
            std::unordered_map<std::string, int> distinct;
            for (int c = 0; c < C; c++)
                if (!q->cache_map.count(key[c])) distinct.emplace(key[c], c);
            if (distinct.empty()) return;
            int free_slots = 0;
            for (int sl = 0; sl < q->cache_slots; sl++) free_slots += q->slot_pin[sl] == 0;
            if (free_slots < (int)distinct.size() + 8) return;     // leave room for the calls that are about to come
            for (auto &kv : distinct) {
                while (q->slot_pin[q->cache_next] != 0) q->cache_next = (q->cache_next + 1) % q->cache_slots;
                const int sl = q->cache_next;
                q->cache_next = (q->cache_next + 1) % q->cache_slots;
                if (!q->slot_key[sl].empty()) q->cache_map.erase(q->slot_key[sl]);
                q->slot_key[sl] = kv.first;
                q->cache_map[kv.first] = sl;
                q->slot_ready[sl] = 0;
                q->slot_bg[sl] = 1;
                q->slot_pin[sl]++;
                miss.push_back(kv.second);
                slots.push_back(sl);
            }
        }
        // from here on the slots are published as "in flight": on any failure they must be withdrawn
        q->bg_slots = slots;
        q->bg_keys.clear();
        for (int c : miss) q->bg_keys.push_back(key[c]);
        q->bg_busy = true;
        bool started = false;
        try {
            if (!q->bg_call) {
                q->bg_call.reset(new icp_proposal_s::Call());
                ICP_CUDA(cudaStreamCreateWithFlags(&q->bg_call->stream, cudaStreamNonBlocking));
            }
            if (!q->bg_ev) ICP_CUDA(cudaEventCreateWithFlags(&q->bg_ev, cudaEventDisableTiming));
            icp_proposal_s::Call &cs = *q->bg_call;
            cudaStream_t s = cs.stream;
            const int nm = (int)miss.size();
            cs.h_aux.ensure(sizeof(double) * (size_t)nm * Lt + sizeof(int) * (size_t)nm);
            double *hth = reinterpret_cast<double *>(cs.h_aux.p);
            int *hslot = reinterpret_cast<int *>(hth + (size_t)nm * Lt);
            for (int i = 0; i < nm; i++) {
                memcpy(hth + (size_t)i * Lt, theta_host + (size_t)miss[i] * Lt, sizeof(double) * Lt);
                hslot[i] = slots[i];
            }
            cs.s_theta2.ensure((size_t)nm * Lt);
            cs.s_slot.ensure(nm);
            run_call_graph(cs, call_graphs_enabled(), ((uint64_t)1 << 56) | (uint64_t)(uint32_t)nm, proposal_call_ptrs(q, cs), s, [&] {
                ICP_CUDA(cudaMemcpyAsync(cs.s_theta2.p, hth, sizeof(double) * (size_t)nm * Lt, cudaMemcpyHostToDevice, s));
                ICP_CUDA(cudaMemcpyAsync(cs.s_slot.p, hslot, sizeof(int) * (size_t)nm, cudaMemcpyHostToDevice, s));
                posterior_pipeline(q, nm, cs.s_theta2.p, nullptr, cs.work, q->cache_L.p, q->cache_mu.p, cs.s_slot.p, s, nullptr,
                                   q->prm.factor == ICP_FACTOR_SVD ? q->cache_W.p : nullptr);
            });
            ICP_CUDA(cudaEventRecord(q->bg_ev, s));
            started = true;
        } catch (...) {
            cudaGetLastError();
        }
        if (!started) {      // withdraw: forget the keys, wake anyone who already waits for them
            if (q->bg_call && q->bg_call->stream) cudaStreamSynchronize(q->bg_call->stream);
            {
                std::lock_guard<std::mutex> g(q->cache_lock);
                for (size_t i = 0; i < q->bg_slots.size(); i++) {
                    const int sl = q->bg_slots[i];
                    q->cache_map.erase(q->bg_keys[i]); q->slot_key[sl].clear();
                    q->slot_ready[sl] = 1; q->slot_bg[sl] = 0; q->slot_pin[sl]--;
                }
            }
            q->bg_slots.clear(); q->bg_keys.clear(); q->bg_busy = false;
            q->cache_cv.notify_all();
        }
    } catch (...) {
    }
}

namespace {
struct PosteriorLease {
    icp_proposal p;
    std::shared_lock<std::shared_mutex> rd;   // the slot arrays stay where they are
    std::vector<int> slot;                    // [C]
    std::vector<int> pinned;                  // distinct slots this call pinned
    PosteriorLease(icp_proposal p_, icp_proposal_s::Call &cs, int C, const double *theta_host, cudaStream_t s, bool graph);
    ~PosteriorLease() { unpin(); }
    void unpin() {
        if (pinned.empty()) return;
        {
            std::lock_guard<std::mutex> g(p->cache_lock);
            for (int sl : pinned) p->slot_pin[sl]--;
        }
        pinned.clear();
        p->cache_cv.notify_all();
    }
};

PosteriorLease::PosteriorLease(icp_proposal p_, icp_proposal_s::Call &cs, int C, const double *theta_host, cudaStream_t s, bool graph)
    : p(p_) {
    icp_model m = p->model;
    const int Kp = m->Kp, Lt = m->K + kTheta0;
    // the 20 states Memoize keeps and room for a handful of concurrent calls of this size (a call that finds every slot pinned
    // by others waits for one of them to finish, holding nothing)
    const int want = 32 + 6 * C;
    rd = std::shared_lock<std::shared_mutex>(p->cache_rw);
    while (p->cache_slots < want) {
        rd.unlock();
        {
            std::unique_lock<std::shared_mutex> wr(p->cache_rw);   // no call in flight holds a slot now
            { std::lock_guard<std::mutex> bg(p->bg_mu); bg_finalize_locked(p); }   // nor the background computation
            if (p->cache_slots < want) {
                p->slot_bg.assign(want, 0);
                p->cache_map.clear();
                p->slot_key.assign(want, std::string());
                p->slot_pin.assign(want, 0);
                p->slot_ready.assign(want, 0);
                p->cache_L.alloc((size_t)want * Kp * Kp);
                p->cache_mu.alloc((size_t)want * Kp);
                if (p->prm.factor == ICP_FACTOR_SVD) p->cache_W.alloc((size_t)want * Kp * Kp);
                p->cache_next = 0;
                p->cache_slots = want;
            }
        }
        rd.lock();
    }
    std::vector<std::string> key(C);
    for (int c = 0; c < C; c++) key[c].assign((const char *)(theta_host + (size_t)c * Lt), sizeof(double) * Lt);
    slot.assign(C, -1);
    std::vector<int> miss, wait_for;
    {
        std::unique_lock<std::mutex> g(p->cache_lock);
        for (;;) {
            // hits and distinct missing keys first, nothing is modified until every miss can have a slot
            std::unordered_map<std::string, int> distinct_miss;
            std::vector<char> mine(p->cache_slots, 0);
            for (int c = 0; c < C; c++) {
                auto it = p->cache_map.find(key[c]);
                if (it != p->cache_map.end()) mine[it->second] = 1;
                else distinct_miss.emplace(key[c], -1);
            }
            int free_slots = 0;
            for (int sl = 0; sl < p->cache_slots; sl++) free_slots += (p->slot_pin[sl] == 0 && !mine[sl]);
            if (free_slots < (int)distinct_miss.size()) { p->cache_cv.wait(g); continue; }   // holding nothing while waiting
            for (int c = 0; c < C; c++) {
                auto it = p->cache_map.find(key[c]);
                if (it != p->cache_map.end()) {
                    slot[c] = it->second;
                    if (!p->slot_ready[slot[c]]) wait_for.push_back(c);   // another call is computing it
                    continue;
                }
                int &sl = distinct_miss[key[c]];
                if (sl < 0) {
                    while (p->slot_pin[p->cache_next] != 0 || mine[p->cache_next]) p->cache_next = (p->cache_next + 1) % p->cache_slots;
                    sl = p->cache_next;
                    p->cache_next = (p->cache_next + 1) % p->cache_slots;
                    mine[sl] = 1;
                    if (!p->slot_key[sl].empty()) p->cache_map.erase(p->slot_key[sl]);
                    p->slot_key[sl] = key[c];
                    p->slot_ready[sl] = 0;
                    miss.push_back(c);
                }
                slot[c] = sl;
            }
            // publish the new keys only now: the lookups above must not take this call's own misses for hits
            for (int c : miss) p->cache_map[key[c]] = slot[c];
            for (int sl = 0; sl < p->cache_slots; sl++)
                if (mine[sl]) { p->slot_pin[sl]++; pinned.push_back(sl); }
            break;
        }
    }
    if (!miss.empty()) {
        const int nm = (int)miss.size();
        try {
            cs.h_aux.ensure(sizeof(double) * (size_t)nm * Lt + sizeof(int) * (size_t)nm);
            double *hth = reinterpret_cast<double *>(cs.h_aux.p);
            int *hslot = reinterpret_cast<int *>(hth + (size_t)nm * Lt);
            for (int i = 0; i < nm; i++) {
                memcpy(hth + (size_t)i * Lt, theta_host + (size_t)miss[i] * Lt, sizeof(double) * Lt);
                hslot[i] = slot[miss[i]];
            }
            cs.s_theta2.ensure((size_t)nm * Lt);
            cs.s_slot.ensure(nm);
            run_call_graph(cs, graph, call_key(CALL_POSTERIOR, nm), proposal_call_ptrs(p, cs), s, [&] {
                h2d(cs.s_theta2.p, hth, sizeof(double) * (size_t)nm * Lt, s);
                h2d(cs.s_slot.p, hslot, sizeof(int) * (size_t)nm, s);
                posterior_pipeline(p, nm, cs.s_theta2.p, nullptr, cs.work, p->cache_L.p, p->cache_mu.p, cs.s_slot.p, s, nullptr,
                                   p->prm.factor == ICP_FACTOR_SVD ? p->cache_W.p : nullptr);
            });
            ICP_CUDA(cudaStreamSynchronize(s));  // the slots are complete for every stream
        } catch (...) {
            {   // forget the keys, wake the calls waiting for these slots (they fail on the key check below)
                std::lock_guard<std::mutex> g(p->cache_lock);
                for (int c : miss) { p->cache_map.erase(key[c]); p->slot_key[slot[c]].clear(); p->slot_ready[slot[c]] = 1; }
            }
            p->cache_cv.notify_all();
            unpin();
            throw;
        }
        {
            std::lock_guard<std::mutex> g(p->cache_lock);
            for (int c : miss) p->slot_ready[slot[c]] = 1;
        }
        p->cache_cv.notify_all();
    }
    if (!wait_for.empty()) {
        bool on_bg = false;
        {
            std::lock_guard<std::mutex> g(p->cache_lock);
            for (int c : wait_for) on_bg = on_bg || (!p->slot_ready[slot[c]] && (size_t)slot[c] < p->slot_bg.size() && p->slot_bg[slot[c]]);
        }
        if (on_bg) { std::lock_guard<std::mutex> bg(p->bg_mu); bg_finalize_locked(p); }   // the speculative posterior: wait for its event
        std::unique_lock<std::mutex> g(p->cache_lock);
        for (int c : wait_for) {
            p->cache_cv.wait(g, [&] { return p->slot_ready[slot[c]] != 0; });
            if (p->slot_key[slot[c]] != key[c]) {
                g.unlock();
                unpin();
                throw StatusError{ICP_ERR_CUDA, "the posterior this call waited for failed in a concurrent call"};
            }
        }
    }
}
}  // namespace

extern "C" int32_t icp_proposal_clear_cache(icp_proposal p) {
    icp_ctx _ctx = p ? p->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        std::unique_lock<std::shared_mutex> wr(p->cache_rw);   // waits for the calls in flight
        { std::lock_guard<std::mutex> bg(p->bg_mu); bg_finalize_locked(p); }
        p->cache_map.clear();
        for (auto &k : p->slot_key) k.clear();
    ICP_API_END
}

extern "C" int32_t icp_propose(icp_proposal p, int32_t C, const double *theta, const double *z, double *theta_out) {
    const bool self_contained = p && proposal_self_contained(p);
    ICP_API_BEGIN_HANDLE(icp_proposal_s, p, self_contained)
    if (C == 0) return ICP_OK;
    ICP_REQUIRE(C > 0, "C must be >= 0");
    icp_model m = p->model;
    ICP_REQUIRE(theta && z && theta_out, "null array");
    const bool graph = self_contained && call_graphs_enabled();
    const int Lt = m->K + kTheta0;
    const size_t nth = (size_t)C * Lt, nz = (size_t)C * m->K;
    PosteriorLease post(p, cs, C, theta, s, graph);
    cs.h_in.ensure(sizeof(double) * (nth + nz) + sizeof(int) * (size_t)C);
    cs.h_out.ensure(sizeof(double) * nth);
    double *hth = reinterpret_cast<double *>(cs.h_in.p), *hz = hth + nth;
    int *hslot = reinterpret_cast<int *>(hz + nz);
    memcpy(hth, theta, sizeof(double) * nth);
    memcpy(hz, z, sizeof(double) * nz);
    memcpy(hslot, post.slot.data(), sizeof(int) * (size_t)C);
    cs.s_theta.ensure(nth); cs.s_z.ensure(nz); cs.s_qslot.ensure(C); cs.s_out.ensure(nth);
    run_call_graph(cs, graph, call_key(CALL_PROPOSE, C), proposal_call_ptrs(p, cs), s, [&] {
        h2d(cs.s_theta.p, hth, sizeof(double) * nth, s);
        h2d(cs.s_z.p, hz, sizeof(double) * nz, s);
        h2d(cs.s_qslot.p, hslot, sizeof(int) * (size_t)C, s);
        launch_propose(m->dev(), C, p->prm.step_length, cs.s_theta.p, cs.s_z.p, p->cache_L.p, p->cache_mu.p, cs.s_qslot.p,
                       cs.s_out.p, s, p->prm.factor == ICP_FACTOR_SVD ? p->cache_W.p : nullptr);
        d2h(cs.h_out.p, cs.s_out.p, sizeof(double) * nth, s);
    });
    ICP_CUDA(cudaStreamSynchronize(s));
    memcpy(theta_out, cs.h_out.p, sizeof(double) * nth);
    post.unpin();
    post.rd.unlock();
    {   // the host will ask every ICP component for the transition back from theta': start those posteriors now
        std::vector<icp_proposal> siblings;
        {
            std::lock_guard<std::mutex> g(m->props_mu);
            for (icp_proposal q : m->proposals)
                if (q->target == p->target) siblings.push_back(q);
        }
        for (icp_proposal q : siblings) prefetch_posterior(q, C, theta_out);
    }
    ICP_API_END
}

extern "C" int32_t icp_log_transition(icp_proposal p, int32_t C, const double *from, const double *to, double *out) {
    const bool self_contained = p && proposal_self_contained(p);
    ICP_API_BEGIN_HANDLE(icp_proposal_s, p, self_contained)
    if (C == 0) return ICP_OK;
    ICP_REQUIRE(C > 0, "C must be >= 0");
    icp_model m = p->model;
    ICP_REQUIRE(from && to && out, "null array");
    const bool graph = self_contained && call_graphs_enabled();
    const size_t nth = (size_t)C * (m->K + kTheta0);
    PosteriorLease post(p, cs, C, from, s, graph);
    cs.h_in.ensure(sizeof(double) * 2 * nth + sizeof(int) * (size_t)C);
    cs.h_out.ensure(sizeof(double) * (size_t)C);
    double *hfrom = reinterpret_cast<double *>(cs.h_in.p), *hto = hfrom + nth;
    int *hslot = reinterpret_cast<int *>(hto + nth);
    memcpy(hfrom, from, sizeof(double) * nth);
    memcpy(hto, to, sizeof(double) * nth);
    memcpy(hslot, post.slot.data(), sizeof(int) * (size_t)C);
    cs.s_theta.ensure(nth); cs.s_theta2.ensure(nth); cs.s_qslot.ensure(C); cs.s_out.ensure((size_t)C);
    run_call_graph(cs, graph, call_key(CALL_LOG_TRANSITION, C), proposal_call_ptrs(p, cs), s, [&] {
        h2d(cs.s_theta.p, hfrom, sizeof(double) * nth, s);
        h2d(cs.s_theta2.p, hto, sizeof(double) * nth, s);
        h2d(cs.s_qslot.p, hslot, sizeof(int) * (size_t)C, s);
        launch_log_transition(C, m->K, m->Kp, p->prm.step_length, cs.s_theta.p, cs.s_theta2.p, p->cache_L.p, p->cache_mu.p,
                              cs.s_qslot.p, cs.s_out.p, s);
        d2h(cs.h_out.p, cs.s_out.p, sizeof(double) * (size_t)C, s);
    });
    ICP_CUDA(cudaStreamSynchronize(s));
    memcpy(out, cs.h_out.p, sizeof(double) * (size_t)C);
    ICP_API_END
}

// deterministic ICP iteration: posterior mean with isotropic noise, re-projection S mu, step
__global__ void k_std_icp_step(int C, int K, int Kp, double step, const double *__restrict__ S,
                               const double *__restrict__ mu, const double *__restrict__ alpha,
                               double *__restrict__ alpha_out) {
    int c = blockIdx.x;
    for (int j = threadIdx.x; j < K; j += blockDim.x) {
        double acc = 0.0;
        for (int k = 0; k < Kp; k++) acc = fma(S[(size_t)k * Kp + j], mu[(size_t)c * Kp + k], acc);
        double a = alpha[(size_t)c * K + j];
        alpha_out[(size_t)c * K + j] = a + (acc - a) * step;  // IcpBasedSurfaceFitting.scala:84-85
    }
}

static int32_t std_icp_iteration_impl(icp_model m, icp_target t, int32_t direction, const int32_t *model_point_ids,
                                      int32_t n_ids, const double *target_points, int32_t n_tp, double sigma2,
                                      double step_length, int32_t C, const double *alpha, const double *theta, double *alpha_out);

extern "C" int32_t icp_std_icp_iteration(icp_model m, icp_target t, int32_t direction, const int32_t *model_point_ids,
                                         int32_t n_ids, const double *target_points, int32_t n_tp, double sigma2,
                                         double step_length, int32_t C, const double *alpha, double *alpha_out) {
    return std_icp_iteration_impl(m, t, direction, model_point_ids, n_ids, target_points, n_tp, sigma2, step_length, C, alpha,
                                  nullptr, alpha_out);
}

extern "C" int32_t icp_std_icp_iteration_theta(icp_model m, icp_target t, int32_t direction, const int32_t *model_point_ids,
                                               int32_t n_ids, const double *target_points, int32_t n_tp, double sigma2,
                                               double step_length, int32_t C, const double *theta, double *alpha_out) {
    if (C > 0 && !theta) return ICP_ERR_INVALID_ARGUMENT;
    return std_icp_iteration_impl(m, t, direction, model_point_ids, n_ids, target_points, n_tp, sigma2, step_length, C, nullptr,
                                  theta, alpha_out);
}

// alpha != null: identity pose (IcpRegistration passes the rigid identity); theta != null: currentTrans from theta
static int32_t std_icp_iteration_impl(icp_model m, icp_target t, int32_t direction, const int32_t *model_point_ids,
                                      int32_t n_ids, const double *target_points, int32_t n_tp, double sigma2,
                                      double step_length, int32_t C, const double *alpha, const double *theta, double *alpha_out) {
    ICP_API_BEGIN(m ? m->ctx : nullptr)
    ICP_REQUIRE(t && t->ctx == m->ctx, "bad target");
    ICP_REQUIRE(direction == ICP_MODEL_SAMPLING || direction == ICP_TARGET_SAMPLING, "bad direction");
    ICP_REQUIRE(sigma2 > 0, "sigma2 must be > 0");
    if (C == 0) return ICP_OK;
    ICP_REQUIRE((alpha || theta) && alpha_out, "null array");
    check_ids(m->N, model_point_ids, n_ids);
    cudaStream_t s = _ctx->stream;
    const int K = m->K, Kp = m->Kp, Lt = K + kTheta0;
    // identity pose: theta = [1, 0.., alpha]; otherwise the caller's rigid transform (model.transform(currentTrans), :61)
    std::vector<double> th((size_t)C * Lt, 0.0), al((size_t)C * K);
    for (int c = 0; c < C; c++) {
        if (theta) {
            memcpy(&th[(size_t)c * Lt], theta + (size_t)c * Lt, sizeof(double) * Lt);
            memcpy(&al[(size_t)c * K], theta + (size_t)c * Lt + kTheta0, sizeof(double) * K);
        } else {
            th[(size_t)c * Lt] = 1.0;
            memcpy(&th[(size_t)c * Lt + kTheta0], alpha + (size_t)c * K, sizeof(double) * K);
            memcpy(&al[(size_t)c * K], alpha + (size_t)c * K, sizeof(double) * K);
        }
    }
    icp_proposal_s tmp;
    tmp.model = m; tmp.target = t;
    tmp.prm.step_length = step_length; tmp.prm.tangential_noise = 1; tmp.prm.noise_along_normal = 1;
    tmp.prm.direction = direction; tmp.prm.boundary_aware = 0; tmp.prm.factor = ICP_FACTOR_CHOLESKY; tmp.prm.rank_update = ICP_RANK_UPDATE_FP64;
    tmp.n_ids = n_ids; tmp.n_tp = n_tp;
    tmp.ids.upload(model_point_ids, n_ids, s);
    tmp.tp.upload(target_points, (size_t)3 * n_tp, s);
    DevBuf<double> dth, dL, dmu, da, dout;
    dth.upload(th.data(), th.size(), s);
    dL.alloc((size_t)C * Kp * Kp); dmu.alloc((size_t)C * Kp);
    da.upload(al.data(), (size_t)C * K, s); dout.alloc((size_t)C * K);
    // run the pipeline with isotropic noise: patch ObsArgs through a local copy of the pipeline
    {
        icp_proposal p = &tmp;
        PosteriorWork &w = tmp.work;
        ModelDev md = m->dev();
        w.X.ensure((size_t)C * m->N * 3);
        launch_reconstruct(md, C, dth.p, w.X.p, s);
        const bool tsamp = direction == ICP_TARGET_SAMPLING;
        int n = tsamp ? n_tp : n_ids;
        size_t tot = (size_t)C * std::max(n, 1);
        w.vid.ensure(tot); w.F.ensure(9 * tot); w.y.ensure(3 * tot); w.nobs.ensure(C);
        w.M.ensure((size_t)C * Kp * Kp); w.b.ensure((size_t)C * Kp); w.status.ensure(C);
        ObsArgs oa{};
        oa.m = md; oa.prm = p->prm; oa.C = C; oa.theta = dth.p; oa.X = w.X.p; oa.iso = 1; oa.iso_sigma2 = sigma2;
        oa.world_frame = 1;   // :81 model.posterior(corr, sigma) on the untransformed model, targets as they are
        if (tsamp) {
            w.prim.ensure(tot);
            nearest_model_vertex(m, C, w.X.p, n, tmp.tp.p, 0, nullptr, w.prim.p, s);
            oa.tp = tmp.tp.p; oa.near_vid = w.prim.p;
        } else {
            w.cp.ensure(3 * tot);
            NearestArgs a;
            a.bvh = &t->tri_bvh; a.prim_data = t->tri_data.p; a.wide = t->wide(); a.sm_count = t->ctx->sm_count; a.C = C; a.nq = n;
            a.Xq = w.X.p; a.q_ids = tmp.ids.p; a.Nq = m->N; a.out_cp = w.cp.p;
            launch_nearest(a, s);
            oa.ids = tmp.ids.p; oa.cp = w.cp.p; oa.cp_stride = n; oa.cp_map = nullptr;
        }
        ObsDev od{n, w.vid.p, w.F.p, w.y.p, w.nobs.p};
        launch_observations(oa, od, s);
        launch_posterior_build(md, C, od, w.M.p, w.b.p, s);
        w.Mp.ensure((size_t)C * (Kp / 8) * (Kp / 8 + 1) / 2 * 64);
        launch_cholesky_solve(C, K, Kp, w.M.p, w.b.p, dL.p, dmu.p, nullptr, w.status.p, s, w.Mp.p);
    }
    k_std_icp_step<<<C, 128, 0, s>>>(C, K, Kp, step_length, m->S.p, dmu.p, da.p, dout.p);
    ICP_CUDA(cudaGetLastError());
    download(alpha_out, dout.p, (size_t)C * K, s);
    sync_stream(_ctx);
    ICP_API_END
}

// ---------------------------------------------------------------------------------------------------
// (6) evaluators
// ---------------------------------------------------------------------------------------------------
extern "C" int32_t icp_evaluator_create(icp_model m, icp_target t, const icp_evaluator_params *params,
                                        const int32_t *model_point_ids, int32_t n_ids, const double *target_points,
                                        int32_t n_tp, icp_evaluator *out) {
    icp_evaluator e = nullptr;
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(m && t && params && out, "null argument");
        ICP_REQUIRE(m->ctx == t->ctx, "model and target belong to different contexts");
        CtxLock lock(_ctx);
        ICP_REQUIRE(params->kind >= ICP_EVAL_ACCEPT_ALL && params->kind <= ICP_EVAL_COLLECTIVE, "bad evaluator kind");
        ICP_REQUIRE(params->mode >= ICP_MODEL_TO_TARGET && params->mode <= ICP_SYMMETRIC, "bad evaluation mode");
        cudaStream_t s = _ctx->stream;
        e = new icp_evaluator_s();
        e->model = m; e->target = t; e->prm = *params;
        if (params->kind == ICP_EVAL_HAUSDORFF) {
            // MeshMetrics.hausdorffDistance: every vertex of both meshes
            std::vector<int> all(m->N);
            for (int i = 0; i < m->N; i++) all[i] = i;
            e->n_ids = m->N; e->ids.upload(all.data(), all.size(), s);
            { std::vector<int> pm = morton_perm(m->h_ref, all.data(), m->N); e->qperm.upload(pm.data(), pm.size(), s); sync_stream(_ctx); }
            e->n_tp = t->Nt; e->tp.alloc((size_t)3 * t->Nt);
            ICP_CUDA(cudaMemcpyAsync(e->tp.p, t->verts.p, sizeof(double) * 3 * t->Nt, cudaMemcpyDeviceToDevice, s));
            ICP_REQUIRE(params->p0 > 0, "Exponential rate must be > 0");
        } else {
            check_ids(m->N, model_point_ids, n_ids);
            ICP_REQUIRE(n_tp >= 0 && (n_tp == 0 || target_points != nullptr), "bad target point list");
            e->n_ids = n_ids; e->ids.upload(model_point_ids, n_ids, s);
            if (n_ids > 0) { std::vector<int> pm = morton_perm(m->h_ref, model_point_ids, n_ids); e->qperm.upload(pm.data(), pm.size(), s); sync_stream(_ctx); }
            e->n_tp = n_tp; e->tp.upload(target_points, (size_t)3 * n_tp, s);
            if (params->kind != ICP_EVAL_ACCEPT_ALL) ICP_REQUIRE(params->p1 > 0, "Gaussian std-dev must be > 0");
            if (params->kind == ICP_EVAL_COLLECTIVE) ICP_REQUIRE(params->p2 > 0, "Exponential rate must be > 0");
        }
        sync_stream(_ctx);
        m->refs++; t->refs++;
        *out = e;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete e;
        return rc;
    }
}

extern "C" int32_t icp_evaluator_destroy(icp_evaluator e) {
    if (!e) return ICP_OK;
    icp_ctx _ctx = e->model->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_REQUIRE(e->refs == 0, "evaluator is still used by a chain: destroy the chain first");
        drain_calls(e);
        sync_stream(_ctx);
        e->model->refs--; e->target->refs--;
        delete e;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

namespace icp {

void evaluator_pipeline(icp_evaluator e, EvalWork &w, int C, const double *d_theta, const double *d_X, double *d_values,
                        int *d_status, cudaStream_t s, const TargetSet *ts) {
    if (C <= 0) return;
    icp_model m = e->model;
    icp_target t = e->target;
    const bool has_boundary = ts ? ts->has_boundary : t->has_boundary;
    const TargetRec *mt_rec = ts ? ts->rec : nullptr;
    const int *mt_idx = ts ? ts->tidx : nullptr;
    // the target -> model lists: the evaluator's own, or every entry's copy of its target's list
    const int n_tp = ts ? ts->n_tp : e->n_tp;
    ModelDev md = m->dev();
    const int kind = e->prm.kind, mode = e->prm.mode;
    EvalReduceArgs ra{};
    ra.prm = e->prm; ra.C = C; ra.K = m->K; ra.theta = d_theta; ra.values = d_values; ra.status = d_status;
    if (kind != ICP_EVAL_ACCEPT_ALL) {
        if (!d_X) {
            w.X.ensure((size_t)C * m->N * 3);
            launch_reconstruct(md, C, d_theta, w.X.p, s);
            d_X = w.X.p;
        }
        const bool use_m = kind == ICP_EVAL_HAUSDORFF || mode != ICP_TARGET_TO_MODEL;
        const bool use_t = kind == ICP_EVAL_HAUSDORFF || mode != ICP_MODEL_TO_TARGET;
        const bool collective = kind == ICP_EVAL_COLLECTIVE;
        // Hausdorff: only the largest distance of the two directions is used, so both traversals share one running maximum
        // per chain and stop every query that cannot raise it (k_nearest, HDMAX). Not when the model -> target closest points
        // are shared with an ICP proposal (they must be exact then). ICPCUDA_HAUSDORFF_PRUNE=0 switches it off.
        static const bool hd_prune_on = !(getenv("ICPCUDA_HAUSDORFF_PRUNE") && getenv("ICPCUDA_HAUSDORFF_PRUNE")[0] == '0');
        unsigned long long *hd_max = nullptr;
        if (kind == ICP_EVAL_HAUSDORFF && hd_prune_on && !w.force_cp_m2t) {
            w.hd_max.ensure(C);
            ICP_CUDA(cudaMemsetAsync(w.hd_max.p, 0, sizeof(unsigned long long) * (size_t)C, s));
            hd_max = w.hd_max.p;
        }
        if (use_m && e->n_ids > 0) {
            size_t tot = (size_t)C * e->n_ids;
            w.d2_m2t.ensure(tot);
            NearestArgs a;
            a.bvh = &t->tri_bvh; a.prim_data = t->tri_data.p; a.wide = t->wide(); a.sm_count = t->ctx->sm_count; a.C = C; a.nq = e->n_ids;
            a.Xq = d_X; a.q_ids = e->ids.p; a.Nq = m->N; a.out_d2 = w.d2_m2t.p; a.perm = e->qperm.p;
            a.mt_rec = mt_rec; a.mt_idx = mt_idx;
            if (w.seed_m2t.n < tot) { w.seed_m2t.ensure(tot); ICP_CUDA(cudaMemsetAsync(w.seed_m2t.p, 0xFF, sizeof(int) * tot, s)); }
            a.seed_slot = w.seed_m2t.p;
            if (collective || w.force_cp_m2t) { w.cp_m2t.ensure(3 * tot); a.out_cp = w.cp_m2t.p; }
            a.chain_max = hd_max;
            launch_nearest(a, s);
            if (collective && has_boundary) {
                // CollectiveAverage...:46-47: nearest target vertex of the closest point, dropped when on the boundary
                w.prim.ensure(tot); w.skip_m2t.ensure(tot);
                NearestArgs v;
                v.bvh = &t->vert_bvh; v.prim_data = t->vert_data.p; v.C = C; v.nq = e->n_ids; v.q = w.cp_m2t.p;
                v.q_per_chain = 1; v.out_prim = w.prim.p;
                v.mt_rec = mt_rec; v.mt_idx = mt_idx;
                launch_nearest(v, s);
                launch_lookup_flags((int64_t)tot, w.prim.p, t->boundary.p, t->Nt, w.skip_m2t.p, s, mt_rec, mt_idx, e->n_ids);
                ra.skip_m2t = w.skip_m2t.p;
            }
        }
        if (use_t && n_tp > 0) {
            size_t tot = (size_t)C * n_tp;
            w.d2_t2m.ensure(tot);
            bvh_refit(m->tri_bvh, C, d_X, m->N, m->tris.p, s);
            NearestArgs a;
            a.bvh = &m->tri_bvh; a.X = d_X; a.tris = m->tris.p; a.N = m->N; a.C = C; a.nq = n_tp;
            a.q = ts ? ts->tp : e->tp.p; a.q_per_chain = ts ? 1 : 0;
            a.out_d2 = w.d2_t2m.p;
            if (w.seed_t2m.n < tot) { w.seed_t2m.ensure(tot); ICP_CUDA(cudaMemsetAsync(w.seed_t2m.p, 0xFF, sizeof(int) * tot, s)); }
            a.seed_slot = w.seed_t2m.p;
            if (collective) { w.cp_t2m.ensure(3 * tot); a.out_cp = w.cp_t2m.p; }
            a.chain_max = hd_max;
            launch_nearest(a, s);
            if (collective && has_boundary) {
                // CollectiveAverage...:58-59: id of the nearest vertex of the MODEL sample, looked up in the
                // TARGET's boundary table (SURVEY Appendix B3)
                w.prim.ensure(tot); w.skip_t2m.ensure(tot);
                nearest_model_vertex(m, C, d_X, n_tp, w.cp_t2m.p, 1, nullptr, w.prim.p, s);
                launch_lookup_flags((int64_t)tot, w.prim.p, t->boundary.p, t->Nt, w.skip_t2m.p, s, mt_rec, mt_idx, n_tp);
                ra.skip_t2m = w.skip_t2m.p;
            }
        }
        ra.n_m2t = use_m ? e->n_ids : 0; ra.d2_m2t = w.d2_m2t.p;
        ra.n_t2m = use_t ? n_tp : 0; ra.d2_t2m = w.d2_t2m.p;
    }
    launch_eval_reduce(ra, s);
}

}  // namespace icp

extern "C" int32_t icp_eval_log_value(icp_evaluator e, int32_t C, const double *theta, double *values, int32_t *status) {
    const bool self_contained = e && evaluator_self_contained(e);
    ICP_API_BEGIN_HANDLE(icp_evaluator_s, e, self_contained)
    if (C == 0) return ICP_OK;
    ICP_REQUIRE(C > 0 && theta != nullptr, "bad theta array");
    ICP_REQUIRE(values != nullptr, "values is null");
    const bool graph = self_contained && call_graphs_enabled();
    const size_t nth = (size_t)C * (e->model->K + kTheta0);
    cs.h_in.ensure(sizeof(double) * nth);
    cs.h_out.ensure(sizeof(double) * 3 * (size_t)C + sizeof(int) * (size_t)C);
    double *hval = reinterpret_cast<double *>(cs.h_out.p);
    int *hst = reinterpret_cast<int *>(hval + 3 * (size_t)C);
    memcpy(cs.h_in.p, theta, sizeof(double) * nth);
    cs.s_theta.ensure(nth);
    cs.s_values.ensure((size_t)3 * C);
    cs.s_status.ensure(C);
    run_call_graph(cs, graph, call_key(CALL_EVAL, C), evaluator_call_ptrs(cs), s, [&] {
        h2d(cs.s_theta.p, cs.h_in.p, sizeof(double) * nth, s);
        evaluator_pipeline(e, cs.work, C, cs.s_theta.p, nullptr, cs.s_values.p, cs.s_status.p, s);
        d2h(hval, cs.s_values.p, sizeof(double) * 3 * (size_t)C, s);
        d2h(hst, cs.s_status.p, sizeof(int) * (size_t)C, s);
    });
    ICP_CUDA(cudaStreamSynchronize(s));
    memcpy(values, hval, sizeof(double) * 3 * (size_t)C);
    if (status) memcpy(status, hst, sizeof(int) * (size_t)C);
    ICP_API_END
}

extern "C" int32_t icp_eval_prior(icp_model m, int32_t C, const double *theta, double *out) {
    ICP_API_BEGIN(m ? m->ctx : nullptr)
    if (C == 0) return ICP_OK;
    ICP_REQUIRE(out != nullptr, "out is null");
    cudaStream_t s = _ctx->stream;
    upload_theta(m, C, theta, m->s_theta, s);
    m->s_d.ensure(C);
    launch_prior(C, m->K, m->s_theta.p, m->s_d.p, s);
    download(out, m->s_d.p, C, s);
    sync_stream(_ctx);
    ICP_API_END
}

