// comm.cu - multi-GPU entry points of the C ABI and the posterior variability maps they reduce.
//
// Chains, random-init restarts and targets are independent (RunMHRandomInitComparison.scala:66-86,
// StdIcpVsChainICPrandomInitComparisonAll.scala:107-122), so a sharded run needs no collective on the per-sample path.
// What remains is the end-of-run exchange BASELINE.json names: the gather of the chain logs and the reduction of the
// posterior statistics (apps/util/PosteriorVariability.scala:30-73 over LogHelper.logSamples2shapes). Both go through
// NCCL directly (no torch, no MPI): the library dlopens libnccl.so.2 on the first icp_comm_* call, so a single-GPU host
// needs no NCCL at all, and it fails loudly when a multi-GPU call cannot find it.
#include <dlfcn.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "icp_device.cuh"
#include "icp_internal.h"

using namespace icp;

// ---- the handful of NCCL entry points used here (ABI of NCCL 2.x; nccl.h is not needed to build) -----------------------
namespace {
typedef void *nccl_comm_t;
struct nccl_uid { char internal[128]; };
enum { kNcclUint8 = 1, kNcclInt32 = 2, kNcclInt64 = 4, kNcclFloat64 = 8, kNcclSum = 0 };
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(nccl_uid *) = nullptr;
    int (*CommInitRank)(nccl_comm_t *, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    int (*GetVersion)(int *) = nullptr;
};
NcclApi g_nccl;
std::mutex g_nccl_mu;

const NcclApi &nccl() {
    std::lock_guard<std::mutex> lk(g_nccl_mu);
    if (g_nccl.h) return g_nccl;
    const char *env = getenv("ICPCUDA_NCCL_LIB");
    const char *cands[] = {env, "libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *c : cands) {
        if (!c || !c[0]) continue;
        h = dlopen(c, RTLD_NOW | RTLD_LOCAL);
        if (h) break;
    }
    if (!h) throw StatusError{ICP_ERR_CUDA, "NCCL not found: the multi-GPU entry points need libnccl.so.2 (set ICPCUDA_NCCL_LIB)"};
    NcclApi a;
    a.h = h;
#define ICP_NCCL_SYM(field, name)                                   \
    *(void **)(&a.field) = dlsym(h, name);                          \
    if (!a.field) throw StatusError{ICP_ERR_CUDA, std::string("NCCL symbol missing: ") + name};
    ICP_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    ICP_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    ICP_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    ICP_NCCL_SYM(AllGather, "ncclAllGather")
    ICP_NCCL_SYM(AllReduce, "ncclAllReduce")
    ICP_NCCL_SYM(GroupStart, "ncclGroupStart")
    ICP_NCCL_SYM(GroupEnd, "ncclGroupEnd")
    ICP_NCCL_SYM(GetErrorString, "ncclGetErrorString")
    ICP_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef ICP_NCCL_SYM
    g_nccl = a;
    return g_nccl;
}

void nccl_check(int rc, const char *what) {
    if (rc != 0) throw StatusError{ICP_ERR_CUDA, std::string("NCCL error in ") + what + ": " + nccl().GetErrorString(rc)};
}
}  // namespace

struct icp_comm_s {
    icp_ctx ctx = nullptr;
    int rank = 0, world = 1;
    nccl_comm_t comm = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

extern "C" int32_t icp_comm_unique_id(icp_ctx ctx, uint8_t id[ICP_COMM_UNIQUE_ID_BYTES]) {
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx && id, "null argument");
        CtxLock lock(ctx);
        static_assert(ICP_COMM_UNIQUE_ID_BYTES == sizeof(nccl_uid), "unique id size");
        nccl_uid u;
        nccl_check(nccl().GetUniqueId(&u), "ncclGetUniqueId");
        memcpy(id, &u, sizeof u);
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_comm_init(icp_ctx ctx, int32_t rank, int32_t world, const uint8_t id[ICP_COMM_UNIQUE_ID_BYTES],
                                 icp_comm *out) {
    icp_ctx _ctx = ctx;
    icp_comm c = nullptr;
    try {
        ICP_REQUIRE(ctx && id && out, "null argument");
        ICP_REQUIRE(world >= 1 && rank >= 0 && rank < world, "rank must be in [0, world)");
        CtxLock lock(ctx);
        c = new icp_comm_s();
        c->ctx = ctx; c->rank = rank; c->world = world;
        nccl_uid u;
        memcpy(&u, id, sizeof u);
        nccl_check(nccl().CommInitRank(&c->comm, world, u, rank), "ncclCommInitRank");
        ICP_CUDA(cudaEventCreate(&c->e0));
        ICP_CUDA(cudaEventCreate(&c->e1));
        *out = c;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete c;
        return rc;
    }
}

extern "C" int32_t icp_comm_destroy(icp_comm c) {
    if (!c) return ICP_OK;
    icp_ctx _ctx = c->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_CUDA(cudaStreamSynchronize(_ctx->stream));
        if (c->comm) nccl().CommDestroy(c->comm);
        if (c->e0) cudaEventDestroy(c->e0);
        if (c->e1) cudaEventDestroy(c->e1);
        delete c;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_comm_info(icp_comm c, int32_t *rank, int32_t *world, int32_t *nccl_version) {
    if (!c) return ICP_ERR_INVALID_ARGUMENT;
    if (rank) *rank = c->rank;
    if (world) *world = c->world;
    if (nccl_version) { int v = 0; nccl().GetVersion(&v); *nccl_version = v; }
    return ICP_OK;
}

// All-gather of the chain logs of a sharded run (JSONAcceptRejectLogger records of every chain on every rank).
extern "C" int32_t icp_chainlog_gather(icp_comm c, int32_t n_steps, int32_t C, int32_t K, const icp_chain_io *local_dev,
                                       const icp_chain_io *gathered_dev, double *device_ms, int64_t *bytes_received) {
    icp_ctx _ctx = c ? c->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        ICP_REQUIRE(local_dev && gathered_dev && n_steps >= 0 && C >= 1 && K >= 1, "bad arguments");
        CtxLock lock(_ctx);
        cudaStream_t s = _ctx->stream;
        const NcclApi &nc = nccl();
        const size_t rec = (size_t)n_steps * C, Lt = (size_t)K + kTheta0;
        int64_t bytes = 0;
        ICP_CUDA(cudaEventRecord(c->e0, s));
        nccl_check(nc.GroupStart(), "ncclGroupStart");
        auto gather = [&](const void *src, void *dst, size_t count, int dtype, size_t elem) {
            if (!src && !dst) return;
            ICP_REQUIRE(src && dst, "a log array must be given on both sides (local and gathered) or on neither");
            if (count == 0) return;
            nccl_check(nc.AllGather(src, dst, count, dtype, c->comm, s), "ncclAllGather");
            bytes += (int64_t)(count * elem) * c->world;
        };
        gather(local_dev->log_component, gathered_dev->log_component, rec, kNcclInt32, 4);
        gather(local_dev->log_accepted, gathered_dev->log_accepted, rec, kNcclUint8, 1);
        gather(local_dev->log_values, gathered_dev->log_values, rec * 3, kNcclFloat64, 8);
        gather(local_dev->log_theta, gathered_dev->log_theta, rec * Lt, kNcclFloat64, 8);
        gather(local_dev->theta_final, gathered_dev->theta_final, (size_t)C * Lt, kNcclFloat64, 8);
        gather(local_dev->n_accepted, gathered_dev->n_accepted, (size_t)C, kNcclInt64, 8);
        gather(local_dev->status, gathered_dev->status, (size_t)C, kNcclInt32, 4);
        gather(local_dev->theta_best, gathered_dev->theta_best, (size_t)C * Lt, kNcclFloat64, 8);
        gather(local_dev->value_best, gathered_dev->value_best, (size_t)C, kNcclFloat64, 8);
        nccl_check(nc.GroupEnd(), "ncclGroupEnd");
        ICP_CUDA(cudaEventRecord(c->e1, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        float ms = 0;
        ICP_CUDA(cudaEventElapsedTime(&ms, c->e0, c->e1));
        if (device_ms) *device_ms = ms;
        if (bytes_received) *bytes_received = bytes;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

static void comm_allreduce_sum_f64(icp_comm c, double *buf, size_t n, cudaStream_t s);
static void comm_allreduce_sum_i64(icp_comm c, long long *buf, size_t n, cudaStream_t s);

// ---------------------------------------------------------------------------------------------------
// Posterior variability maps from chain samples (apps/util/PosteriorVariability.scala:30-73 over the shapes of
// apps/util/LogHelper.scala:39-41): S parameter vectors -> batched reconstruction (+ vertex normals) -> per-vertex
// mean, sample covariance (divisor S - 1), its trace, and the variance along a direction n (the reference mesh's
// vertex normal, or the un-normalised mean of the samples' unit vertex normals when sum_normals != 0).
// Two passes like the reference (mean first, then centred moments). Thread / vertex so that a warp reads 768
// contiguous bytes of one sample; the samples are split over gridDim.y partitions whose partial sums are combined in
// partition order (deterministic).
// ---------------------------------------------------------------------------------------------------
constexpr int kVarThreads = 128;

__global__ void __launch_bounds__(kVarThreads) k_var_sums(int S, int N, const double *__restrict__ X,
                                                          const double *__restrict__ Nrm, double *__restrict__ part) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    const int P = gridDim.y, p = blockIdx.y;
    const int s0 = (int)((long long)S * p / P), s1 = (int)((long long)S * (p + 1) / P);
    double a[6] = {0, 0, 0, 0, 0, 0};
    for (int s = s0; s < s1; s++) {
        const double *x = X + ((size_t)s * N + v) * 3;
        a[0] += x[0]; a[1] += x[1]; a[2] += x[2];
        if (Nrm) {
            const double *n = Nrm + ((size_t)s * N + v) * 3;
            a[3] += n[0]; a[4] += n[1]; a[5] += n[2];
        }
    }
    double *o = part + ((size_t)p * N + v) * 6;
#pragma unroll
    for (int k = 0; k < 6; k++) o[k] = a[k];
}

// mean[v] = sum / S; dir[v] = mean unit normal (sum_normals) or the given reference normal
__global__ void k_var_means(int S, int N, int P, const double *__restrict__ part, const double *__restrict__ ref_normals,
                            double *__restrict__ mean, double *__restrict__ dir) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    double a[6] = {0, 0, 0, 0, 0, 0};
    for (int p = 0; p < P; p++)
#pragma unroll
        for (int k = 0; k < 6; k++) a[k] += part[((size_t)p * N + v) * 6 + k];
    const double inv = 1.0 / S;
#pragma unroll
    for (int k = 0; k < 3; k++) mean[3 * v + k] = a[k] * inv;
#pragma unroll
    for (int k = 0; k < 3; k++) dir[3 * v + k] = ref_normals ? ref_normals[3 * v + k] : a[3 + k] * inv;
}

__global__ void __launch_bounds__(kVarThreads) k_var_moments(int S, int N, const double *__restrict__ X,
                                                             const double *__restrict__ mean, const double *__restrict__ dir,
                                                             double *__restrict__ part) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    const int P = gridDim.y, p = blockIdx.y;
    const int s0 = (int)((long long)S * p / P), s1 = (int)((long long)S * (p + 1) / P);
    const double mx = mean[3 * v], my = mean[3 * v + 1], mz = mean[3 * v + 2];
    const double nx = dir[3 * v], ny = dir[3 * v + 1], nz = dir[3 * v + 2];
    double a[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int s = s0; s < s1; s++) {
        const double *x = X + ((size_t)s * N + v) * 3;
        const double dx = x[0] - mx, dy = x[1] - my, dz = x[2] - mz;
        a[0] += dx * dx; a[1] += dy * dy; a[2] += dz * dz;
        a[3] += dx * dy; a[4] += dx * dz; a[5] += dy * dz;
        const double t = nx * dx + ny * dy + nz * dz;
        a[6] += t * t;
    }
    double *o = part + ((size_t)p * N + v) * 7;
#pragma unroll
    for (int k = 0; k < 7; k++) o[k] = a[k];
}

__global__ void k_var_finish(int S, int N, int P, const double *__restrict__ part, double *__restrict__ cov,
                             double *__restrict__ total, double *__restrict__ along) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    double a[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int p = 0; p < P; p++)
#pragma unroll
        for (int k = 0; k < 7; k++) a[k] += part[((size_t)p * N + v) * 7 + k];
    const double inv = 1.0 / (double)(S - 1);   // S == 1: 0 * inf = NaN, as the reference's 0.0 * (1.0 / 0)
#pragma unroll
    for (int k = 0; k < 7; k++) a[k] *= inv;
    double *c = cov + 9 * (size_t)v;
    c[0] = a[0]; c[4] = a[1]; c[8] = a[2];
    c[1] = c[3] = a[3]; c[2] = c[6] = a[4]; c[5] = c[7] = a[5];
    total[v] = a[0] + a[1] + a[2];
    along[v] = a[6];
}

// the finish of the maps the chain runner accumulates (icp_chain_statistics, stats.cu)
void icp::launch_var_finish(int S, int N, const double *d_tot7, double *d_cov, double *d_total, double *d_along, cudaStream_t s) {
    k_var_finish<<<(N + kVarThreads - 1) / kVarThreads, kVarThreads, 0, s>>>(S, N, 1, d_tot7, d_cov, d_total, d_along);
    ICP_CUDA(cudaGetLastError());
}


// per-vertex totals over the partitions (deterministic partition order): tot[v][W] = sum_p part[p][v][W]
template <int W>
__global__ void k_var_collapse(int N, int P, const double *__restrict__ part, double *__restrict__ tot) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    double a[W];
#pragma unroll
    for (int k = 0; k < W; k++) a[k] = 0.0;
    for (int p = 0; p < P; p++)
#pragma unroll
        for (int k = 0; k < W; k++) a[k] += part[((size_t)p * N + v) * W + k];
#pragma unroll
    for (int k = 0; k < W; k++) tot[(size_t)v * W + k] = a[k];
}

// S_local samples of this rank; with a communicator the sums are all-reduced, so every rank ends with the maps over the
// samples of ALL ranks (two passes like the reference: global mean first, then moments centred on it - no cancellation)
static void variability_impl(icp_model m, icp_comm comm, int S_local, const double *theta, int sum_normals, const double *theta_ref,
                             double *mean, double *cov, double *total_variance, double *normal_variance, int64_t *S_total_out) {
    icp_ctx ctx = m->ctx;
    cudaStream_t s = ctx->stream;
    const int N = m->N;
    const size_t n3 = (size_t)N * 3;
    DevBuf<double> X, Nrm, refX, refN, part, tot, d_mean, d_dir, d_cov, d_total, d_along;
    DevBuf<long long> d_cnt;
    const int Sl = std::max(S_local, 0);
    if (Sl > 0) {
        m->s_theta.upload(theta, (size_t)Sl * (m->K + kTheta0), s);
        X.alloc((size_t)Sl * n3);
        launch_reconstruct(m->dev(), Sl, m->s_theta.p, X.p, s);
    }
    const double *ref_normals = nullptr;
    if (sum_normals) {
        if (Sl > 0) { Nrm.alloc((size_t)Sl * n3); launch_vertex_normals(m->dev(), Sl, X.p, Nrm.p, s); }
    } else {
        // normals of `ref`: transformedMesh(theta_ref), or the model's reference mesh when theta_ref is NULL
        refN.alloc(n3);
        const double *rx = m->ref.p;
        DevBuf<double> th;
        if (theta_ref) {
            th.upload(theta_ref, (size_t)(m->K + kTheta0), s);
            refX.alloc(n3);
            launch_reconstruct(m->dev(), 1, th.p, refX.p, s);
            rx = refX.p;
            ICP_CUDA(cudaStreamSynchronize(s));   // th leaves scope
        }
        launch_vertex_normals(m->dev(), 1, rx, refN.p, s);
        ref_normals = refN.p;
    }
    const int vb = (N + kVarThreads - 1) / kVarThreads;
    int P = (4 * 148 + vb - 1) / vb;   // about four waves of CTAs
    if (P > Sl) P = Sl;
    if (P < 1) P = 1;
    part.alloc((size_t)P * N * 7);
    tot.alloc((size_t)N * 7);
    d_mean.alloc(n3); d_dir.alloc(n3); d_cov.alloc((size_t)N * 9); d_total.alloc(N); d_along.alloc(N);
    long long S = Sl;
    // pass 1: sums of positions (and unit normals)
    if (Sl > 0) {
        k_var_sums<<<dim3(vb, P), kVarThreads, 0, s>>>(Sl, N, X.p, sum_normals ? Nrm.p : nullptr, part.p);
        ICP_CUDA(cudaGetLastError());
        k_var_collapse<6><<<vb, kVarThreads, 0, s>>>(N, P, part.p, tot.p);
    } else {
        ICP_CUDA(cudaMemsetAsync(tot.p, 0, sizeof(double) * (size_t)N * 7, s));
    }
    ICP_CUDA(cudaGetLastError());
    if (comm) {
        d_cnt.alloc(1);
        ICP_CUDA(cudaMemcpyAsync(d_cnt.p, &S, sizeof S, cudaMemcpyHostToDevice, s));
        comm_allreduce_sum_f64(comm, tot.p, (size_t)N * 6, s);
        comm_allreduce_sum_i64(comm, d_cnt.p, 1, s);
        ICP_CUDA(cudaMemcpyAsync(&S, d_cnt.p, sizeof S, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
    }
    ICP_REQUIRE(S >= 1, "posterior variability needs at least one sample");
    k_var_means<<<vb, kVarThreads, 0, s>>>((int)S, N, 1, tot.p, ref_normals, d_mean.p, d_dir.p);
    ICP_CUDA(cudaGetLastError());
    // pass 2: moments centred on the (global) mean
    if (Sl > 0) {
        k_var_moments<<<dim3(vb, P), kVarThreads, 0, s>>>(Sl, N, X.p, d_mean.p, d_dir.p, part.p);
        ICP_CUDA(cudaGetLastError());
        k_var_collapse<7><<<vb, kVarThreads, 0, s>>>(N, P, part.p, tot.p);
    } else {
        ICP_CUDA(cudaMemsetAsync(tot.p, 0, sizeof(double) * (size_t)N * 7, s));
    }
    ICP_CUDA(cudaGetLastError());
    if (comm) comm_allreduce_sum_f64(comm, tot.p, (size_t)N * 7, s);
    k_var_finish<<<vb, kVarThreads, 0, s>>>((int)S, N, 1, tot.p, d_cov.p, d_total.p, d_along.p);
    ICP_CUDA(cudaGetLastError());
    auto dl = [&](double *h, const double *d, size_t n) {
        if (h) ICP_CUDA(cudaMemcpyAsync(h, d, n * sizeof(double), cudaMemcpyDeviceToHost, s));
    };
    dl(mean, d_mean.p, n3); dl(cov, d_cov.p, (size_t)N * 9); dl(total_variance, d_total.p, N); dl(normal_variance, d_along.p, N);
    ICP_CUDA(cudaStreamSynchronize(s));
    if (S_total_out) *S_total_out = S;
}

static void comm_allreduce_sum_f64(icp_comm c, double *buf, size_t n, cudaStream_t s) {
    nccl_check(nccl().AllReduce(buf, buf, n, kNcclFloat64, kNcclSum, c->comm, s), "ncclAllReduce");
}
static void comm_allreduce_sum_i64(icp_comm c, long long *buf, size_t n, cudaStream_t s) {
    nccl_check(nccl().AllReduce(buf, buf, n, kNcclInt64, kNcclSum, c->comm, s), "ncclAllReduce");
}

extern "C" int32_t icp_posterior_variability(icp_model m, int32_t S, const double *theta, int32_t sum_normals,
                                             const double *theta_ref, double *mean, double *cov, double *total_variance,
                                             double *normal_variance) {
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        CtxLock lock(_ctx);
        ICP_REQUIRE(S >= 1 && theta != nullptr, "posterior variability needs at least one sample");
        variability_impl(m, nullptr, S, theta, sum_normals, theta_ref, mean, cov, total_variance, normal_variance, nullptr);
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_variability_allreduce(icp_comm c, icp_model m, int32_t S_local, const double *theta_local,
                                             int32_t sum_normals, const double *theta_ref, double *mean, double *cov,
                                             double *total_variance, double *normal_variance, int64_t *S_total) {
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr && c != nullptr, "null handle");
        ICP_REQUIRE(c->ctx == _ctx, "communicator and model belong to different contexts");
        CtxLock lock(_ctx);
        ICP_REQUIRE(S_local >= 0 && (S_local == 0 || theta_local != nullptr), "bad sample array");
        variability_impl(m, c, S_local, theta_local, sum_normals, theta_ref, mean, cov, total_variance, normal_variance, S_total);
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}
