// stdicp.cu - IcpBasedSurfaceFitting.runfitting (api/other/IcpBasedSurfaceFitting.scala:46-126) for C independent fits as a
// device-resident loop: section (5b) of the C ABI.
//
// One iteration of a fit is  alpha' = alpha + (S^T mu - alpha) step,  mu = (I + G / sigma2)^-1 Q^T r / sigma2  with isotropic
// noise, no boundary filter and world-frame residuals r (what icp_std_icp_iteration computes per call).
//  - Model sampling: every fit observes the same model points, so G = G_s = sum_i Q_i^T Q_i is one constant matrix and
//    alpha' = alpha + (T_sigma Q_s^T r - alpha) step with the K x Kp projector T_sigma = S^T (sigma2 I + G_s)^-1, formed once per
//    sigma of a run. An iteration is then reconstruct + closest points + ONE DMMA kernel for all fits (k_si_project).
//  - Target sampling: the observations depend on the state; the rank update + Cholesky of the MH runner (fused / packed, or
//    the general pair above rank 104), then k_si_target_step.
// Each iteration sorts its fits into a model-sampling range and a target-sampling range (k_si_gather, k_si_scatter); the
// split is known on the host before the run (caller directions, or the Philox coin, a pure function of seed, fit, iteration),
// and one CUDA graph per (C, split, sigma) is captured and replayed.
// A handle may hold several targets (icp_std_icp_create_targets): every fit names its own, a model-sampling slot walks its
// target's BVH (the multi-target k_nearest) and a target-sampling slot reads its target's point list. G_s, the projectors
// and the graphs depend on the model and the model point ids only, so every fit equals its single-target run bit for bit.
#include <cmath>
#include <cstring>
#include <map>
#include <string>

#include "icp_device.cuh"

using namespace icp;

namespace {

constexpr int kSiFits = 8;       // fits per CTA of k_si_project: the N dimension of one DMMA tile
constexpr int kSiWarps = 8;

// device-resident descriptors of the current run: the iteration graphs hold the address of this record, not its contents,
// so a run with other log buffers or another iteration count replays the same graphs
struct RunIo {
    const int *perm;        // [iters][C] work slot -> fit, model-sampling fits first (ascending), then target-sampling
    double *log_alpha;      // [iters][C][K] (nullable)
    int *log_direction;     // [iters][C] (nullable)
};

__global__ void k_si_init(int C, int Lt, const double *__restrict__ theta0, double *__restrict__ theta, int *__restrict__ status,
                          int *__restrict__ done, int *__restrict__ iter) {
    const int c = blockIdx.x;
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    for (int e = threadIdx.x; e < Lt; e += blockDim.x) {
        const double v = theta0[(size_t)c * Lt + e];
        theta[(size_t)c * Lt + e] = v;
        if (!isfinite(v)) bad = 1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        status[c] = bad ? ICP_STD_ICP_NON_FINITE : 0;   // :94-104: the first iteration throws, theta0's coefficients are returned
        done[c] = 0;
        if (c == 0) *iter = 0;
    }
}

// work slot p <- fit perm[iter][p]: parameters (a stopped fit runs on the identity instance so that every query stays finite;
// its result is discarded), its closest-point traversal seeds and, on a target set (tidx != nullptr), its target
__global__ void k_si_gather(int C, int Lt, int nm, int n_ids, int n_tp, const int *__restrict__ iter, const RunIo *__restrict__ io,
                            const double *__restrict__ theta, const int *__restrict__ status, double *__restrict__ theta_w,
                            const int *__restrict__ seed_m, const int *__restrict__ seed_t, int *__restrict__ wseed_m,
                            int *__restrict__ wseed_t, const int *__restrict__ tidx, int *__restrict__ wtidx) {
    const int p = blockIdx.x, c = io->perm[(size_t)(*iter) * C + p];
    const bool stopped = status[c] != 0;
    if (tidx && threadIdx.x == 0) wtidx[p] = tidx[c];
    for (int e = threadIdx.x; e < Lt; e += blockDim.x)
        theta_w[(size_t)p * Lt + e] = stopped ? (e == 0 ? 1.0 : 0.0) : theta[(size_t)c * Lt + e];
    if (p < nm) for (int i = threadIdx.x; i < n_ids; i += blockDim.x) wseed_m[(size_t)p * n_ids + i] = seed_m[(size_t)c * n_ids + i];
    else for (int i = threadIdx.x; i < n_tp; i += blockDim.x) wseed_t[(size_t)(p - nm) * n_tp + i] = seed_t[(size_t)c * n_tp + i];
}

// fit perm[iter][p] <- work slot p: the new coefficients unless the fit stopped now or before, the log rows, the seeds
__global__ void k_si_scatter(int C, int K, int Lt, int nm, int n_ids, int n_tp, const int *__restrict__ iter, const RunIo *__restrict__ io,
                             const double *__restrict__ theta_w, const int *__restrict__ wstat, double *__restrict__ theta,
                             int *__restrict__ status, int *__restrict__ done, int *__restrict__ seed_m, int *__restrict__ seed_t,
                             const int *__restrict__ wseed_m, const int *__restrict__ wseed_t) {
    const int p = blockIdx.x, it = *iter, c = io->perm[(size_t)it * C + p];
    const int st = status[c], ws = wstat[p];
    const bool take = st == 0 && ws == 0;
    __syncthreads();   // every thread has read status[c] before thread 0 rewrites it
    double *a = theta + (size_t)c * Lt + kTheta0;
    const double *aw = theta_w + (size_t)p * Lt + kTheta0;
    double *row = io->log_alpha ? io->log_alpha + ((size_t)it * C + c) * K : nullptr;
    for (int j = threadIdx.x; j < K; j += blockDim.x) {
        const double v = take ? aw[j] : a[j];
        a[j] = v;
        if (row) row[j] = v;
    }
    if (threadIdx.x == 0) {
        if (take) done[c] += 1;
        else if (st == 0) status[c] = ws;
        if (io->log_direction) io->log_direction[(size_t)it * C + c] = p < nm ? ICP_MODEL_SAMPLING : ICP_TARGET_SAMPLING;
    }
    if (p < nm) for (int i = threadIdx.x; i < n_ids; i += blockDim.x) seed_m[(size_t)c * n_ids + i] = wseed_m[(size_t)p * n_ids + i];
    else for (int i = threadIdx.x; i < n_tp; i += blockDim.x) seed_t[(size_t)c * n_tp + i] = wseed_t[(size_t)(p - nm) * n_tp + i];
}

__global__ void k_si_next(int *iter) { *iter += 1; }

// M = sigma2 I + G_s (padding rows / columns of G_s are zero: sigma2 on the padded diagonal)
__global__ void k_si_shift(int Kp, double sigma2, const double *__restrict__ G, double *__restrict__ M, double *__restrict__ b) {
    const int i = blockIdx.x;
    for (int j = threadIdx.x; j < Kp; j += blockDim.x) M[(size_t)i * Kp + j] = G[(size_t)i * Kp + j] + (i == j ? sigma2 : 0.0);
    if (threadIdx.x == 0) b[i] = 0.0;
}

// warp-wide sum, result in every lane
__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// row j of T = S^T M^-1 (M = L L^T symmetric): T_j = M^-1 s with s = column j of S, by a forward and a back substitution with the
// factor (one warp per row, rows j >= K zero)
__global__ void __launch_bounds__(32) k_si_projector(int K, int Kp, const double *__restrict__ L, const double *__restrict__ S,
                                                    double *__restrict__ T) {
    extern __shared__ double x[];
    const int j = blockIdx.x, lane = threadIdx.x;
    double *Tj = T + (size_t)j * Kp;
    if (j >= K) {
        for (int k = lane; k < Kp; k += 32) Tj[k] = 0.0;
        return;
    }
    for (int k = lane; k < Kp; k += 32) x[k] = S[(size_t)k * Kp + j];
    __syncwarp();
    for (int i = 0; i < Kp; i++) {            // L y = s
        double acc = 0.0;
        for (int k = lane; k < i; k += 32) acc = fma(L[(size_t)i * Kp + k], x[k], acc);
        acc = warp_sum(acc);
        __syncwarp();
        if (lane == 0) x[i] = (x[i] - acc) / L[(size_t)i * Kp + i];
        __syncwarp();
    }
    for (int i = Kp - 1; i >= 0; i--) {       // L^T x = y
        double acc = 0.0;
        for (int k = i + 1 + lane; k < Kp; k += 32) acc = fma(L[(size_t)k * Kp + i], x[k], acc);
        acc = warp_sum(acc);
        __syncwarp();
        if (lane == 0) x[i] = (x[i] - acc) / L[(size_t)i * Kp + i];
        __syncwarp();
    }
    for (int k = lane; k < Kp; k += 32) Tj[k] = x[k];
}

// Model sampling, kSiFits fits per CTA on the FP64 tensor pipe (mma.sync m8n8k4 f64, SASS DMMA):
//   B = Q_s^T R  (Kp x 8): A operand = rows 3 id_i + d of Q (gathered), B operand = the residuals r = cp - ref - mean of the
//                          8 fits, formed while they are loaded; the 3 n reduction is split over the warps and summed in warp order
//   alpha' = alpha + (T B - alpha) step  (K x 8): A operand = T, B operand = B from shared memory
// A fit whose projector factor was not positive definite, or whose new coefficients are not finite, keeps its coefficients
// (wstat != 0). NB: row blocks of 8 (Kp / 8 <= NBMAX).
template <int NBMAX>
__global__ void __launch_bounds__(kSiWarps * 32) k_si_project(ModelDev m, int nm, int n_ids, int NB, double step,
                                                              const int *__restrict__ ids, const double *__restrict__ cp,
                                                              const double *__restrict__ T, const int *__restrict__ proj_status,
                                                              double *__restrict__ theta_w, int *__restrict__ wstat) {
    __shared__ double sB[NBMAX * 8][kSiFits];      // B[k][f]
    __shared__ double sA[kSiFits][NBMAX * 8];      // alpha'[f][j]
    __shared__ int sbad[kSiFits];
    const int Kp = m.Kp, K = m.K, Lt = K + kTheta0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, row = lane >> 2, col = lane & 3;
    const int f0 = blockIdx.x * kSiFits, nf = min(kSiFits, nm - f0);
    if (threadIdx.x < kSiFits) sbad[threadIdx.x] = 0;
    double acc[NBMAX][2];
#pragma unroll
    for (int kb = 0; kb < NBMAX; kb++) acc[kb][0] = acc[kb][1] = 0.0;
    const int J = 3 * n_ids, nchunks = (J + 3) >> 2;
    for (int ch = warp; ch < nchunks; ch += kSiWarps) {
        const int j = 4 * ch + col;       // reduction index of this lane, both operands
        double b = 0.0;
        int qrow = -1;
        if (j < J) {
            const int i = j / 3, d = j - 3 * i, id = __ldg(ids + i);
            qrow = 3 * id + d;
            if (row < nf) b = (__ldg(cp + ((size_t)(f0 + row) * n_ids + i) * 3 + d) - __ldg(m.ref + qrow)) - __ldg(m.mean + qrow);
        }
        const double *q = qrow >= 0 ? m.Q + (size_t)qrow * Kp + row : nullptr;
#pragma unroll
        for (int kb = 0; kb < NBMAX; kb++)
            if (kb < NB) dmma_8x8x4(acc[kb][0], acc[kb][1], q ? __ldg(q + 8 * kb) : 0.0, b);
    }
    // C[8 kb + row][2 col + e]: the warps' partial sums, added in warp order (independent of the batch and the schedule)
    for (int w = 0; w < kSiWarps; w++) {
        if (warp == w) {
#pragma unroll
            for (int kb = 0; kb < NBMAX; kb++)
                if (kb < NB)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        double &dst = sB[8 * kb + row][2 * col + e];
                        dst = w == 0 ? acc[kb][e] : dst + acc[kb][e];
                    }
        }
        __syncthreads();
    }
    const bool proj_bad = *proj_status != 0;
    for (int jb = warp; jb < NB; jb += kSiWarps) {
        double c0 = 0.0, c1 = 0.0;
        const double *Trow = T + (size_t)(8 * jb + row) * Kp;
        for (int kc = 0; kc < Kp / 4; kc++) dmma_8x8x4(c0, c1, __ldg(Trow + 4 * kc + col), sB[4 * kc + col][row]);
        const int j = 8 * jb + row;
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int f = 2 * col + e;
            if (j < K && f < nf) {
                const double a = theta_w[(size_t)(f0 + f) * Lt + kTheta0 + j];
                const double v = a + ((e ? c1 : c0) - a) * step;   // IcpBasedSurfaceFitting.scala:84-85
                sA[f][j] = v;
                if (!isfinite(v)) sbad[f] = ICP_STD_ICP_NON_FINITE;
            }
        }
    }
    __syncthreads();
    for (int f = warp; f < nf; f += kSiWarps) {
        const int st = proj_bad ? ICP_STD_ICP_NOT_POSITIVE_DEFINITE : sbad[f];
        if (st == 0)
            for (int j = lane; j < K; j += 32) theta_w[(size_t)(f0 + f) * Lt + kTheta0 + j] = sA[f][j];
        if (lane == 0) wstat[f0 + f] = st;
    }
}

// Target sampling: alpha' = alpha + (S^T mu - alpha) step (k_std_icp_step) unless the factorisation failed or alpha' is not finite
__global__ void __launch_bounds__(128) k_si_target_step(int nt, int K, int Kp, double step, const double *__restrict__ S,
                                                        const double *__restrict__ mu, const int *__restrict__ fstatus,
                                                        double *__restrict__ theta_w, int *__restrict__ wstat) {
    extern __shared__ double sa[];
    const int c = blockIdx.x, Lt = K + kTheta0;
    double *a = theta_w + (size_t)c * Lt + kTheta0;
    int mine = 0;
    for (int j = threadIdx.x; j < K; j += blockDim.x) {
        double acc = 0.0;
        for (int k = 0; k < Kp; k++) acc = fma(S[(size_t)k * Kp + j], mu[(size_t)c * Kp + k], acc);
        const double v = a[j] + (acc - a[j]) * step;
        sa[j] = v;
        mine |= !isfinite(v);
    }
    const int bad = __syncthreads_or(mine);
    const int st = fstatus[c] ? ICP_STD_ICP_NOT_POSITIVE_DEFINITE : bad ? ICP_STD_ICP_NON_FINITE : 0;
    if (st == 0)
        for (int j = threadIdx.x; j < K; j += blockDim.x) a[j] = sa[j];
    if (threadIdx.x == 0) wstat[c] = st;
}

// ---- host Philox4x32-10, bit-identical to chain_philox (icp_device.cuh) ----
uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
void host_philox(uint64_t seed, uint64_t chain, uint32_t step, uint32_t block, uint32_t out[4]) {
    uint32_t c0 = (uint32_t)chain, c1 = (uint32_t)(chain >> 32), c2 = step, c3 = block;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
struct icp_std_icp_s {
    icp_model model = nullptr;
    icp_target target = nullptr;              // targets[0]: the primitive kind and the single-target structures
    int n_ids = 0, n_tp = 0, max_fits = 0, direction = 0;
    double step = 1.0;
    DevBuf<int> ids;
    DevBuf<double> tp, Gs;                    // tp: [G][n_tp][3], the entries' point lists end to end
    // target set (icp_std_icp_create_targets); with one target nothing below is allocated and every launch is the
    // single-target one
    int n_targets = 1;
    std::vector<icp_target> targets;          // [G] (references held)
    DevBuf<TargetRec> trec;                   // [G]
    std::vector<int> tidx_req;                // icp_std_icp_set_target_index: the target of every fit of the next runs
    DevBuf<int> tidx, wtidx;                  // [max_fits] target of every fit / of every work slot
    DevBuf<double> tp_w;                      // [max_fits][n_tp][3] point lists of the target-sampling work slots
    // workspaces, sized for max_fits at the first run (graph capture cannot allocate)
    bool sized = false;
    DevBuf<double> theta, theta_w, theta0, X, cp, F, y, L, mu, b, Mp, M;
    DevBuf<int> status, done, wstat, iter, seed_m, seed_t, wseed_m, wseed_t, prim, vid, nobs, fstatus;
    // per run: projectors T [n_sigma][Kp][Kp] and their factorisation status, the split of every iteration, staged outputs
    DevBuf<double> T, PM, PL, Pmu, Pb, PMp;
    DevBuf<int> pstatus, perm, log_dir;
    DevBuf<double> log_alpha, alpha_out;
    DevBuf<RunIo> io;
    struct Graph { cudaGraphExec_t exec = nullptr; int nodes = 0; bool eager = false; };
    std::map<std::string, Graph> graphs;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double last_ms = 0;
    int64_t last_launches = 0;
    void drop_graphs() {
        for (auto &g : graphs) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
        graphs.clear();
    }
    ~icp_std_icp_s() {
        drop_graphs();
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
    }
};

extern "C" int32_t icp_std_icp_create_targets(icp_model m, int32_t n_targets, const icp_std_icp_target *targets,
                                              const int32_t *model_point_ids, int32_t n_ids, int32_t n_tp, double step_length,
                                              int32_t direction, int32_t max_fits, icp_std_icp *out) {
    icp_std_icp h = nullptr;
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(m && targets && out && n_targets >= 1, "null argument");
        ICP_REQUIRE(direction == ICP_MODEL_SAMPLING || direction == ICP_TARGET_SAMPLING || direction == ICP_MODEL_AND_TARGET_SAMPLING,
                    "bad direction");
        ICP_REQUIRE(max_fits >= 1, "max_fits must be >= 1");
        ICP_REQUIRE(std::isfinite(step_length), "step_length must be finite");
        ICP_REQUIRE(n_ids >= 1 && model_point_ids, "model sampling needs at least one model point id");
        ICP_REQUIRE(n_tp >= 1, "target sampling needs at least one target point");
        for (int i = 0; i < n_ids; i++) ICP_REQUIRE(model_point_ids[i] >= 0 && model_point_ids[i] < m->N, "model point id out of range");
        for (int g = 0; g < n_targets; g++) {
            const std::string e = "targets[" + std::to_string(g) + "]";
            ICP_REQUIRE(targets[g].target, e + ".target is null");
            ICP_REQUIRE(targets[g].target_points, e + ".target_points is null");
            ICP_REQUIRE(targets[g].target->ctx == m->ctx, e + ".target: model and target belong to different contexts");
            for (int i = 0; i < 3 * n_tp; i++)
                ICP_REQUIRE(std::isfinite(targets[g].target_points[i]), e + ".target_points must be finite");
        }
        CtxLock lock(_ctx);
        cudaStream_t s = _ctx->stream;
        h = new icp_std_icp_s();
        h->model = m; h->target = targets[0].target; h->n_ids = n_ids; h->n_tp = n_tp; h->max_fits = max_fits;
        h->direction = direction; h->step = step_length; h->n_targets = n_targets;
        for (int g = 0; g < n_targets; g++) h->targets.push_back(targets[g].target);
        h->ids.upload(model_point_ids, n_ids, s);
        h->tp.alloc((size_t)n_targets * n_tp * 3);
        for (int g = 0; g < n_targets; g++)
            ICP_CUDA(cudaMemcpyAsync(h->tp.p + (size_t)g * n_tp * 3, targets[g].target_points, sizeof(double) * n_tp * 3,
                                     cudaMemcpyHostToDevice, s));
        if (n_targets > 1) {
            upload_target_table(h->targets, h->trec, s);
            // fixed addresses: the iteration graphs read them
            h->tidx.alloc(max_fits); h->wtidx.alloc(max_fits);
            h->tp_w.alloc((size_t)max_fits * n_tp * 3);
        }
        h->Gs.alloc((size_t)m->Kp * m->Kp);
        launch_gram_rows(m->dev(), n_ids, h->ids.p, h->Gs.p, s);
        ICP_CUDA(cudaEventCreate(&h->ev0));
        ICP_CUDA(cudaEventCreate(&h->ev1));
        ICP_CUDA(cudaStreamSynchronize(s));
        m->refs++;
        for (icp_target t : h->targets) t->refs++;
        *out = h;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete h;
        return rc;
    }
}

extern "C" int32_t icp_std_icp_create(icp_model m, icp_target t, const int32_t *model_point_ids, int32_t n_ids,
                                      const double *target_points, int32_t n_tp, double step_length, int32_t direction,
                                      int32_t max_fits, icp_std_icp *out) {
    const icp_std_icp_target one{t, target_points};
    return icp_std_icp_create_targets(m, 1, &one, model_point_ids, n_ids, n_tp, step_length, direction, max_fits, out);
}

extern "C" int32_t icp_std_icp_set_target_index(icp_std_icp h, int32_t C, const int32_t *target_index) {
    icp_ctx _ctx = h ? h->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr && target_index != nullptr, "null argument");
        CtxLock lock(_ctx);
        ICP_REQUIRE(C >= 1 && C <= h->max_fits, "C must be in [1, max_fits]");
        for (int i = 0; i < C; i++)
            ICP_REQUIRE(target_index[i] >= 0 && target_index[i] < h->n_targets,
                        "target_index[" + std::to_string(i) + "] = " + std::to_string(target_index[i]) + " is outside [0, n_targets)");
        h->tidx_req.assign(target_index, target_index + C);
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_std_icp_destroy(icp_std_icp h) {
    if (!h) return ICP_OK;
    icp_ctx _ctx = h->model->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_CUDA(cudaStreamSynchronize(_ctx->stream));
        h->model->refs--;
        for (icp_target t : h->targets) t->refs--;
        delete h;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

namespace {

void size_workspaces(icp_std_icp h) {
    if (h->sized) return;
    icp_model m = h->model;
    const size_t C = h->max_fits, Lt = m->K + kTheta0, Kp = m->Kp, nt = h->n_tp, ni = h->n_ids;
    const size_t NB = Kp / 8;
    h->theta.alloc(C * Lt); h->theta_w.alloc(C * Lt); h->theta0.alloc(C * Lt);
    h->X.alloc(C * m->N * 3); h->cp.alloc(C * ni * 3);
    h->status.alloc(C); h->done.alloc(C); h->wstat.alloc(C); h->iter.alloc(1); h->fstatus.alloc(C);
    h->seed_m.alloc(C * ni); h->wseed_m.alloc(C * ni); h->seed_t.alloc(C * nt); h->wseed_t.alloc(C * nt);
    h->prim.alloc(C * nt); h->vid.alloc(C * nt); h->F.alloc(C * nt * 9); h->y.alloc(C * nt * 3); h->nobs.alloc(2 * C);
    h->L.alloc(C * Kp * Kp); h->mu.alloc(C * Kp); h->b.alloc(C * Kp); h->Mp.alloc(C * NB * (NB + 1) / 2 * 64);
    if (NB > 13) h->M.alloc(C * Kp * Kp);   // the general rank update + Cholesky pair above rank 104 (launch_posterior_fused)
    h->PM.alloc(Kp * Kp); h->PL.alloc(Kp * Kp); h->Pmu.alloc(Kp); h->Pb.alloc(Kp); h->PMp.alloc(NB * (NB + 1) / 2 * 64);
    h->io.alloc(1);
    h->sized = true;
}

// one iteration of C fits, nm of them model sampling (work slots [0, nm)), at projector / noise sigma index si
void enqueue_iteration(icp_std_icp h, int C, int nm, int si, double sigma2, cudaStream_t s) {
    icp_model m = h->model;
    icp_target t = h->target;
    const ModelDev md = m->dev();
    const int K = m->K, Kp = m->Kp, Lt = K + kTheta0, nt = C - nm, ni = h->n_ids, ntp = h->n_tp;
    const bool multi = h->n_targets > 1;
    k_si_gather<<<C, 128, 0, s>>>(C, Lt, nm, ni, ntp, h->iter.p, h->io.p, h->theta.p, h->status.p, h->theta_w.p, h->seed_m.p,
                                  h->seed_t.p, h->wseed_m.p, h->wseed_t.p, multi ? h->tidx.p : nullptr, h->wtidx.p);
    ICP_CUDA(cudaGetLastError());
    launch_reconstruct(md, C, h->theta_w.p, h->X.p, s);
    if (nm > 0) {
        // :73 target.operations.closestPointOnSurface of the sampled model points
        NearestArgs a;
        a.bvh = &t->tri_bvh; a.prim_data = t->tri_data.p; a.wide = t->wide(); a.sm_count = t->ctx->sm_count; a.C = nm; a.nq = ni;
        a.Xq = h->X.p; a.q_ids = h->ids.p; a.Nq = m->N; a.out_cp = h->cp.p; a.seed_slot = h->wseed_m.p;
        if (multi) { a.mt_rec = h->trec.p; a.mt_idx = h->wtidx.p; }   // slot p walks the BVH of its own target
        launch_nearest(a, s);
        const int NB = Kp / 8, grid = (nm + kSiFits - 1) / kSiFits;
        const double *T = h->T.p + (size_t)si * Kp * Kp;
        const int *ps = h->pstatus.p + si;
        if (NB <= 7) k_si_project<7><<<grid, kSiWarps * 32, 0, s>>>(md, nm, ni, NB, h->step, h->ids.p, h->cp.p, T, ps, h->theta_w.p, h->wstat.p);
        else if (NB <= 13) k_si_project<13><<<grid, kSiWarps * 32, 0, s>>>(md, nm, ni, NB, h->step, h->ids.p, h->cp.p, T, ps, h->theta_w.p, h->wstat.p);
        else k_si_project<28><<<grid, kSiWarps * 32, 0, s>>>(md, nm, ni, NB, h->step, h->ids.p, h->cp.p, T, ps, h->theta_w.p, h->wstat.p);
        ICP_CUDA(cudaGetLastError());
    }
    if (nt > 0) {
        // :118 currentMesh.pointSet.findClosestPoint(targetPoint), then model.posterior(corr, sigma2) (:81) with isotropic noise
        double *th_t = h->theta_w.p + (size_t)nm * Lt;
        const double *X_t = h->X.p + (size_t)nm * m->N * 3;
        // on a target set every slot reads its own target's point list, gathered into [nt][n_tp][3]
        const double *tp = h->tp.p;
        if (multi) {
            launch_gather_target_rows(nt, 3 * ntp, h->wtidx.p + nm, h->tp.p, h->tp_w.p, s);
            tp = h->tp_w.p;
        }
        nearest_model_vertex(m, nt, X_t, ntp, tp, multi ? 1 : 0, h->wseed_t.p, h->prim.p, s);
        ObsArgs oa{};
        oa.m = md; oa.C = nt; oa.theta = th_t; oa.X = X_t;
        oa.prm.step_length = h->step; oa.prm.tangential_noise = 1; oa.prm.noise_along_normal = 1;
        oa.prm.direction = ICP_TARGET_SAMPLING; oa.prm.boundary_aware = 0; oa.prm.factor = ICP_FACTOR_CHOLESKY;
        oa.prm.rank_update = ICP_RANK_UPDATE_FP64;
        oa.tp = tp; oa.tp_per_chain = multi ? 1 : 0; oa.near_vid = h->prim.p; oa.iso = 1; oa.iso_sigma2 = sigma2; oa.world_frame = 1;
        ObsDev od{ntp, h->vid.p, h->F.p, h->y.p, h->nobs.p};
        od.nrows = h->nobs.p + nt;
        launch_observations(oa, od, s);
        if (!launch_posterior_fused(md, nt, od, nullptr, nullptr, h->L.p, h->mu.p, nullptr, h->fstatus.p, h->Mp.p, h->b.p, s)) {
            launch_posterior_build(md, nt, od, h->M.p, h->b.p, s);
            launch_cholesky_solve(nt, K, Kp, h->M.p, h->b.p, h->L.p, h->mu.p, nullptr, h->fstatus.p, s, h->Mp.p);
        }
        k_si_target_step<<<nt, 128, sizeof(double) * K, s>>>(nt, K, Kp, h->step, m->S.p, h->mu.p, h->fstatus.p, th_t, h->wstat.p + nm);
        ICP_CUDA(cudaGetLastError());
    }
    k_si_scatter<<<C, 128, 0, s>>>(C, K, Lt, nm, ni, ntp, h->iter.p, h->io.p, h->theta_w.p, h->wstat.p, h->theta.p, h->status.p,
                                   h->done.p, h->seed_m.p, h->seed_t.p, h->wseed_m.p, h->wseed_t.p);
    k_si_next<<<1, 1, 0, s>>>(h->iter.p);
    ICP_CUDA(cudaGetLastError());
}

// directions of every iteration and fit: the caller's, the handle's fixed one, or the Philox coin
std::vector<int> plan_directions(icp_std_icp h, int C, int iters, const int32_t *h_dirs, uint64_t seed, uint64_t off) {
    std::vector<int> dir((size_t)iters * C);
    for (size_t e = 0; e < dir.size(); e++) {
        if (h_dirs) {
            ICP_REQUIRE(h_dirs[e] == ICP_MODEL_SAMPLING || h_dirs[e] == ICP_TARGET_SAMPLING, "directions must be 0 or 1");
            dir[e] = h_dirs[e];
        } else if (h->direction != ICP_MODEL_AND_TARGET_SAMPLING) {
            dir[e] = h->direction;
        } else {
            // IcpBasedSurfaceFitting.scala:67 `if (rand.nextDouble() < 0.5) ModelSampling else TargetSampling`: Philox block 0 of
            // (seed, global fit id, iteration), words x / y as the 53-bit uniform of the chain runner (u53)
            const int it = (int)(e / C), c = (int)(e % C);
            uint32_t r[4];
            host_philox(seed, off + (uint64_t)c, (uint32_t)it, 0u, r);
            const double u = (double)(((uint64_t)(r[0] >> 5) << 26) | (uint64_t)(r[1] >> 6)) * (1.0 / 9007199254740992.0);
            dir[e] = u < 0.5 ? ICP_MODEL_SAMPLING : ICP_TARGET_SAMPLING;
        }
    }
    return dir;
}

void std_icp_run(icp_std_icp h, int C, const double *theta0_dev, int n_sigma, const double *sigma2, int num_iterations,
                 const std::vector<int> &dir, double *log_alpha, int *log_direction, bool async) {
    icp_model m = h->model;
    icp_ctx ctx = m->ctx;
    cudaStream_t s = ctx->stream;
    const int K = m->K, Kp = m->Kp, Lt = K + kTheta0, per = num_iterations + 1, iters = n_sigma * per;
    // the split of every iteration: model-sampling fits first
    std::vector<int> perm((size_t)iters * C), nm(iters);
    for (int it = 0; it < iters; it++) {
        int *row = perm.data() + (size_t)it * C, q = 0;
        for (int c = 0; c < C; c++) if (dir[(size_t)it * C + c] == ICP_MODEL_SAMPLING) row[q++] = c;
        nm[it] = q;
        for (int c = 0; c < C; c++) if (dir[(size_t)it * C + c] != ICP_MODEL_SAMPLING) row[q++] = c;
    }
    h->perm.ensure(std::max<size_t>(perm.size(), 1));
    if ((size_t)h->T.n < (size_t)n_sigma * Kp * Kp) { h->T.alloc((size_t)std::max(n_sigma, 4) * Kp * Kp); h->pstatus.alloc(std::max(n_sigma, 4)); }
    ICP_CUDA(cudaEventRecord(h->ev0, s));
    int64_t launches = 0;
    ICP_CUDA(cudaMemcpyAsync(h->perm.p, perm.data(), sizeof(int) * perm.size(), cudaMemcpyHostToDevice, s));
    RunIo rio{h->perm.p, log_alpha, log_direction};
    ICP_CUDA(cudaMemcpyAsync(h->io.p, &rio, sizeof rio, cudaMemcpyHostToDevice, s));
    if (h->n_targets > 1)
        ICP_CUDA(cudaMemcpyAsync(h->tidx.p, h->tidx_req.data(), sizeof(int) * (size_t)C, cudaMemcpyHostToDevice, s));
    ICP_CUDA(cudaMemsetAsync(h->seed_m.p, 0xFF, sizeof(int) * (size_t)C * h->n_ids, s));   // no traversal seed yet
    ICP_CUDA(cudaMemsetAsync(h->seed_t.p, 0xFF, sizeof(int) * (size_t)C * h->n_tp, s));
    k_si_init<<<C, 128, 0, s>>>(C, Lt, theta0_dev, h->theta.p, h->status.p, h->done.p, h->iter.p);
    ICP_CUDA(cudaGetLastError());
    launches += 3;
    // T_sigma = S^T (sigma2 I + G_s)^-1 for every sigma that has a model-sampling iteration
    for (int si = 0; si < n_sigma; si++) {
        bool any = false;
        for (int it = si * per; it < (si + 1) * per && !any; it++) any = nm[it] > 0;
        if (!any) continue;
        k_si_shift<<<Kp, 64, 0, s>>>(Kp, sigma2[si], h->Gs.p, h->PM.p, h->Pb.p);
        ICP_CUDA(cudaGetLastError());
        launch_cholesky_solve(1, K, Kp, h->PM.p, h->Pb.p, h->PL.p, h->Pmu.p, nullptr, h->pstatus.p + si, s, h->PMp.p);
        k_si_projector<<<Kp, 32, sizeof(double) * Kp, s>>>(K, Kp, h->PL.p, m->S.p, h->T.p + (size_t)si * Kp * Kp);
        ICP_CUDA(cudaGetLastError());
        launches += Kp > 160 ? 4 : 3;
    }
    // iterations: one graph per (C, split, sigma), captured at its first use and replayed
    std::string base;
    {
        const void *bufs[] = {m->vert_bvh.nodes.p, m->vert_bvh.nodebox.p, m->vert_bvh.counters.p, h->T.p, h->pstatus.p, h->trec.p,
                              h->wtidx.p};
        base.append((const char *)bufs, sizeof bufs);
        base.append((const char *)&C, sizeof C);
    }
    if (h->graphs.size() > 256) h->drop_graphs();
    for (int it = 0; it < iters; it++) {
        const int si = it / per;
        std::string key = base;
        key.append((const char *)&nm[it], sizeof(int));
        key.append((const char *)&si, sizeof si);
        key.append((const char *)&sigma2[si], sizeof(double));
        auto &g = h->graphs[key];
        if (!g.exec && !g.eager) {
            cudaGraph_t graph = nullptr;
            bool ok = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                try { enqueue_iteration(h, C, nm[it], si, sigma2[si], s); } catch (...) { ok = false; }
                if (cudaStreamEndCapture(s, &graph) != cudaSuccess || !graph) ok = false;
            }
            if (ok) {
                size_t nn = 0;
                cudaGraphGetNodes(graph, nullptr, &nn);
                std::vector<cudaGraphNode_t> nodes(nn);
                cudaGraphGetNodes(graph, nodes.data(), &nn);
                for (size_t i = 0; i < nn; i++) {
                    cudaGraphNodeType ty;
                    if (cudaGraphNodeGetType(nodes[i], &ty) == cudaSuccess && (ty == cudaGraphNodeTypeKernel || ty == cudaGraphNodeTypeMemset)) g.nodes++;
                }
                if (cudaGraphInstantiate(&g.exec, graph, 0) != cudaSuccess) { g.exec = nullptr; ok = false; }
            }
            if (graph) cudaGraphDestroy(graph);
            if (!ok) { cudaGetLastError(); g.eager = true; }   // not capturable here (e.g. a lazily grown model scratch): stay eager
        }
        if (g.exec) ICP_CUDA(cudaGraphLaunch(g.exec, s));
        else enqueue_iteration(h, C, nm[it], si, sigma2[si], s);
        launches += g.nodes;
    }
    ICP_CUDA(cudaEventRecord(h->ev1, s));
    h->last_launches = launches;
    h->last_ms = 0;
    if (!async) {
        ICP_CUDA(cudaStreamSynchronize(s));
        float ms = 0;
        cudaEventElapsedTime(&ms, h->ev0, h->ev1);
        h->last_ms = ms;
    }
}

void check_run_args(icp_std_icp h, int C, const void *theta0, int n_sigma, const double *sigma2, int num_iterations, const void *io) {
    ICP_REQUIRE(theta0 && sigma2 && io, "null argument");
    ICP_REQUIRE(C >= 1 && C <= h->max_fits, "C must be in [1, max_fits]");
    ICP_REQUIRE(n_sigma >= 1, "n_sigma must be >= 1");
    for (int i = 0; i < n_sigma; i++) ICP_REQUIRE(std::isfinite(sigma2[i]) && sigma2[i] > 0, "every sigma2 must be finite and > 0");
    ICP_REQUIRE(num_iterations >= 0, "num_iterations must be >= 0");
    ICP_REQUIRE((long long)n_sigma * (num_iterations + 1) <= (1LL << 30), "too many iterations");
    ICP_REQUIRE(h->n_targets == 1 || (int)h->tidx_req.size() == C,
                "a handle with several targets needs icp_std_icp_set_target_index with C = " + std::to_string(C) + " entries before a run");
}

}  // namespace

extern "C" int32_t icp_std_icp_run(icp_std_icp h, int32_t C, const double *theta0, int32_t n_sigma, const double *sigma2,
                                   int32_t num_iterations, const icp_std_icp_io *io) {
    icp_ctx _ctx = h ? h->model->ctx : nullptr;
    try {
        ICP_REQUIRE(h, "null handle");
        check_run_args(h, C, theta0, n_sigma, sigma2, num_iterations, io);
        CtxLock lock(_ctx);
        cudaStream_t s = _ctx->stream;
        icp_model m = h->model;
        const int K = m->K, Lt = K + kTheta0, iters = n_sigma * (num_iterations + 1);
        std::vector<int> dir = plan_directions(h, C, iters, io->directions, io->seed, io->fit_id_offset);
        size_workspaces(h);
        ICP_CUDA(cudaMemcpyAsync(h->theta0.p, theta0, sizeof(double) * (size_t)C * Lt, cudaMemcpyHostToDevice, s));
        if (io->log_alpha) h->log_alpha.ensure((size_t)iters * C * K);
        if (io->log_direction) h->log_dir.ensure((size_t)iters * C);
        std_icp_run(h, C, h->theta0.p, n_sigma, sigma2, num_iterations, dir, io->log_alpha ? h->log_alpha.p : nullptr,
                    io->log_direction ? h->log_dir.p : nullptr, true);
        if (io->log_alpha) ICP_CUDA(cudaMemcpyAsync(io->log_alpha, h->log_alpha.p, sizeof(double) * (size_t)iters * C * K, cudaMemcpyDeviceToHost, s));
        if (io->log_direction) ICP_CUDA(cudaMemcpyAsync(io->log_direction, h->log_dir.p, sizeof(int) * (size_t)iters * C, cudaMemcpyDeviceToHost, s));
        if (io->alpha_final)
            ICP_CUDA(cudaMemcpy2DAsync(io->alpha_final, sizeof(double) * K, h->theta.p + kTheta0, sizeof(double) * Lt, sizeof(double) * K, C,
                                       cudaMemcpyDeviceToHost, s));
        if (io->status) ICP_CUDA(cudaMemcpyAsync(io->status, h->status.p, sizeof(int) * C, cudaMemcpyDeviceToHost, s));
        if (io->iterations_done) ICP_CUDA(cudaMemcpyAsync(io->iterations_done, h->done.p, sizeof(int) * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        float ms = 0;
        cudaEventElapsedTime(&ms, h->ev0, h->ev1);
        h->last_ms = ms;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_std_icp_run_device(icp_std_icp h, int32_t C, const double *theta0_dev, int32_t n_sigma, const double *sigma2,
                                          int32_t num_iterations, const icp_std_icp_io *io_dev, int32_t async) {
    icp_ctx _ctx = h ? h->model->ctx : nullptr;
    try {
        ICP_REQUIRE(h, "null handle");
        check_run_args(h, C, theta0_dev, n_sigma, sigma2, num_iterations, io_dev);
        CtxLock lock(_ctx);
        cudaStream_t s = _ctx->stream;
        icp_model m = h->model;
        const int K = m->K, Lt = K + kTheta0, iters = n_sigma * (num_iterations + 1);
        std::vector<int> hd;
        if (io_dev->directions) {   // the split of every iteration is decided on the host
            hd.resize((size_t)iters * C);
            ICP_CUDA(cudaMemcpyAsync(hd.data(), io_dev->directions, sizeof(int) * hd.size(), cudaMemcpyDeviceToHost, s));
            ICP_CUDA(cudaStreamSynchronize(s));
        }
        std::vector<int> dir = plan_directions(h, C, iters, io_dev->directions ? hd.data() : nullptr, io_dev->seed, io_dev->fit_id_offset);
        size_workspaces(h);
        std_icp_run(h, C, theta0_dev, n_sigma, sigma2, num_iterations, dir, io_dev->log_alpha, io_dev->log_direction, true);
        if (io_dev->alpha_final)
            ICP_CUDA(cudaMemcpy2DAsync(io_dev->alpha_final, sizeof(double) * K, h->theta.p + kTheta0, sizeof(double) * Lt, sizeof(double) * K, C,
                                       cudaMemcpyDeviceToDevice, s));
        if (io_dev->status) ICP_CUDA(cudaMemcpyAsync(io_dev->status, h->status.p, sizeof(int) * C, cudaMemcpyDeviceToDevice, s));
        if (io_dev->iterations_done) ICP_CUDA(cudaMemcpyAsync(io_dev->iterations_done, h->done.p, sizeof(int) * C, cudaMemcpyDeviceToDevice, s));
        if (!async) {
            ICP_CUDA(cudaStreamSynchronize(s));
            float ms = 0;
            cudaEventElapsedTime(&ms, h->ev0, h->ev1);
            h->last_ms = ms;
        }
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_std_icp_last_run_stats(icp_std_icp h, double *device_ms, int64_t *launches) {
    if (!h) return ICP_ERR_INVALID_ARGUMENT;
    icp_ctx _ctx = h->model->ctx;
    try {
        CtxLock lock(_ctx);
        if (h->last_ms == 0) {   // an asynchronous run: its events have been recorded, wait for the second
            ICP_CUDA(cudaEventSynchronize(h->ev1));
            float ms = 0;
            if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) == cudaSuccess) h->last_ms = ms;
            cudaGetLastError();
        }
        if (device_ms) *device_ms = h->last_ms;
        if (launches) *launches = h->last_launches;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}
