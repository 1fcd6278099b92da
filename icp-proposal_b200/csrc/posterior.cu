// posterior.cu - the ICP proposal's GP posterior over sampled correspondences.
//
// Replaces (all paths relative to src/main/scala of the reference):
//   launch_observations      modelBased/targetBasedClosestPointsEstimation + surfaceNormalDependantNoise
//                            (api/sampling/proposals/NonRigidIcpProposal.scala:88-131,
//                             api/sampling/SurfaceNoiseHelpers.scala:32-60)
//   launch_posterior_build   interpolatedModel.posterior(obs) (NonRigidIcpProposal.scala:152), the
//                            M = I + sum Q_i^T Sigma_i^-1 Q_i and b = sum Q_i^T Sigma_i^-1 y_i of
//                            LowRankGaussianProcess.regression (SURVEY Appendix A3)
//   launch_cholesky_solve    pinv(M) and mean_coeffs -> Cholesky M = L L^T, mu = M^-1 b
//   launch_propose           propose (NonRigidIcpProposal.scala:53-68) via Appendix A6
//   launch_log_transition    logTransitionProbability (NonRigidIcpProposal.scala:71-85) via Appendix A7
//
// Sigma_i^-1 = F_i^T F_i with F_i rows n/sd_n, t1/sd_t, t2/sd_t (orthonormal frame of the vertex
// normal), so M = I + A^T A with A = stack(F_i Q_i): a batched symmetric rank-3n update in FP64.
#include <algorithm>
#include <cstdlib>

#include "icp_device.cuh"
#include "icp_internal.h"

namespace icp {

// ---------------------------------------------------------------------------------------------------
// observations
// ---------------------------------------------------------------------------------------------------
// One CTA per chain: the chain's mesh is staged in shared memory, then one
// thread per observation gathers the one-ring of its vertex from shared memory - the gather is 4 dependent
// index -> index -> index -> coordinate loads per adjacent triangle, which costs ~30 cycles each from shared
// memory instead of an L2 round trip.
// rows of the whitening frame of vertex id: n / sd_n, t1 / sd_t, t2 / sd_t (SurfaceNoiseHelpers.scala:32-60)
__device__ __forceinline__ void whitening_frame(const ObsArgs &a, const double *Xc, int id, double (&f)[9]) {
    if (a.iso) {
        double w = 1.0 / sqrt(a.iso_sigma2);
        for (int k = 0; k < 9; k++) f[k] = 0.0;
        f[0] = f[4] = f[8] = w;
        return;
    }
    double nx, ny, nz;
    vertex_normal_dev(a.m, Xc, id, nx, ny, nz);                 // :100,120 currentMesh.vertexNormals.atPoint(id)
    // SurfaceNoiseHelpers.scala:39: normalize again
    double nn = sqrt(nx * nx + ny * ny + nz * nz);
    nx /= nn; ny /= nn; nz /= nn;
    // :44-48 candidate = n x e_x; (inverted) fallback test; n x e_y otherwise
    double c0 = 0.0, c1 = nz, c2 = -ny;
    double t1x, t1y, t1z;
    if (c0 * c0 + c1 * c1 + c2 * c2 < 0.0001) { t1x = c0; t1y = c1; t1z = c2; }
    else { t1x = -nz; t1y = 0.0; t1z = nx; }
    double tn = sqrt(t1x * t1x + t1y * t1y + t1z * t1z);
    t1x /= tn; t1y /= tn; t1z /= tn;                             // 0/0 = NaN exactly where the reference yields NaN
    double t2x = ny * t1z - nz * t1y, t2y = nz * t1x - nx * t1z, t2z = nx * t1y - ny * t1x;
    double t2n = sqrt(t2x * t2x + t2y * t2y + t2z * t2z);
    t2x /= t2n; t2y /= t2n; t2z /= t2n;
    double wn = 1.0 / a.prm.noise_along_normal, wt = 1.0 / a.prm.tangential_noise;
    f[0] = nx * wn; f[1] = ny * wn; f[2] = nz * wn;
    f[3] = t1x * wt; f[4] = t1y * wt; f[5] = t1z * wt;
    f[6] = t2x * wt; f[7] = t2y * wt; f[8] = t2z * wt;
}

// Target sampling, one CTA per chain: observations that share their closest model vertex v also share the frame F_v
// (it depends on the vertex normal only), so their m_v contributions  Q_v^T F_v^T F_v Q_v  and  Q_v^T F_v^T F_v y_i
// collapse into ONE row triple  sqrt(m_v) F_v Q_v  with right-hand side  F_v (sum_i y_i) / sqrt(m_v).  With 2000
// target points on a 1622-vertex model ~40 % of the rows disappear before the rank update (used when n >= N / 2).  The grouping is a
// counting sort by vertex id in shared memory; every segment is put in ascending observation order before its y_i
// are summed, so the result does not depend on the order the atomics landed in.
__device__ __forceinline__ void observations_grouped(const ObsArgs &a, const ObsDev &o, int c, const double *sX, int *s_int) {
    const ModelDev &m = a.m;
    const int N = m.N, n = o.n, tid = threadIdx.x, nt = blockDim.x;
    int *s_cnt = s_int, *s_off = s_cnt + N, *s_slot = s_off + N, *s_cur = s_slot + N, *s_seg = s_cur + N;
    __shared__ int s_part[2][256], s_tot[2];
    const int *near = a.near_vid + (size_t)c * n;
    const double *tp = a.tp + (a.tp_per_chain ? (size_t)c * n * 3 : 0);
    for (int v = tid; v < N; v += nt) { s_cnt[v] = 0; s_cur[v] = 0; }
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
        int id = near[i];                                               // :118 findClosestPoint on the current mesh
        if (id >= 0 && !(a.prm.boundary_aware && m.boundary[id])) atomicAdd(&s_cnt[id], 1);  // :119,124
    }
    __syncthreads();
    // exclusive scans of the counts (segment offsets) and of the non-empty flags (output slots)
    const int per = (N + nt - 1) / nt, v0 = tid * per, v1 = min(N, v0 + per);
    int sc = 0, sf = 0;
    for (int v = v0; v < v1; v++) { sc += s_cnt[v]; sf += s_cnt[v] > 0; }
    s_part[0][tid] = sc; s_part[1][tid] = sf;
    __syncthreads();
    if (tid < 2) {
        int run = 0;
        for (int t = 0; t < nt; t++) { int x = s_part[tid][t]; s_part[tid][t] = run; run += x; }
        s_tot[tid] = run;
    }
    __syncthreads();
    sc = s_part[0][tid]; sf = s_part[1][tid];
    for (int v = v0; v < v1; v++) { s_off[v] = sc; s_slot[v] = sf; sc += s_cnt[v]; sf += s_cnt[v] > 0; }
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
        int id = near[i];
        if (id >= 0 && !(a.prm.boundary_aware && m.boundary[id])) s_seg[s_off[id] + atomicAdd(&s_cur[id], 1)] = i;
    }
    __syncthreads();
    const int kept = s_tot[0], rows = s_tot[1];
    if (tid == 0) { o.nobs[c] = kept; if (o.nrows) o.nrows[c] = rows; }
    const double *th = a.theta + (size_t)c * (m.K + kTheta0);
    double R[9];
    pose_matrix(th, R);
    for (int v = tid; v < N; v += nt) {
        const int mv = s_cnt[v];
        if (mv == 0) continue;
        int *seg = s_seg + s_off[v];
        for (int p = 1; p < mv; p++) {                                   // ascending observation order
            int key = seg[p], q = p - 1;
            while (q >= 0 && seg[q] > key) { seg[q + 1] = seg[q]; q--; }
            seg[q + 1] = key;
        }
        double f[9];
        whitening_frame(a, sX, v, f);
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        for (int p = 0; p < mv; p++) {
            const int i = seg[p];
            double ix, iy, iz;
            if (a.world_frame) { ix = tp[3 * i]; iy = tp[3 * i + 1]; iz = tp[3 * i + 2]; }
            else inverse_pose(th, R, tp[3 * i], tp[3 * i + 1], tp[3 * i + 2], ix, iy, iz);  // :129
            s0 += (ix - m.ref[3 * v]) - m.mean[3 * v];
            s1 += (iy - m.ref[3 * v + 1]) - m.mean[3 * v + 1];
            s2 += (iz - m.ref[3 * v + 2]) - m.mean[3 * v + 2];
        }
        const long long g = (long long)c * n + s_slot[v];
        double *F = o.F + 9 * g, *y = o.y + 3 * g;
        o.vid[g] = v;
        if (mv > 1) {
            const double w = sqrt((double)mv);
            for (int k = 0; k < 9; k++) f[k] *= w;
            s0 /= mv; s1 /= mv; s2 /= mv;                                // F_v sum / sqrt(m) = (sqrt(m) F_v) (sum / m)
        }
        for (int k = 0; k < 9; k++) F[k] = f[k];
        y[0] = f[0] * s0 + f[1] * s1 + f[2] * s2;
        y[1] = f[3] * s0 + f[4] * s1 + f[5] * s2;
        y[2] = f[6] * s0 + f[7] * s1 + f[8] * s2;
    }
    for (int u = rows + tid; u < n; u += nt) {                           // unused slots contribute nothing
        const long long g = (long long)c * n + u;
        o.vid[g] = -1;
        for (int k = 0; k < 9; k++) o.F[9 * g + k] = 0.0;
        o.y[3 * g] = o.y[3 * g + 1] = o.y[3 * g + 2] = 0.0;
    }
}

// stages chain c's mesh in shared memory (coalesced, 8 loads in flight per thread)
__device__ __forceinline__ void stage_mesh(const ObsArgs &a, int c, double *sX) {
    const int n3 = 3 * a.m.N;
    const double *Xg = a.X + (size_t)c * n3;
    for (int e0 = threadIdx.x; e0 < n3; e0 += 8 * blockDim.x) {
        double tmp[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { int e = e0 + u * blockDim.x; tmp[u] = e < n3 ? __ldg(Xg + e) : 0.0; }
#pragma unroll
        for (int u = 0; u < 8; u++) { int e = e0 + u * blockDim.x; if (e < n3) sX[e] = tmp[u]; }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256) k_observations_grouped(ObsArgs a, ObsDev o) {
    extern __shared__ double sX[];
    stage_mesh(a, blockIdx.x, sX);
    observations_grouped(a, o, blockIdx.x, sX, reinterpret_cast<int *>(sX + 3 * a.m.N));
}

template <bool STAGED>
__global__ void __launch_bounds__(256) k_observations(ObsArgs a, ObsDev o) {
    extern __shared__ double sX[];
    const ModelDev &m = a.m;
    int c;
    long long g;
    int i;
    const double *Xc;
    if (STAGED) {
        c = blockIdx.x;
        stage_mesh(a, c, sX);
        Xc = sX;
        if (threadIdx.x == 0 && o.nrows) o.nrows[o.row ? o.row[c] : c] = o.n;
    } else {
        long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (gt >= (long long)a.C * o.n) return;
        c = (int)(gt / o.n);
        if (gt % o.n == 0 && o.nrows) o.nrows[o.row ? o.row[c] : c] = o.n;
        Xc = a.X + (size_t)c * m.N * 3;
    }
    const int r = o.row ? o.row[c] : c;   // where chain c's observations go
    const double *th = a.theta + (size_t)c * (m.K + kTheta0);
    for (int i0 = STAGED ? threadIdx.x : 0; i0 < (STAGED ? o.n : 1); i0 += blockDim.x) {
        if (STAGED) { i = i0; g = (long long)c * o.n + i; }
        else { g = (long long)blockIdx.x * blockDim.x + threadIdx.x; i = (int)(g % o.n); }
        int id;
        double tx, ty, tz;
        bool drop = false;
        if (a.prm.direction == ICP_TARGET_SAMPLING) {
            id = a.near_vid[g];                                         // :118 findClosestPoint on the current mesh
            const double *tpi = a.tp + ((a.tp_per_chain ? (size_t)c * o.n : 0) + i) * 3;
            tx = tpi[0]; ty = tpi[1]; tz = tpi[2];
            if (id < 0) drop = true;
            else if (a.prm.boundary_aware && m.boundary[id]) drop = true;  // :119,124
        } else {
            id = a.ids[i];
            const double *cpp = a.cp + ((size_t)c * a.cp_stride + (a.cp_map ? a.cp_map[i] : i)) * 3;
            tx = cpp[0]; ty = cpp[1]; tz = cpp[2];                          // :97 closest point on the target
            if (a.prm.boundary_aware && a.cp_on_boundary && a.cp_on_boundary[g]) drop = true;  // :99,104
        }
        const long long go = (long long)r * o.n + i;
        double *F = o.F + 9 * go, *y = o.y + 3 * go;
        if (drop) {
            o.vid[go] = -1;
            for (int k = 0; k < 9; k++) F[k] = 0.0;
            y[0] = y[1] = y[2] = 0.0;
            continue;
        }
        atomicAdd(&o.nobs[c], 1);
        o.vid[go] = id;
        double f[9];
        whitening_frame(a, Xc, id, f);
        double R[9];
        pose_matrix(th, R);
        double ix, iy, iz;
        if (a.world_frame) { ix = tx; iy = ty; iz = tz; }
        else inverse_pose(th, R, tx, ty, tz, ix, iy, iz);               // :108,129 inversePoseTransform(targetPoint)
        double y0 = (ix - m.ref[3 * id]) - m.mean[3 * id], y1 = (iy - m.ref[3 * id + 1]) - m.mean[3 * id + 1],
               y2 = (iz - m.ref[3 * id + 2]) - m.mean[3 * id + 2];
        for (int k = 0; k < 9; k++) F[k] = f[k];
        y[0] = f[0] * y0 + f[1] * y1 + f[2] * y2;
        y[1] = f[3] * y0 + f[4] * y1 + f[5] * y2;
        y[2] = f[6] * y0 + f[7] * y1 + f[8] * y2;
        if (o.nonfinite) {
            bool fin = isfinite(y[0]) && isfinite(y[1]) && isfinite(y[2]);
            for (int k = 0; k < 9; k++) fin = fin && isfinite(f[k]);
            if (!fin) o.nonfinite[r] = 1;
        }
    }
}

void launch_observations(const ObsArgs &a, const ObsDev &o, cudaStream_t s) {
    ProfScope _ps(ST_OBSERVATIONS, s);
    long long total = (long long)a.C * o.n;
    if (o.nrows == o.nobs + a.C) {   // the usual layout: one clear for both counters
        ICP_CUDA(cudaMemsetAsync(o.nobs, 0, sizeof(int) * 2 * a.C, s));
    } else {
        ICP_CUDA(cudaMemsetAsync(o.nobs, 0, sizeof(int) * a.C, s));
        // (rows addressed through o.row: k_observations writes the row count of every chain it observes)
        if (o.nrows && !o.row) ICP_CUDA(cudaMemsetAsync(o.nrows, 0, sizeof(int) * a.C, s));
    }
    if (total <= 0) return;
    static const bool no_group = getenv("ICPCUDA_NO_GROUPING") && getenv("ICPCUDA_NO_GROUPING")[0] == '1';
    // grouping needs the per-chain row count to be honoured downstream (o.nrows); it pays once vertices are shared
    // often (n target points on N vertices leave ~N (1 - exp(-n / N)) distinct ones): below n = N / 2 fewer than
    // a fifth of the rows would go, less than the sort costs
    const int grouped = a.prm.direction == ICP_TARGET_SAMPLING && o.nrows && !no_group && 2 * (long long)o.n >= a.m.N;
    size_t smem = sizeof(double) * 3 * (size_t)a.m.N;
    size_t smem_g = smem + sizeof(int) * (4 * (size_t)a.m.N + o.n);
    if (grouped && smem_g <= 160 * 1024) {
        ICP_CUDA(cudaFuncSetAttribute(k_observations_grouped, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g));
        k_observations_grouped<<<a.C, 256, smem_g, s>>>(a, o);
    } else if (smem <= 160 * 1024 && o.n >= 32) {
        ICP_CUDA(cudaFuncSetAttribute(k_observations<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_observations<true><<<a.C, 256, smem, s>>>(a, o);
    } else {
        k_observations<false><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(a, o);
    }
    ICP_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------
// M = I + A^T A, b = A^T y   (one CTA per chain, FP64)
// ---------------------------------------------------------------------------------------------------
constexpr int kPbThreads = 256;
constexpr int kPbObs = 8;  // observations (x3 rows) staged per chunk

__device__ __forceinline__ void tri_index(int idx, int &ti, int &tj) {
    // idx -> (ti, tj) with tj <= ti, row-major over the lower triangle
    int t = (int)((sqrt(8.0 * idx + 1.0) - 1.0) * 0.5);
    while ((t + 1) * (t + 2) / 2 <= idx) t++;
    while (t * (t + 1) / 2 > idx) t--;
    ti = t;
    tj = idx - t * (t + 1) / 2;
}

template <int TILES>  // 4x4 register tiles per thread
__global__ void __launch_bounds__(kPbThreads) k_posterior_build(ModelDev m, ObsDev o, double *__restrict__ M,
                                                                double *__restrict__ bvec) {
    extern __shared__ double sm[];
    const int Kp = m.Kp, nt = Kp / 4, ntiles = nt * (nt + 1) / 2;
    double *sA = sm;                              // [3 kPbObs][Kp]
    double *sy = sm + (size_t)3 * kPbObs * Kp;    // [3 kPbObs]
    int c = blockIdx.x;
    const int *vid = o.vid + (size_t)c * o.n;
    const double *F = o.F + (size_t)c * o.n * 9;
    const double *y = o.y + (size_t)c * o.n * 3;

    int ti[TILES], tj[TILES];
    bool on[TILES];
    double acc[TILES][4][4];
#pragma unroll
    for (int t = 0; t < TILES; t++) {
        int idx = threadIdx.x + t * kPbThreads;
        on[t] = idx < ntiles;
        tri_index(on[t] ? idx : 0, ti[t], tj[t]);
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[t][r][q] = 0.0;
    }
    double bacc = 0.0;

    for (int base = 0; base < o.n; base += kPbObs) {
        int nobs = min(kPbObs, o.n - base);
        // stage A rows of this chunk: A[3 o + r][j] = sum_d F[o][r][d] Q[3 vid + d][j]
        for (int e = threadIdx.x; e < kPbObs * Kp; e += kPbThreads) {
            int ob = e / Kp, j = e % Kp;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0;
            if (ob < nobs) {
                int v = vid[base + ob];
                if (v >= 0) {
                    const double *f = F + (size_t)(base + ob) * 9;
                    const double *q = m.Q + (size_t)3 * v * Kp + j;
                    double q0 = __ldg(q), q1 = __ldg(q + Kp), q2 = __ldg(q + 2 * Kp);
                    a0 = f[0] * q0 + f[1] * q1 + f[2] * q2;
                    a1 = f[3] * q0 + f[4] * q1 + f[5] * q2;
                    a2 = f[6] * q0 + f[7] * q1 + f[8] * q2;
                }
            }
            sA[(3 * ob) * Kp + j] = a0;
            sA[(3 * ob + 1) * Kp + j] = a1;
            sA[(3 * ob + 2) * Kp + j] = a2;
        }
        if (threadIdx.x < 3 * kPbObs) {
            int ob = threadIdx.x / 3;
            sy[threadIdx.x] = (ob < nobs && vid[base + ob] >= 0) ? y[(size_t)(base + ob) * 3 + threadIdx.x % 3] : 0.0;
        }
        __syncthreads();
        const int rows = 3 * kPbObs;
#pragma unroll
        for (int t = 0; t < TILES; t++) {
            if (!on[t]) continue;
            const double *pa = sA + 4 * ti[t], *pb = sA + 4 * tj[t];
#pragma unroll 4
            for (int r = 0; r < rows; r++) {
                double2 a01 = *reinterpret_cast<const double2 *>(pa + r * Kp), a23 = *reinterpret_cast<const double2 *>(pa + r * Kp + 2);
                double2 b01 = *reinterpret_cast<const double2 *>(pb + r * Kp), b23 = *reinterpret_cast<const double2 *>(pb + r * Kp + 2);
                double av[4] = {a01.x, a01.y, a23.x, a23.y}, bv[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
                for (int p = 0; p < 4; p++)
#pragma unroll
                    for (int q = 0; q < 4; q++) acc[t][p][q] = fma(av[p], bv[q], acc[t][p][q]);
            }
        }
        if (threadIdx.x < Kp) {
            for (int r = 0; r < rows; r++) bacc = fma(sA[r * Kp + threadIdx.x], sy[r], bacc);
        }
        __syncthreads();
    }
    double *Mc = M + (size_t)c * Kp * Kp;
#pragma unroll
    for (int t = 0; t < TILES; t++) {
        if (!on[t]) continue;
#pragma unroll
        for (int p = 0; p < 4; p++)
#pragma unroll
            for (int q = 0; q < 4; q++) {
                int i = 4 * ti[t] + p, j = 4 * tj[t] + q;
                double v = acc[t][p][q] + (i == j ? 1.0 : 0.0);
                Mc[(size_t)i * Kp + j] = v;
                if (ti[t] != tj[t]) Mc[(size_t)j * Kp + i] = v;
            }
    }
    if (threadIdx.x < Kp) bvec[(size_t)c * Kp + threadIdx.x] = bacc;
}


// ---- tensor-pipe version: mma.sync.m8n8k4.f64 (DMMA) ----------------------------------------------------
// M (Kp x Kp) is cut into 8 x 8 blocks; only the NB (NB + 1) / 2 blocks of the lower triangle are computed.
// They are numbered row-major and dealt out in contiguous runs to the warps of the CTA; each warp keeps its
// blocks as DMMA accumulator fragments in registers for the whole pass over the observations. One staged
// chunk = 8 observations = 24 rows of A = 6 k4-steps. For a block (bi, bj) and a k4-step the A- and
// B-operand fragments are the SAME access pattern into the staged rows (element [k][8 b + i] for lane
// (i = lane / 4, k = lane % 4)), so a fragment loaded for column block b serves as A operand of block row b
// and as B operand of block column b. Row stride Kp + 4 makes the fragment loads bank-conflict free.
// dmma_8x8x4: icp_device.cuh

constexpr int kMmaRows = 3 * kPbObs;  // 24 staged rows = 6 k4-steps
constexpr int kProdWarps = 2;         // producer warps (stage A = F Q into shared memory, accumulate b)
constexpr int kMaxNB = 28;         // largest supported Kp / 8 (K <= 224: the packed factorisation must fit shared memory)
constexpr int kMaxStagedIds = 4096;  // observation ids staged in shared memory by the producers

__device__ __forceinline__ void cp_async_16(void *smem_dst, const void *gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_16_ca(void *smem_dst, const void *gsrc) {   // allocates in L1
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_8(void *smem_dst, const void *gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int kRawStages = 2;         // producer ring: passes of raw basis rows in flight per thread

template <int ID>
__device__ __forceinline__ void named_bar_sync(int n) { asm volatile("bar.sync %0, %1;" ::"n"(ID), "r"(n) : "memory"); }
template <int ID>
__device__ __forceinline__ void named_bar_arrive(int n) { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "r"(n) : "memory"); }

// Warp-specialised: warps [0, nwc) are MMA consumers, the last kProdWarps warps are producers. Two staged
// buffers; named barriers FULL(1 + buf) / EMPTY(3 + buf) hand them back and forth, so the gather of the
// basis rows (L2 latency) and the 3 x 3 whitening overlap with the DMMA stream of the previous chunk.
// RPO = rows of A per observation. RPO = 3: the general whitened rows F_i Q_i. RPO = 1 (constant-Gram fast path,
// model sampling with every observation kept and sd_n <= sd_t): Sigma_i^-1 = I / sd_t^2 + kappa n n^T with
// kappa = 1/sd_n^2 - 1/sd_t^2, so M = I + Gs / sd_t^2 + sum_i (sqrt(kappa) Q_i^T n_i)(...)^T where
// Gs = sum_i Q_i^T Q_i is a constant of the proposal: one row per observation, a third of the DMMA work.
template <int NBLK, int NBMAX, int NWC, int RPO>
__global__ void __launch_bounds__((NWC + kProdWarps) * 32) k_posterior_build_mma(ModelDev m, ObsDev o,
                                                                                 double *__restrict__ M,
                                                                                 double *__restrict__ bvec,
                                                                                 int nblk_total,
                                                                                 const double *__restrict__ Gs,
                                                                                 double gs_scale, double row_scale) {
    extern __shared__ double sm[];
    const int Kp = m.Kp, ld = Kp + 4, NB = Kp >> 3;
    const int bufsz = kMmaRows * ld;
    double *sA = sm;                    // [2][24][ld]
    const int c = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int nthreads = (NWC + kProdWarps) * 32, nwc = NWC;
    constexpr int kObsChunk = kMmaRows / RPO;   // observations per staged chunk (8 or 24)
    const int nrows = o.nrows ? o.nrows[c] : o.n;   // slots in use (uniform over the CTA)
    const int nchunks = (nrows + kObsChunk - 1) / kObsChunk;
    if (warp < nwc) {
        // ------------------------------- consumers: DMMA ------------------------------------------------
        const int per = (nblk_total + nwc - 1) / nwc;
        const int b0 = warp * per;
        const int nmine = max(0, min(nblk_total, b0 + per) - b0);
        int bi0, bj0;
        tri_index(b0 < nblk_total ? b0 : 0, bi0, bj0);
        double acc[NBLK][2];
#pragma unroll
        for (int s = 0; s < NBLK; s++) acc[s][0] = acc[s][1] = 0.0;
        const int frag = (lane & 3) * ld + (lane >> 2);
        named_bar_arrive<3>(nthreads);  // both buffers start empty
        named_bar_arrive<4>(nthreads);
        for (int ch = 0; ch < nchunks; ch++) {
            const int buf = ch & 1;
            if (buf == 0) named_bar_sync<1>(nthreads); else named_bar_sync<2>(nthreads);
            const double *base = sA + buf * bufsz + frag;
            int bi = bi0, bj = bj0;
            double fa[6];
#pragma unroll
            for (int k = 0; k < 6; k++) fa[k] = base[k * 4 * ld + 8 * bi];
            // blocks are taken two at a time when both lie in the same block row (same A fragment): their DMMAs are
            // interleaved so that consecutive DMMAs never accumulate into the same registers
#pragma unroll
            for (int s = 0; s < NBLK; s += 2) {
                if (s + 1 < NBLK && s + 1 < nmine && bj + 1 <= bi) {
#pragma unroll
                    for (int half = 0; half < 2; half++) {
                        double f0[3], f1[3];
#pragma unroll
                        for (int k = 0; k < 3; k++) {
                            f0[k] = base[(3 * half + k) * 4 * ld + 8 * bj];
                            f1[k] = base[(3 * half + k) * 4 * ld + 8 * bj + 8];
                        }
#pragma unroll
                        for (int k = 0; k < 3; k++) {
                            dmma_8x8x4(acc[s][0], acc[s][1], fa[3 * half + k], f0[k]);
                            dmma_8x8x4(acc[s + 1 < NBLK ? s + 1 : s][0], acc[s + 1 < NBLK ? s + 1 : s][1], fa[3 * half + k], f1[k]);
                        }
                    }
                    bj += 2;
                    if (bj > bi) {
                        bj = 0;
                        if (++bi < NB) {
#pragma unroll
                            for (int k = 0; k < 6; k++) fa[k] = base[k * 4 * ld + 8 * bi];
                        }
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        if (s + u < NBLK && s + u < nmine) {
                            double fb[6];
#pragma unroll
                            for (int k = 0; k < 6; k++) fb[k] = base[k * 4 * ld + 8 * bj];
#pragma unroll
                            for (int k = 0; k < 6; k++) dmma_8x8x4(acc[s + u < NBLK ? s + u : s][0], acc[s + u < NBLK ? s + u : s][1], fa[k], fb[k]);
                            if (++bj > bi) {
                                bj = 0;
                                if (++bi < NB) {
#pragma unroll
                                    for (int k = 0; k < 6; k++) fa[k] = base[k * 4 * ld + 8 * bi];
                                }
                            }
                        }
                    }
                }
            }
            if (buf == 0) named_bar_arrive<3>(nthreads); else named_bar_arrive<4>(nthreads);
        }
        double *Mc = M + (size_t)c * Kp * Kp;
        int bi = bi0, bj = bj0;
#pragma unroll
        for (int s = 0; s < NBLK; s++) {
            if (s < nmine) {
                int i = 8 * bi + (lane >> 2), j = 8 * bj + 2 * (lane & 3);
                double v0 = acc[s][0] + (i == j ? 1.0 : 0.0), v1 = acc[s][1] + (i == j + 1 ? 1.0 : 0.0);
                if (RPO == 1) {
                    double2 g = __ldg(reinterpret_cast<const double2 *>(Gs + (size_t)i * Kp + j));
                    v0 = fma(g.x, gs_scale, v0);
                    v1 = fma(g.y, gs_scale, v1);
                }
                *reinterpret_cast<double2 *>(Mc + (size_t)i * Kp + j) = make_double2(v0, v1);
                if (bi != bj) {
                    Mc[(size_t)j * Kp + i] = v0;
                    Mc[(size_t)(j + 1) * Kp + i] = v1;
                }
                if (++bj > bi) { bj = 0; ++bi; }
            }
        }
    } else {
        // ------------------------------- producers: gather + whiten ----------------------------------------
        const int pt = tid - nwc * 32;          // 0 .. 63
        const int ob = pt >> 3, cg = pt & 7;     // observation slot within the chunk, column group
        const int *vid = o.vid + (size_t)c * o.n;
        const double *F = o.F + (size_t)c * o.n * 9;
        const double *y = o.y + (size_t)c * o.n * 3;
        double bacc[NBMAX];
#pragma unroll
        for (int i = 0; i < NBMAX; i++) bacc[i] = 0.0;
        // the vertex ids gate the addresses of every basis-row load: stage them in shared memory once so that a
        // pass pays one L2 round trip (ids -> rows would be two dependent ones)
        int *svid = reinterpret_cast<int *>(sm + 2 * bufsz + 8 * Kp);
        const bool vid_staged = o.n <= kMaxStagedIds;
        if (vid_staged) {
            for (int e = pt; e < nrows; e += kProdWarps * 32) svid[e] = __ldg(&vid[e]);
            named_bar_sync<5>(kProdWarps * 32);
        }
        for (int ch = 0; ch < nchunks; ch++) {
            const int buf = ch & 1;
#pragma unroll 1
            for (int pass = 0; pass < kObsChunk / 8; pass++) {
                const int lo = pass * 8 + ob;            // observation slot within the chunk
                const int gi = ch * kObsChunk + lo;
                int v = -1;
                double f[9], yy[3];
                if (gi < nrows) v = vid_staged ? svid[gi] : __ldg(&vid[gi]);
                if (v >= 0) {
#pragma unroll
                    for (int k = 0; k < 9; k++) f[k] = __ldg(F + (size_t)gi * 9 + k);
#pragma unroll
                    for (int k = 0; k < 3; k++) yy[k] = __ldg(y + (size_t)gi * 3 + k);
                } else {
#pragma unroll
                    for (int k = 0; k < 9; k++) f[k] = 0.0;
                    yy[0] = yy[1] = yy[2] = 0.0;
                }
                const double *q = m.Q + (size_t)3 * (v >= 0 ? v : 0) * Kp + cg;
                double *dst = sA + buf * bufsz + (RPO * lo) * ld + cg;
                // column blocks in chunks of kCH: the large-rank instantiation must not hold 3 x 28 basis entries at once
                constexpr int kCH = NBMAX > 14 ? 7 : NBMAX;
#pragma unroll
                for (int h0 = 0; h0 < NBMAX; h0 += kCH) {
                    double q0[kCH], q1[kCH], q2[kCH];
#pragma unroll
                    for (int u = 0; u < kCH; u++) {
                        const int i = h0 + u;
                        if (i < NBMAX && i < NB) { q0[u] = __ldg(q + 8 * i); q1[u] = __ldg(q + Kp + 8 * i); q2[u] = __ldg(q + 2 * Kp + 8 * i); }
                    }
                    if (pass == 0 && h0 == 0) {  // consumers are done with this buffer
                        if (buf == 0) named_bar_sync<3>(nthreads); else named_bar_sync<4>(nthreads);
                    }
#pragma unroll
                    for (int u = 0; u < kCH; u++) {
                        const int i = h0 + u;
                        if (i < NBMAX && i < NB) {
                            double a0 = f[0] * q0[u] + f[1] * q1[u] + f[2] * q2[u];
                            double a1 = f[3] * q0[u] + f[4] * q1[u] + f[5] * q2[u];
                            double a2 = f[6] * q0[u] + f[7] * q1[u] + f[8] * q2[u];
                            if (RPO == 3) { dst[8 * i] = a0; dst[ld + 8 * i] = a1; dst[2 * ld + 8 * i] = a2; }
                            else dst[8 * i] = a0 * row_scale;
                            bacc[i] = fma(a0, yy[0], fma(a1, yy[1], fma(a2, yy[2], bacc[i])));
                        }
                    }
                }
            }
            if (buf == 0) named_bar_arrive<1>(nthreads); else named_bar_arrive<2>(nthreads);
        }
        // reduce b over the 8 observation slots (fixed order: deterministic)
        named_bar_sync<5>(kProdWarps * 32);      // producers only
        // the last two buffers may still be read by consumers: use the tail of the shared allocation
        double *sb = sm + 2 * bufsz;             // [8][Kp]
#pragma unroll
        for (int i = 0; i < NBMAX; i++)
            if (i < NB) sb[ob * Kp + cg + 8 * i] = bacc[i];
        named_bar_sync<5>(kProdWarps * 32);
        for (int j = pt; j < Kp; j += kProdWarps * 32) {
            double t = 0.0;
#pragma unroll
            for (int r = 0; r < 8; r++) t += sb[r * Kp + j];
            bvec[(size_t)c * Kp + j] = t;
        }
    }
}

template <int NBLK, int NBMAX, int NWC>
static void launch_pb_mma(const ModelDev &m, int C, const ObsDev &o, double *d_M, double *d_b, int total, const GramFast *gf,
                          cudaStream_t s) {
    size_t smem = sizeof(double) * ((size_t)2 * kMmaRows * (m.Kp + 4) + 8 * m.Kp) + sizeof(int) * (size_t)std::min(o.n, kMaxStagedIds);
    if (gf) {
        ICP_CUDA(cudaFuncSetAttribute(k_posterior_build_mma<NBLK, NBMAX, NWC, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_posterior_build_mma<NBLK, NBMAX, NWC, 1><<<C, (NWC + kProdWarps) * 32, smem, s>>>(m, o, d_M, d_b, total, gf->Gs, gf->gs_scale, gf->row_scale);
    } else {
        ICP_CUDA(cudaFuncSetAttribute(k_posterior_build_mma<NBLK, NBMAX, NWC, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_posterior_build_mma<NBLK, NBMAX, NWC, 3><<<C, (NWC + kProdWarps) * 32, smem, s>>>(m, o, d_M, d_b, total, nullptr, 0.0, 1.0);
    }
}

void launch_posterior_build(const ModelDev &m, int C, const ObsDev &o, double *d_M, double *d_b, cudaStream_t s, const GramFast *gf) {
    ProfScope _ps(ST_POSTERIOR_BUILD, s);
    if (C <= 0) return;
    static const bool no_mma = getenv("ICPCUDA_NO_DMMA") && getenv("ICPCUDA_NO_DMMA")[0] == '1';
    {
        int NB = m.Kp / 8, total = NB * (NB + 1) / 2;
        if (!no_mma && NB <= kMaxNB) {
            if (NB <= 4) launch_pb_mma<4, 4, 4>(m, C, o, d_M, d_b, total, gf, s);
            else if (NB <= 7) launch_pb_mma<8, 7, 4>(m, C, o, d_M, d_b, total, gf, s);
            else if (NB <= 13) launch_pb_mma<24, 13, 4>(m, C, o, d_M, d_b, total, gf, s);
            else if (NB <= 20) launch_pb_mma<28, 20, 8>(m, C, o, d_M, d_b, total, gf, s);
            else launch_pb_mma<36, 28, 12>(m, C, o, d_M, d_b, total, gf, s);
            ICP_CUDA(cudaGetLastError());
            return;
        }
    }
    int nt = m.Kp / 4, ntiles = nt * (nt + 1) / 2;
    size_t smem = sizeof(double) * ((size_t)3 * kPbObs * m.Kp + 3 * kPbObs);
    ICP_REQUIRE(m.Kp <= kPbThreads, "rank too large for the posterior build kernel (K <= 256)");
    int tiles = (ntiles + kPbThreads - 1) / kPbThreads;
    if (tiles <= 1) k_posterior_build<1><<<C, kPbThreads, smem, s>>>(m, o, d_M, d_b);
    else if (tiles <= 2) k_posterior_build<2><<<C, kPbThreads, smem, s>>>(m, o, d_M, d_b);
    else if (tiles <= 4) k_posterior_build<4><<<C, kPbThreads, smem, s>>>(m, o, d_M, d_b);
    else if (tiles <= 8) k_posterior_build<8><<<C, kPbThreads, smem, s>>>(m, o, d_M, d_b);
    else throw ArgError{"rank too large for the posterior build kernel"};
    ICP_CUDA(cudaGetLastError());
}

// Gs[i][j] = sum over the proposal's model points p and d < 3 of Q[3 p + d][i] Q[3 p + d][j] (one-off per proposal)
__global__ void k_gram_rows(int n_ids, const int *__restrict__ ids, int Kp, const double *__restrict__ Q, double *__restrict__ G) {
    int i = blockIdx.x, j = threadIdx.x;
    if (j >= Kp) return;
    double acc = 0;
    for (int t = 0; t < n_ids; t++) {
        const double *q = Q + (size_t)3 * ids[t] * Kp;
        for (int d = 0; d < 3; d++) acc = fma(q[d * Kp + i], q[d * Kp + j], acc);
    }
    G[(size_t)i * Kp + j] = acc;
}

void launch_gram_rows(const ModelDev &m, int n_ids, const int *d_ids, double *d_G, cudaStream_t s) {
    k_gram_rows<<<m.Kp, ((m.Kp + 31) / 32) * 32, 0, s>>>(n_ids, d_ids, m.Kp, m.Q, d_G);
    ICP_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------
// Cholesky M = L L^T with the right-hand side carried as an extra row (forward solve for free),
// then back substitution L^T mu = y. One CTA per matrix, matrix resident in shared memory.
// ---------------------------------------------------------------------------------------------------
constexpr int kChThreads = 256;

__global__ void __launch_bounds__(kChThreads) k_cholesky_solve(int K, int Kp, const double *__restrict__ M,
                                                               const double *__restrict__ bvec, double *__restrict__ L,
                                                               double *__restrict__ mu, const int *__restrict__ out_slot,
                                                               int *__restrict__ status) {
    extern __shared__ double sm[];
    const int ld = Kp + 1;        // odd stride: column accesses are bank-conflict free
    double *A = sm;               // [Kp + 1][ld]: rows 0..Kp-1 lower triangle of M, row Kp = b
    double *x = sm + (size_t)(Kp + 1) * ld;  // [Kp] solution
    __shared__ int bad;
    int c = blockIdx.x;
    const double *Mc = M + (size_t)c * Kp * Kp;
    if (threadIdx.x == 0) bad = 0;
    for (int e = threadIdx.x; e < Kp * Kp; e += kChThreads) {
        int i = e / Kp, j = e % Kp;
        A[i * ld + j] = Mc[e];
    }
    for (int j = threadIdx.x; j < Kp; j += kChThreads) A[Kp * ld + j] = bvec[(size_t)c * Kp + j];
    __syncthreads();
    const int R = Kp + 1;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    for (int j = 0; j < Kp; j++) {
        double ajj = A[j * ld + j];
        if (!(ajj > 0.0 && ajj < INFINITY)) { if (threadIdx.x == 0) bad = 1; }   // an infinite pivot only yields NaN
        double inv = 1.0 / sqrt(ajj);
        __syncthreads();  // everyone has read the pivot before it is overwritten
        for (int i = j + threadIdx.x; i < R; i += kChThreads) A[i * ld + j] *= inv;  // i == j: a/sqrt(a) = sqrt(a)
        __syncthreads();
        // trailing update of the lower triangle (and of the b row)
        for (int i = j + 1 + ty; i < R; i += 16) {
            double lij = A[i * ld + j];
            int kmax = i < Kp ? i : Kp - 1;
            for (int k = j + 1 + tx; k <= kmax; k += 16) A[i * ld + k] = fma(-lij, A[k * ld + j], A[i * ld + k]);
        }
        __syncthreads();
    }
    // A row Kp now holds y = L^-1 b. Back substitution L^T x = y, column oriented.
    for (int j = threadIdx.x; j < Kp; j += kChThreads) x[j] = A[Kp * ld + j];
    __syncthreads();
    for (int i = Kp - 1; i >= 0; i--) {
        double xi = x[i] / A[i * ld + i];
        __syncthreads();
        if (threadIdx.x == 0) x[i] = xi;
        for (int k = threadIdx.x; k < i; k += kChThreads) x[k] = fma(-A[i * ld + k], xi, x[k]);
        __syncthreads();
    }
    int oc = out_slot ? out_slot[c] : c;
    double *Lc = L + (size_t)oc * Kp * Kp;
    bool isbad = bad != 0;
    for (int e = threadIdx.x; e < Kp * Kp; e += kChThreads) {
        int i = e / Kp, j = e % Kp;
        double v = j <= i ? A[i * ld + j] : 0.0;
        Lc[e] = isbad ? NAN : v;
    }
    for (int j = threadIdx.x; j < Kp; j += kChThreads) mu[(size_t)oc * Kp + j] = isbad ? NAN : x[j];
    if (threadIdx.x == 0 && status) status[c] = isbad ? 1 : 0;
    (void)K;
}


// ---- blocked left-looking Cholesky with DMMA updates --------------------------------------------------------
// 8 x 8 blocks; the right-hand side b rides along as block row NB (row Kp real, 7 zero rows), so that after
// the factorisation it holds y = L^-1 b. Per block column bj:
//   (1) every block (bi >= bj, bj) -= sum_{p < bj} L(bi, p) L(bj, p)^T      DMMA m8n8k4, blocks dealt to the warps
//   (2) every thread factors the 8 x 8 diagonal block redundantly in registers (no warp / block hand-offs on
//       the sqrt -> reciprocal chain) and solves its own row(s) of the panel against it.
// Back substitution L^T x = y runs 8 unknowns at a time the same way.
constexpr int kCh2Threads = 128;

#ifdef ICP_FUSED_TIMING
// experiment build only (ICPCUDA_LIB_TAG=timing ICPCUDA_NVCC_EXTRA=-DICP_FUSED_TIMING, tools/fused_timing.py):
// per-CTA clock64() phase times
constexpr int kFtStride = 12;
__device__ long long g_ft[kFtStride * 8192];
#define ICP_FT(...) __VA_ARGS__
#else
#define ICP_FT(...)
#endif

// Factorises the matrix staged in shared memory (A: [Kp + 8][Kp + 4], lower triangle of M in rows 0..Kp-1, b in row Kp,
// rows Kp+1..Kp+7 zero), solves M mu = b and stores L (lower triangle only) and mu. Every one of the NT threads of the CTA
// must call it (it synchronises the CTA); *bad (shared) must have been cleared before the preceding barrier.
// ymean: store y = L^-1 b (the chain runner's mean slot) instead of mu, and skip the back substitution.
template <int NT>
__device__ void chol_factor_solve_store(double *A, int Kp, int *bad, double *__restrict__ Lc, double *__restrict__ muc,
                                        int *__restrict__ status, bool ymean) {
    const int ld = Kp + 4, NB = Kp >> 3, R = Kp + 8;
    double *dinv = A + (size_t)R * ld;      // [Kp] reciprocals of the diagonal of L
    double *xs = dinv + Kp;                 // [Kp] running right-hand side of the back substitution
    double *xo = xs + Kp;                   // [Kp] solution
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int fr = lane >> 2, fc = lane & 3;
    ICP_FT(const long long ftc0 = clock64();)
    for (int bj = 0; bj < NB; bj++) {
        if (bj > 0) {
            for (int bi = bj + warp; bi <= NB; bi += NT / 32) {
                double *pc = A + (8 * bi + fr) * ld + 8 * bj + 2 * fc;
                double2 cc = *reinterpret_cast<double2 *>(pc);
                const double *pa = A + (8 * bi + fr) * ld + fc;
                const double *pb = A + (8 * bj + fr) * ld + fc;
                // two accumulators halve the dependent DMMA chain
                double e0 = 0.0, e1 = 0.0;
#pragma unroll 4
                for (int k = 0; k < 8 * bj; k += 8) {
                    dmma_8x8x4(cc.x, cc.y, -pa[k], pb[k]);
                    dmma_8x8x4(e0, e1, -pa[k + 4], pb[k + 4]);
                }
                cc.x += e0; cc.y += e1;
                *reinterpret_cast<double2 *>(pc) = cc;
            }
            __syncthreads();
        }
        // diagonal block, factored redundantly by every thread
        double l[8][8], inv[8];
        const double *D = A + (8 * bj) * ld + 8 * bj;
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int k = 0; k <= i; k++) l[i][k] = D[i * ld + k];
        __syncthreads();
        bool mybad = false;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            double s = l[j][j];
            // 1/sqrt(s) by rsqrt + one Newton step (full double accuracy), sqrt(s) = s * inv: one short dependent
            // chain instead of a software sqrt followed by a software divide
            double r = rsqrt(s);
            r = fma(r * 0.5, fma(-s * r, r, 1.0), r);
            // r > 0 exactly for finite s > 0: s <= 0 and NaN give NaN, and so does s = +Inf (rsqrt 0, the Newton step
            // 0 * Inf), which a test of s > 0 lets through - with no later pivot to catch it when it is the last one
            if (!(r > 0.0)) mybad = true;
            inv[j] = r;
            double d = s * r;
            d = fma(fma(-d, d, s), 0.5 * r, d);
            l[j][j] = d;
#pragma unroll
            for (int i = j + 1; i < 8; i++) l[i][j] *= inv[j];
#pragma unroll
            for (int i = j + 1; i < 8; i++)
#pragma unroll
                for (int k = j + 1; k <= i; k++) l[i][k] = fma(-l[i][j], l[k][j], l[i][k]);
        }
        if (mybad && tid == 0) *bad = 1;
        if (tid < 8) {
            dinv[8 * bj + tid] = inv[tid];
#pragma unroll
            for (int i = 0; i < 8; i++)
                if (i == tid) {
#pragma unroll
                    for (int k = 0; k < 8; k++) A[(8 * bj + i) * ld + 8 * bj + k] = k <= i ? l[i][k] : 0.0;
                }
        }
        for (int r = 8 * bj + 8 + tid; r < R; r += NT) {
            double *row = A + r * ld + 8 * bj;
            double x[8];
#pragma unroll
            for (int j = 0; j < 8; j++) x[j] = row[j];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                double t = x[j];
#pragma unroll
                for (int k = 0; k < j; k++) t = fma(-x[k], l[j][k], t);
                x[j] = t * inv[j];
            }
#pragma unroll
            for (int j = 0; j < 8; j++) row[j] = x[j];
        }
        __syncthreads();
    }
    // back substitution L^T x = y (y = row Kp of A)
    ICP_FT(const long long ftc1 = clock64();)
    for (int k = tid; k < Kp; k += NT) xs[k] = A[Kp * ld + k];
    __syncthreads();
    for (int bj = ymean ? -1 : NB - 1; bj >= 0; bj--) {   // ymean: xs already holds what is stored, no step runs
        const double *D = A + (8 * bj) * ld + 8 * bj;
        double x[8];
#pragma unroll
        for (int i = 7; i >= 0; i--) {
            double t = xs[8 * bj + i];
#pragma unroll
            for (int k = i + 1; k < 8; k++) t = fma(-D[k * ld + i], x[k], t);
            x[i] = t * dinv[8 * bj + i];
        }
        if (tid < 8) {
#pragma unroll
            for (int i = 0; i < 8; i++)
                if (i == tid) xo[8 * bj + i] = x[i];
        }
        for (int k = tid; k < 8 * bj; k += NT) {
            double t = xs[k];
#pragma unroll
            for (int p = 0; p < 8; p++) t = fma(-A[(8 * bj + p) * ld + k], x[p], t);
            xs[k] = t;
        }
        __syncthreads();
    }
    ICP_FT(if (tid == 0 && blockIdx.x < 8192) {
        g_ft[kFtStride * blockIdx.x + 8] = ftc1 - ftc0; g_ft[kFtStride * blockIdx.x + 9] = clock64() - ftc1;
    })
    bool isbad = *bad != 0;
    for (int e = tid; e < Kp * Kp; e += NT) {
        int i = e / Kp, j = e - i * Kp;
        if (j <= i) __stcs(Lc + e, isbad ? NAN : A[i * ld + j]);   // only the lower triangle is ever read; streaming stores
    }
    for (int j = tid; j < Kp; j += NT) __stcs(muc + j, isbad ? NAN : ymean ? xs[j] : xo[j]);
    if (tid == 0 && status) *status = isbad ? 1 : 0;
}

__global__ void __launch_bounds__(kCh2Threads) k_cholesky_solve_mma(int K, int Kp, const double *__restrict__ M,
                                                                     const double *__restrict__ bvec,
                                                                     double *__restrict__ L, double *__restrict__ mu,
                                                                     const int *__restrict__ out_slot,
                                                                     int *__restrict__ status, bool ymean) {
    extern __shared__ double sm[];
    const int ld = Kp + 4, NB = Kp >> 3, R = Kp + 8;
    double *A = sm;                         // [R][ld]
    double *dinv = A + (size_t)R * ld;      // [Kp] reciprocals of the diagonal of L
    double *xs = dinv + Kp;                 // [Kp] running right-hand side of the back substitution
    double *xo = xs + Kp;                   // [Kp] solution
    __shared__ int bad;
    const int c = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double *Mc = M + (size_t)c * Kp * Kp;
    if (tid == 0) bad = 0;
    // lower triangle only; warps take rows, lanes take column pairs, 16 independent 16-byte loads in flight per
    // thread (a dependent load -> store loop costs one L2 round trip per element)
    {
        constexpr int nw = kCh2Threads / 32;
        for (int i0 = warp; i0 < Kp; i0 += 4 * nw) {
            double2 v[4][4];
#pragma unroll
            for (int r = 0; r < 4; r++) {
                int i = i0 + r * nw;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    int j = 2 * (lane + 32 * q);
                    v[r][q] = (i < Kp && j <= i) ? __ldg(reinterpret_cast<const double2 *>(Mc + (size_t)i * Kp + j)) : make_double2(0.0, 0.0);
                }
            }
#pragma unroll
            for (int r = 0; r < 4; r++) {
                int i = i0 + r * nw;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    int j = 2 * (lane + 32 * q);
                    if (i < Kp && j <= i) *reinterpret_cast<double2 *>(A + i * ld + j) = v[r][q];
                }
            }
        }
    }
    for (int e = tid; e < 8 * ld; e += kCh2Threads) {
        int r = e / ld, j = e - r * ld;
        A[(Kp + r) * ld + j] = (r == 0 && j < Kp) ? bvec[(size_t)c * Kp + j] : 0.0;
    }
    __syncthreads();
    int oc = out_slot ? out_slot[c] : c;
    chol_factor_solve_store<kCh2Threads>(A, Kp, &bad, L + (size_t)oc * Kp * Kp, mu + (size_t)oc * Kp, status ? status + c : nullptr, ymean);
    (void)K;
}

// ---- consumer roles for Kp = 104 (13 block rows): rectangular / triangular block sets per warp -----------------------
// Block indices are split into groups A = 0..4, B = 5..8, C = 9..12. The lower triangle then is
//   tri(A) 15 + tri(B) 10 + tri(C) 10 + rect(B x A) 20 + rect(C x A) 20 + rect(C x B) 16 = 91 blocks,
// dealt as  warp 0: B x A (20) | warp 1: C x A (20) | warp 2: C x B + tri(B) (26) | warp 3: tri(A) + tri(C) (25).
// Within a rectangle every row fragment is reused by all its columns and vice versa, and in a triangle the row and
// column fragments coincide: 35 shared-memory fragment loads per k4-step for the 91 DMMAs (the run-length assignment of
// the generic path needs ~100), which takes the shared-memory pipe off the critical path of the tensor pipe.
template <int RB, int CB>
__device__ __forceinline__ void mma_rect_chunk(double (&acc)[RB * CB][2], const double *base, int ld, int r0, int c0) {
#pragma unroll
    for (int k = 0; k < kMmaRows / 4; k++) {
        double fr[RB], fc[CB];
#pragma unroll
        for (int i = 0; i < RB; i++) fr[i] = base[k * 4 * ld + 8 * (r0 + i)];
#pragma unroll
        for (int j = 0; j < CB; j++) fc[j] = base[k * 4 * ld + 8 * (c0 + j)];
#pragma unroll
        for (int i = 0; i < RB; i++)
#pragma unroll
            for (int j = 0; j < CB; j++) dmma_8x8x4(acc[i * CB + j][0], acc[i * CB + j][1], fr[i], fc[j]);
    }
}
template <int TB>
__device__ __forceinline__ void mma_tri_chunk(double (&acc)[TB * (TB + 1) / 2][2], const double *base, int ld, int r0) {
#pragma unroll
    for (int k = 0; k < kMmaRows / 4; k++) {
        double f[TB];
#pragma unroll
        for (int i = 0; i < TB; i++) f[i] = base[k * 4 * ld + 8 * (r0 + i)];
#pragma unroll
        for (int i = 0; i < TB; i++)
#pragma unroll
            for (int j = 0; j <= i; j++) dmma_8x8x4(acc[i * (i + 1) / 2 + j][0], acc[i * (i + 1) / 2 + j][1], f[i], f[j]);
    }
}
// ---- block-packed Cholesky: four chains per SM ---------------------------------------------------------------------
// The factorisation is a chain of Kp dependent pivots (rsqrt -> scale -> update): latency, not throughput. What hides
// latency is residency, so the matrix is kept block-packed in shared memory - only the NB (NB + 1) / 2 lower-triangle
// 8 x 8 blocks, 64 doubles each, 46.6 KB at Kp = 104 instead of 97 KB for the padded square - and four 128-thread CTAs
// share an SM. Inside a block, column bit 2 is flipped on rows with bit 1 set, which makes the DMMA fragment loads
// (rows lane / 4, columns lane % 4 (+ 4)) conflict free without padding. Same left-looking algorithm as
// chol_factor_solve_store; the right-hand side is a vector and takes part in the DMMA update as a block whose rows
// 1..7 are zero.
__device__ __forceinline__ int pk_swz(int r) { return (r & 2) << 1; }
__device__ __forceinline__ int pk_blk(int bi, int bj) { return ((bi * (bi + 1) >> 1) + bj) * 64; }
__device__ __forceinline__ int pk_at(int i, int j) {   // element (i, j) of a stored block
    const int r = i & 7;
    return pk_blk(i >> 3, j >> 3) + r * 8 + ((j & 7) ^ pk_swz(r));
}

constexpr int kCh3Threads = 128;
// NT threads per matrix: 128 (four matrices per SM) for full batches; 256 when every matrix of the launch is resident anyway
// (a few chains are latency-bound: the load, store and column-update phases get twice the threads; the arithmetic of every
// element - and for Kp <= 128 the association of the final quadratic form - does not depend on NT)
// YMEAN (the chain runner's form): the mean slot receives y = L^-1 b instead of mu = L^-T y, and the backward form is
// |L^T w - y|^2 (= |L^T (w - mu)|^2). The back substitution and its scratch drop out; L and y are the same arithmetic.
template <int NT, bool YMEAN>
__global__ void __launch_bounds__(NT, NT == 128 ? 4 : 2) k_cholesky_packed(int Kp, const double *__restrict__ Mp,
                                                                    const double *__restrict__ bvec, double *__restrict__ M_out,
                                                                    double *__restrict__ L, double *__restrict__ mu,
                                                                    const int *__restrict__ out_slot, int *__restrict__ status,
                                                                    QuadArgs qa, const int *__restrict__ list,
                                                                    const int *__restrict__ count) {
    extern __shared__ __align__(16) double sp[];
    const int NB = Kp >> 3, ntri = NB * (NB + 1) / 2;
    double *A = sp;                  // [ntri][64]
    double *yv = A + ntri * 64;      // [Kp] b, then y = L^-1 b
    double *dinv = yv + Kp;          // [Kp] reciprocals of the diagonal of L
    double *xs = dinv + Kp;          // [Kp] running right-hand side of the back substitution (YMEAN: w of the backward form)
    double *xo = xs + Kp;            // [Kp] solution (mu form only)
    __shared__ int bad;
    // entry ent: M / b of the launch's ent-th matrix; chain c: where its factor, status and form go (list form: entries past the
    // count have nothing to do)
    const int ent = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (count && ent >= *count) return;
    const int c = list ? list[ent] : ent;
    const int fr = lane >> 2, fc = lane & 3, sw = pk_swz(fr);
    {
        ICP_FT(const long long ftl = clock64();)
        const double2 *src = reinterpret_cast<const double2 *>(Mp + (size_t)ent * ntri * 64);
        // 16-byte chunk e: block e / 32, row (e / 4) % 8, columns 2 (e % 4), + 1; 8 independent loads in flight per thread
        for (int e0 = tid; e0 < ntri * 32; e0 += 8 * NT) {
            double2 v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) { const int e = e0 + u * NT; if (e < ntri * 32) v[u] = __ldcs(src + e); }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int e = e0 + u * NT, r = (e >> 2) & 7;
                if (e < ntri * 32) *reinterpret_cast<double2 *>(A + (e >> 5) * 64 + r * 8 + ((2 * (e & 3)) ^ pk_swz(r))) = v[u];
            }
        }
        for (int k = tid; k < Kp; k += NT) yv[k] = __ldcs(bvec + (size_t)ent * Kp + k);
        if (tid == 0) bad = 0;
        ICP_FT(if (tid == 0 && c < 8192) g_ft[kFtStride * c + 8] = clock64() - ftl;)
    }
    __syncthreads();
    ICP_FT(const long long ftf = clock64();)
    if (M_out) {   // only the primitive API (icp_posterior) asks for M
        double *Mc = M_out + (size_t)c * Kp * Kp;
        for (int x = tid; x < Kp * Kp; x += NT) {
            const int i = x / Kp, j = x - i * Kp;
            Mc[x] = j <= i ? A[pk_at(i, j)] : A[pk_at(j, i)];
        }
        __syncthreads();
    }
    ICP_FT(long long fph[5] = {0, 0, 0, 0, 0}; long long ftk = clock64();)
    for (int bj = 0; bj < NB; bj++) {
        // Left-looking update of block column bj and the factorisation of its diagonal block run side by side: warp 0 updates
        // the diagonal block and the right-hand side and goes straight on to the 8 dependent pivots (every lane redundantly,
        // so the rsqrt -> scale chain has no hand-offs), the other warps update the blocks below the diagonal meanwhile.
        // One barrier per phase pair instead of two, and the pivot chain hides behind the DMMA updates.
        double *D = A + pk_blk(bj, bj);
        {
            const double *pb = A + pk_blk(bj, 0) + fr * 8;
            const int o0 = fc ^ sw, o1 = o0 ^ 4;
            const int nwork = NT / 32 - 1;
            // warp 0: bi = bj (the diagonal block, then straight on to its factorisation); warps 1..: bi = bj + warp,
            // bj + warp + nwork, ..; the right-hand side (bi = NB) goes to the last warp, which has the fewest blocks left
            for (int it = 0;; it++) {
                int bi;
                if (warp == 0) { if (it > 0) break; bi = bj; }
                else {
                    bi = bj + warp + it * nwork;
                    if (bi >= NB) { if (warp != NT / 32 - 1 || bi >= NB + nwork) break; bi = NB; }
                }
                if (bj == 0) continue;      // nothing to subtract yet
                double e0 = 0.0, e1 = 0.0;   // two accumulators halve the dependent DMMA chain
                if (bi < NB) {
                    double *pc = A + pk_blk(bi, bj) + fr * 8 + ((2 * fc) ^ sw);
                    double2 cc = *reinterpret_cast<double2 *>(pc);
                    const double *pa = A + pk_blk(bi, 0) + fr * 8;
                    // four independent accumulators: the dependent DMMA chain is a quarter of the 2 bj products
                    double g0 = 0.0, g1 = 0.0, h0 = 0.0, h1 = 0.0;
                    int p = 0;
#pragma unroll 2
                    for (; p + 1 < bj; p += 2) {
                        dmma_8x8x4(cc.x, cc.y, -pa[p * 64 + o0], pb[p * 64 + o0]);
                        dmma_8x8x4(e0, e1, -pa[p * 64 + o1], pb[p * 64 + o1]);
                        dmma_8x8x4(g0, g1, -pa[(p + 1) * 64 + o0], pb[(p + 1) * 64 + o0]);
                        dmma_8x8x4(h0, h1, -pa[(p + 1) * 64 + o1], pb[(p + 1) * 64 + o1]);
                    }
                    if (p < bj) {
                        dmma_8x8x4(cc.x, cc.y, -pa[p * 64 + o0], pb[p * 64 + o0]);
                        dmma_8x8x4(e0, e1, -pa[p * 64 + o1], pb[p * 64 + o1]);
                    }
                    cc.x += (e0 + g0) + h0; cc.y += (e1 + g1) + h1;
                    *reinterpret_cast<double2 *>(pc) = cc;
                } else {   // right-hand side: row 0 of the operand block is y, rows 1..7 are zero
                    double2 cc = make_double2(0.0, 0.0);
                    if (fr == 0) cc = *reinterpret_cast<double2 *>(yv + 8 * bj + 2 * fc);
#pragma unroll 4
                    for (int p = 0; p < bj; p++) {
                        const double a0 = fr == 0 ? -yv[8 * p + fc] : 0.0, a1 = fr == 0 ? -yv[8 * p + fc + 4] : 0.0;
                        dmma_8x8x4(cc.x, cc.y, a0, pb[p * 64 + o0]);
                        dmma_8x8x4(e0, e1, a1, pb[p * 64 + o1]);
                    }
                    if (fr == 0) *reinterpret_cast<double2 *>(yv + 8 * bj + 2 * fc) = make_double2(cc.x + e0, cc.y + e1);
                }
            }
        }
        ICP_FT({ const long long n_ = clock64(); fph[0] += n_ - ftk; ftk = n_; })
        if (warp == 0) {
            __syncwarp();
            double l[8][8], inv[8];
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int k = 0; k <= i; k++) l[i][k] = D[i * 8 + (k ^ pk_swz(i))];
            __syncwarp();
            bool mybad = false;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                double s = l[j][j];
                // 1/sqrt(s) by rsqrt + one Newton step (full double accuracy), sqrt(s) = s * inv
                double r = rsqrt(s);
                r = fma(r * 0.5, fma(-s * r, r, 1.0), r);
                if (!(r > 0.0)) mybad = true;   // finite s > 0 only: +Inf gives NaN here (see chol_factor_solve_store)
                inv[j] = r;
                double d = s * r;
                d = fma(fma(-d, d, s), 0.5 * r, d);
                l[j][j] = d;
#pragma unroll
                for (int i = j + 1; i < 8; i++) l[i][j] *= inv[j];
#pragma unroll
                for (int i = j + 1; i < 8; i++)
#pragma unroll
                    for (int k = j + 1; k <= i; k++) l[i][k] = fma(-l[i][j], l[k][j], l[i][k]);
            }
            if (mybad && lane == 0) bad = 1;
            if (lane < 8) {
                dinv[8 * bj + lane] = inv[lane];
#pragma unroll
                for (int i = 0; i < 8; i++)
                    if (i == lane) {
#pragma unroll
                        for (int k = 0; k < 8; k++) D[i * 8 + (k ^ pk_swz(i))] = k <= i ? l[i][k] : 0.0;
                    }
            }
        }
        ICP_FT({ const long long n_ = clock64(); fph[1] += n_ - ftk; ftk = n_; })
        __syncthreads();
        ICP_FT({ const long long n_ = clock64(); fph[2] += n_ - ftk; ftk = n_; })
        if (8 * bj + 8 + tid <= Kp) {   // panel rows (one per thread); r == Kp is the right-hand side
            double l[8][8], inv[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                inv[j] = dinv[8 * bj + j];
#pragma unroll
                for (int k = 0; k < j; k++) l[j][k] = D[j * 8 + (k ^ pk_swz(j))];
            }
            for (int r = 8 * bj + 8 + tid; r <= Kp; r += NT) {
                double x[8];
                double *row = r < Kp ? A + pk_blk(r >> 3, bj) + (r & 7) * 8 : yv + 8 * bj;
                const int rs = r < Kp ? pk_swz(r & 7) : 0;
#pragma unroll
                for (int j = 0; j < 8; j++) x[j] = row[j ^ rs];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    double t = x[j];
#pragma unroll
                    for (int k = 0; k < j; k++) t = fma(-x[k], l[j][k], t);
                    x[j] = t * inv[j];
                }
#pragma unroll
                for (int j = 0; j < 8; j++) row[j ^ rs] = x[j];
            }
        }
        ICP_FT({ const long long n_ = clock64(); fph[3] += n_ - ftk; ftk = n_; })
        __syncthreads();
        ICP_FT({ const long long n_ = clock64(); fph[4] += n_ - ftk; ftk = n_; })
    }
    ICP_FT(if (tid == 0 && c < 8192) for (int k_ = 0; k_ < 5; k_++) g_ft[kFtStride * c + 1 + k_] = fph[k_];)
    // back substitution L^T x = y
    ICP_FT(const long long ftb = clock64(); if (tid == 0 && c < 8192) g_ft[kFtStride * c + 9] = ftb - ftf;)
    if (!YMEAN) {
        for (int k = tid; k < Kp; k += NT) xs[k] = yv[k];
        __syncthreads();
        for (int bj = NB - 1; bj >= 0; bj--) {
            const double *D = A + pk_blk(bj, bj);
            double x[8];
#pragma unroll
            for (int i = 7; i >= 0; i--) {
                double t = xs[8 * bj + i];
#pragma unroll
                for (int k = i + 1; k < 8; k++) t = fma(-D[k * 8 + (i ^ pk_swz(k))], x[k], t);
                x[i] = t * dinv[8 * bj + i];
            }
            if (tid < 8) {
#pragma unroll
                for (int i = 0; i < 8; i++)
                    if (i == tid) xo[8 * bj + i] = x[i];
            }
            for (int k = tid; k < 8 * bj; k += NT) {
                const double *blk = A + pk_blk(bj, k >> 3);   // elements (8 bj + p, k), p = 0..7
                double t = xs[k];
#pragma unroll
                for (int p = 0; p < 8; p++) t = fma(-blk[p * 8 + ((k & 7) ^ pk_swz(p))], x[p], t);
                xs[k] = t;
            }
            __syncthreads();
        }
    }
    ICP_FT(const long long fts = clock64(); if (tid == 0 && c < 8192) g_ft[kFtStride * c + 10] = fts - ftb;)
    const bool isbad = bad != 0;
    const int oc = out_slot ? out_slot[c] : c;
    double *Lc = L + (size_t)oc * Kp * Kp;
    // Only the lower triangle of L is ever read (back substitutions and L^T products), so only it is written: a warp
    // writes row i as i / 2 + 1 column pairs (the pair that straddles the diagonal carries the stored zero). Streaming
    // stores: 43 KB per chain must not evict the basis from L2.
    for (int i = warp; i < Kp; i += NT / 32) {
        const double *rowp = A + pk_blk(i >> 3, 0) + (i & 7) * 8;
        const int rs = pk_swz(i & 7);
        for (int jp = lane; jp <= (i >> 1); jp += 32) {
            const int j = 2 * jp;
            double2 v = *reinterpret_cast<const double2 *>(rowp + (j >> 3) * 64 + ((j & 7) ^ rs));
            if (isbad) v = make_double2(NAN, NAN);
            __stcs(reinterpret_cast<double2 *>(Lc + (size_t)i * Kp + j), v);
        }
    }
    for (int j = tid; j < Kp; j += NT) __stcs(mu + (size_t)oc * Kp + j, isbad ? NAN : YMEAN ? yv[j] : xo[j]);
    if (tid == 0 && status) status[c] = isbad ? 1 : 0;
    if (qa.out) {
        // chain runner: |L^T d|^2 of the transition theta_post -> theta_other while L is still here (k_chain_accept would
        // otherwise read it back from HBM). d = w - mu (YMEAN: w, and y is subtracted after the product) overwrites the
        // right-hand side scratch.
        const int Lt = qa.K + kTheta0;
        const double *tp = qa.theta_post + (size_t)c * Lt + kTheta0, *to = qa.theta_other + (size_t)c * Lt + kTheta0;
        for (int k = tid; k < Kp; k += NT) {
            const double w = k < qa.K ? tp[k] + ((to[k] - tp[k]) / qa.step) : 0.0;
            xs[k] = YMEAN ? w : k < qa.K ? w - xo[k] : 0.0;
        }
        __syncthreads();
        double part = 0.0;
        for (int j = tid; j < Kp; j += NT) {
            double v0 = 0.0, v1 = 0.0;
            int i = j;
            for (; i + 1 < Kp; i += 2) { v0 = fma(A[pk_at(i, j)], xs[i], v0); v1 = fma(A[pk_at(i + 1, j)], xs[i + 1], v1); }
            if (i < Kp) v0 = fma(A[pk_at(i, j)], xs[i], v0);
            const double v = YMEAN ? (v0 + v1) - yv[j] : v0 + v1;
            part = fma(v, v, part);
        }
        // block sum through the (now free) dinv scratch
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        __syncthreads();
        if (lane == 0) dinv[warp] = part;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < NT / 32; w++) t += dinv[w];
            qa.out[c] = isbad ? NAN : t;
        }
    }
    ICP_FT(if (tid == 0 && c < 8192) g_ft[kFtStride * c + 11] = clock64() - fts;)
}

template <int NT, bool YMEAN>
static void launch_cholesky_packed_nt(int C, int Kp, size_t smem_c, const double *d_Mp, const double *d_b, double *d_M, double *d_L,
                                      double *d_mu, const int *d_out_slot, int *d_status, const QuadArgs &q, const int *d_list,
                                      const int *d_count, cudaStream_t s) {
    ICP_CUDA(cudaFuncSetAttribute(k_cholesky_packed<NT, YMEAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c));
    k_cholesky_packed<NT, YMEAN><<<C, NT, smem_c, s>>>(Kp, d_Mp, d_b, d_M, d_L, d_mu, d_out_slot, d_status, q, d_list, d_count);
}

static void run_cholesky_packed(int C, int Kp, size_t smem_c, const double *d_Mp, const double *d_b, double *d_M, double *d_L, double *d_mu,
                                const int *d_out_slot, int *d_status, const QuadArgs *qa, bool ymean, const int *d_list,
                                const int *d_count, cudaStream_t s) {
    const QuadArgs q = qa ? *qa : QuadArgs{};
    // the two ICP posteriors of a step factorise concurrently: up to 148 chains all their matrices are resident at two per SM
    // (measured: 148 chains 605 k -> 646 k samples/s, one chain's round 0.179 -> 0.175 ms; at 296 chains 128 threads win)
    if (C <= 148 && Kp <= 128) {
        if (ymean) launch_cholesky_packed_nt<256, true>(C, Kp, smem_c, d_Mp, d_b, d_M, d_L, d_mu, d_out_slot, d_status, q, d_list, d_count, s);
        else launch_cholesky_packed_nt<256, false>(C, Kp, smem_c, d_Mp, d_b, d_M, d_L, d_mu, d_out_slot, d_status, q, d_list, d_count, s);
    } else {
        if (ymean) launch_cholesky_packed_nt<kCh3Threads, true>(C, Kp, smem_c, d_Mp, d_b, d_M, d_L, d_mu, d_out_slot, d_status, q, d_list, d_count, s);
        else launch_cholesky_packed_nt<kCh3Threads, false>(C, Kp, smem_c, d_Mp, d_b, d_M, d_L, d_mu, d_out_slot, d_status, q, d_list, d_count, s);
    }
}

// accumulator block (bi, bj) -> shared-memory matrix of the factorisation (+ I, + Gs / sd_t^2 on the fast path)
template <int RPO>
__device__ __forceinline__ void store_block(double *sA, int ld, int Kp, int bi, int bj, int lane, const double (&a)[2],
                                            const double *__restrict__ Gs, double gs_scale) {
    int i = 8 * bi + (lane >> 2), j = 8 * bj + 2 * (lane & 3);
    double v0 = a[0] + (i == j ? 1.0 : 0.0), v1 = a[1] + (i == j + 1 ? 1.0 : 0.0);
    if (RPO == 1) {
        double2 g = __ldg(reinterpret_cast<const double2 *>(Gs + (size_t)i * Kp + j));
        v0 = fma(g.x, gs_scale, v0);
        v1 = fma(g.y, gs_scale, v1);
    }
    if (ld > 0) *reinterpret_cast<double2 *>(sA + (size_t)i * ld + j) = make_double2(v0, v1);
    else        // ld == 0: sA is the chain's block-packed matrix in global memory (see k_cholesky_packed); a warp
                // writes one contiguous 512-byte block
        *reinterpret_cast<double2 *>(sA + (size_t)(bi * (bi + 1) / 2 + bj) * 64 + 4 * (lane >> 2) * 2 + 2 * (lane & 3)) =
            make_double2(v0, v1);
}

// Fused variant: posterior build (as k_posterior_build_mma) + Cholesky + solve in one kernel. The accumulator
// fragments go straight into the shared-memory matrix of the factorisation (M never visits global memory unless the
// caller asks for it), and with two CTAs per SM the latency-bound factorisation of one chain overlaps the DMMA
// stream of the other.
// RPO = rows of A per observation. RPO = 3: the general whitened rows F_i Q_i. RPO = 1 (constant-Gram fast path,
// model sampling with every observation kept and sd_n <= sd_t): Sigma_i^-1 = I / sd_t^2 + kappa n n^T with
// kappa = 1/sd_n^2 - 1/sd_t^2, so M = I + Gs / sd_t^2 + sum_i (sqrt(kappa) Q_i^T n_i)(...)^T where
// Gs = sum_i Q_i^T Q_i is a constant of the proposal: one row per observation, a third of the DMMA work.
// CHOL = false: rank update only - the lower-triangle blocks of M go to global memory block-packed (M_out; 64 doubles
// per 8 x 8 block, row-major over the block triangle) and b to mu; k_cholesky_packed factorises them at twice the occupancy.
template <int NBLK, int NBMAX, int NWC, int RPO, bool CHOL>
__global__ void __launch_bounds__((NWC + kProdWarps) * 32, 2) k_posterior_fused(ModelDev m, ObsDev o, double *__restrict__ M_out,
                                                                             int nblk_total, const double *__restrict__ Gs,
                                                                             double gs_scale, double row_scale,
                                                                             double *__restrict__ L, double *__restrict__ mu,
                                                                             const int *__restrict__ out_slot,
                                                                             int *__restrict__ status, bool ymean) {
    extern __shared__ __align__(16) double sm[];
    const int Kp = m.Kp, ld = Kp + 4, NB = Kp >> 3;
    const int bufsz = kMmaRows * ld;
    double *sA = sm;                    // [2][24][ld]; later reused as the matrix of the factorisation
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    // entry ent of the launch is chain c (ObsDev::list), whose observations are row orow (ObsDev::row); CHOL = false writes M
    // and b at ent
    const int ent = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (o.count && ent >= *o.count) return;
    const int c = o.list ? o.list[ent] : ent, orow = o.row ? o.row[c] : c;
    constexpr int nthreads = (NWC + kProdWarps) * 32, nwc = NWC;
    constexpr int kObsChunk = kMmaRows / RPO;   // observations per staged chunk (8 or 24)
    const int nrows = o.nrows ? o.nrows[orow] : o.n;   // slots in use (uniform over the CTA)
    const int nchunks = (nrows + kObsChunk - 1) / kObsChunk;
    double *Mdst = CHOL ? sA : M_out + (size_t)ent * nblk_total * 64;   // where the accumulator blocks go
    const int ldst = CHOL ? ld : 0;
    ICP_FT(long long ft0 = clock64(); long long ftw = 0; long long ftw2 = 0;)
    if (warp < nwc) {
        // ------------------------------- consumers: DMMA ------------------------------------------------
        const int frag = (lane & 3) * ld + (lane >> 2);
        if (NBMAX == 13 && NWC == 4 && NB == 13) {
            // rectangular / triangular roles (see mma_rect_chunk)
            named_bar_arrive<3>(nthreads);  // both buffers start empty
            named_bar_arrive<4>(nthreads);
#define ICP_CONSUME(...)                                                                               \
            for (int ch = 0; ch < nchunks; ch++) {                                                     \
                const int buf = ch & 1;                                                                \
                ICP_FT(long long fta = clock64();)                                                     \
                if (buf == 0) named_bar_sync<1>(nthreads); else named_bar_sync<2>(nthreads);           \
                ICP_FT(ftw += clock64() - fta;)                                                        \
                const double *base = sA + buf * bufsz + frag;                                          \
                __VA_ARGS__                                                                            \
                if (buf == 0) named_bar_arrive<3>(nthreads); else named_bar_arrive<4>(nthreads);       \
            }                                                                                          \
            ICP_FT(if (tid == 0 && c < 8192) { g_ft[kFtStride * c + 1] = ftw; g_ft[kFtStride * c + 2] = clock64() - ft0; }) \
            if (CHOL) named_bar_sync<6>(nthreads); /* staging buffers are free: the matrix takes their place */
            if (warp == 0) {          // rows B (5..8) x cols A (0..4)
                double acc[20][2] = {};
                ICP_CONSUME(mma_rect_chunk<4, 5>(acc, base, ld, 5, 0);)
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 5; j++) store_block<RPO>(Mdst, ldst, Kp, 5 + i, j, lane, acc[i * 5 + j], Gs, gs_scale);
            } else if (warp == 1) {   // rows C (9..12) x cols A
                double acc[20][2] = {};
                ICP_CONSUME(mma_rect_chunk<4, 5>(acc, base, ld, 9, 0);)
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 5; j++) store_block<RPO>(Mdst, ldst, Kp, 9 + i, j, lane, acc[i * 5 + j], Gs, gs_scale);
            } else if (warp == 2) {   // rows C x cols B, and the triangle of B
                double acc[16][2] = {}, tri[10][2] = {};
                ICP_CONSUME(mma_rect_chunk<4, 4>(acc, base, ld, 9, 5); mma_tri_chunk<4>(tri, base, ld, 5);)
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) store_block<RPO>(Mdst, ldst, Kp, 9 + i, 5 + j, lane, acc[i * 4 + j], Gs, gs_scale);
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j <= i; j++) store_block<RPO>(Mdst, ldst, Kp, 5 + i, 5 + j, lane, tri[i * (i + 1) / 2 + j], Gs, gs_scale);
            } else {                  // the triangles of A and of C
                double ta[15][2] = {}, tc[10][2] = {};
                ICP_CONSUME(mma_tri_chunk<5>(ta, base, ld, 0); mma_tri_chunk<4>(tc, base, ld, 9);)
#pragma unroll
                for (int i = 0; i < 5; i++)
#pragma unroll
                    for (int j = 0; j <= i; j++) store_block<RPO>(Mdst, ldst, Kp, i, j, lane, ta[i * (i + 1) / 2 + j], Gs, gs_scale);
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j <= i; j++) store_block<RPO>(Mdst, ldst, Kp, 9 + i, 9 + j, lane, tc[i * (i + 1) / 2 + j], Gs, gs_scale);
            }
#undef ICP_CONSUME
        } else {
        const int per = (nblk_total + nwc - 1) / nwc;
        const int b0 = warp * per;
        const int nmine = max(0, min(nblk_total, b0 + per) - b0);
        int bi0, bj0;
        tri_index(b0 < nblk_total ? b0 : 0, bi0, bj0);
        double acc[NBLK][2];
#pragma unroll
        for (int s = 0; s < NBLK; s++) acc[s][0] = acc[s][1] = 0.0;
        named_bar_arrive<3>(nthreads);  // both buffers start empty
        named_bar_arrive<4>(nthreads);
        for (int ch = 0; ch < nchunks; ch++) {
            const int buf = ch & 1;
            if (buf == 0) named_bar_sync<1>(nthreads); else named_bar_sync<2>(nthreads);
            const double *base = sA + buf * bufsz + frag;
            int bi = bi0, bj = bj0;
            double fa[6];
#pragma unroll
            for (int k = 0; k < 6; k++) fa[k] = base[k * 4 * ld + 8 * bi];
            // blocks are taken two at a time when both lie in the same block row (same A fragment): their DMMAs are
            // interleaved so that consecutive DMMAs never accumulate into the same registers
#pragma unroll
            for (int s = 0; s < NBLK; s += 2) {
                if (s + 1 < NBLK && s + 1 < nmine && bj + 1 <= bi) {
#pragma unroll
                    for (int half = 0; half < 2; half++) {
                        double f0[3], f1[3];
#pragma unroll
                        for (int k = 0; k < 3; k++) {
                            f0[k] = base[(3 * half + k) * 4 * ld + 8 * bj];
                            f1[k] = base[(3 * half + k) * 4 * ld + 8 * bj + 8];
                        }
#pragma unroll
                        for (int k = 0; k < 3; k++) {
                            dmma_8x8x4(acc[s][0], acc[s][1], fa[3 * half + k], f0[k]);
                            dmma_8x8x4(acc[s + 1 < NBLK ? s + 1 : s][0], acc[s + 1 < NBLK ? s + 1 : s][1], fa[3 * half + k], f1[k]);
                        }
                    }
                    bj += 2;
                    if (bj > bi) {
                        bj = 0;
                        if (++bi < NB) {
#pragma unroll
                            for (int k = 0; k < 6; k++) fa[k] = base[k * 4 * ld + 8 * bi];
                        }
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        if (s + u < NBLK && s + u < nmine) {
                            double fb[6];
#pragma unroll
                            for (int k = 0; k < 6; k++) fb[k] = base[k * 4 * ld + 8 * bj];
#pragma unroll
                            for (int k = 0; k < 6; k++) dmma_8x8x4(acc[s + u < NBLK ? s + u : s][0], acc[s + u < NBLK ? s + u : s][1], fa[k], fb[k]);
                            if (++bj > bi) {
                                bj = 0;
                                if (++bi < NB) {
#pragma unroll
                                    for (int k = 0; k < 6; k++) fa[k] = base[k * 4 * ld + 8 * bi];
                                }
                            }
                        }
                    }
                }
            }
            if (buf == 0) named_bar_arrive<3>(nthreads); else named_bar_arrive<4>(nthreads);
        }
        if (CHOL) named_bar_sync<6>(nthreads);   // staging buffers and the b scratch are free: the matrix takes their place
        int bi = bi0, bj = bj0;
#pragma unroll
        for (int s = 0; s < NBLK; s++) {
            if (s < nmine) {
                store_block<RPO>(Mdst, ldst, Kp, bi, bj, lane, acc[s], Gs, gs_scale);
                if (++bj > bi) { bj = 0; ++bi; }
            }
        }
        }
    } else {
        // ------------------------------- producers: gather + whiten ----------------------------------------
        const int pt = tid - nwc * 32;          // 0 .. 63
        const int ob = pt >> 3, cg = pt & 7;     // observation slot within the chunk, column group
        const int *vid = o.vid + (size_t)orow * o.n;
        const double *F = o.F + (size_t)orow * o.n * 9;
        const double *y = o.y + (size_t)orow * o.n * 3;
        constexpr int kNJ = (NBMAX + 1) / 2;     // column pairs per producer thread on the 16-byte path
        double bacc[2 * kNJ];
#pragma unroll
        for (int i = 0; i < 2 * kNJ; i++) bacc[i] = 0.0;
        // the vertex ids gate the addresses of every basis-row load: stage them in shared memory once so that a
        // pass pays one L2 round trip (ids -> rows would be two dependent ones)
        int *svid = reinterpret_cast<int *>(sm + 2 * bufsz + 8 * Kp);
        const bool vid_staged = o.n <= kMaxStagedIds;
        if (vid_staged) {
            for (int e = pt; e < nrows; e += kProdWarps * 32) svid[e] = __ldg(&vid[e]);
            named_bar_sync<5>(kProdWarps * 32);
        }
        if (vid_staged) {
            // cp.async pipeline, private per thread: every producer thread copies exactly the basis entries it will
            // whiten itself - column pairs (2 cg + 16 j, + 1) of its observation's 3 rows, as 16-byte cp.async.ca into
            // its own shared-memory slot - one pass ahead, so the only waits are its own cp.async group and the
            // FULL / EMPTY hand-off with the consumers: no producer-side barriers. 8 lanes cover one 128-byte line; the
            // copies allocate in L1 because the two CTAs of an SM read the same rows (.cg was 2x slower here).
            constexpr int ppc = kObsChunk / 8;            // passes (of 8 observations) per staged chunk
            constexpr int kSlot = 3 * kNJ * 2;            // doubles per thread and stage
            const int npass = nchunks * ppc;
            double *raw = sm + 2 * bufsz + 8 * Kp + ((kMaxStagedIds < o.n ? kMaxStagedIds : o.n) + 3) / 4 * 2;
            double *mine = raw + (size_t)pt * kSlot;      // + (pass % kRawStages) * 64 * kSlot
            // per-observation scalars (F, F y) travel one pass ahead in registers; nothing may consume them before the
            // next pass (they come from DRAM: a use here would stall the producer for a full DRAM round trip per pass)
            double fn[12];
            auto issue = [&](int pp) {                    // basis rows of pass pp -> this thread's slot (one group)
                if (pp < npass) {
                    const int gi = pp * 8 + ob;
                    const int v = gi < nrows ? svid[gi] : -1;
                    const double *src = m.Q + (size_t)3 * (v >= 0 ? v : 0) * Kp + 2 * cg;
                    double *dr = mine + (size_t)(pp % kRawStages) * (kProdWarps * 32) * kSlot;
#pragma unroll
                    for (int d = 0; d < 3; d++)
#pragma unroll
                        for (int j = 0; j < kNJ; j++)
                            if (2 * cg + 16 * j < Kp) cp_async_16_ca(dr + (d * kNJ + j) * 2, src + d * Kp + 16 * j);
                }
                cp_async_commit();
            };
            auto frame = [&](int pp) {
                const int gi = pp * 8 + ob;
                const int vn = gi < nrows ? svid[gi] : -1;
                if (vn >= 0) {
#pragma unroll
                    for (int k = 0; k < 9; k++) fn[k] = __ldg(F + (size_t)gi * 9 + k);
#pragma unroll
                    for (int k = 0; k < 3; k++) fn[9 + k] = __ldg(y + (size_t)gi * 3 + k);
                } else {
#pragma unroll
                    for (int k = 0; k < 12; k++) fn[k] = 0.0;
                }
            };
#pragma unroll
            for (int st = 0; st < kRawStages - 1; st++) issue(st);
            frame(0);
#pragma unroll 1
            for (int pp = 0; pp < npass; pp++) {
                const int ch = pp / ppc, sub = pp - ch * ppc, buf = ch & 1, rb = pp % kRawStages;
                constexpr int kNF = RPO == 1 ? 6 : 12;
                double f[kNF];
                if (RPO == 1) {
                    // only the normal row is staged, and b += Q_i^T (F_i^T F_i y_i) needs no tangential rows either:
                    // g = row_scale * n / sd_n and w = F^T (F y)
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        f[k] = fn[k] * row_scale;
                        f[3 + k] = fn[k] * fn[9] + fn[3 + k] * fn[10] + fn[6 + k] * fn[11];
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < kNF; k++) f[k] = fn[k];
                }
                ICP_FT(long long fta = clock64();)
                if (pp + 1 < npass) frame(pp + 1);
                issue(pp + kRawStages - 1);               // refills the slot read in pass pp - 1
                cp_async_wait<kRawStages - 1>();          // all but the newest kRawStages - 1 groups: pass pp has landed
                ICP_FT(long long ftb = clock64(); ftw2 += ftb - fta;)
                if (sub == 0) {  // consumers are done with this buffer
                    if (buf == 0) named_bar_sync<3>(nthreads); else named_bar_sync<4>(nthreads);
                }
                ICP_FT(ftw += clock64() - ftb;)
                const double2 *rr = reinterpret_cast<const double2 *>(mine + (size_t)rb * (kProdWarps * 32) * kSlot);
                double *dst = sA + buf * bufsz + (RPO * (sub * 8 + ob)) * ld + 2 * cg;
#pragma unroll
                for (int j = 0; j < kNJ; j++) {
                    if (2 * cg + 16 * j < Kp) {
                        const double2 q0 = rr[j], q1 = rr[kNJ + j], q2 = rr[2 * kNJ + j];
                        if (RPO == 1) {
                            *reinterpret_cast<double2 *>(dst + 16 * j) =
                                make_double2(f[0] * q0.x + f[1] * q1.x + f[2] * q2.x, f[0] * q0.y + f[1] * q1.y + f[2] * q2.y);
                            bacc[2 * j] = fma(q0.x, f[3], fma(q1.x, f[4], fma(q2.x, f[5], bacc[2 * j])));
                            bacc[2 * j + 1] = fma(q0.y, f[3], fma(q1.y, f[4], fma(q2.y, f[5], bacc[2 * j + 1])));
                        } else {
                            const double a0x = f[0] * q0.x + f[1] * q1.x + f[2] * q2.x, a0y = f[0] * q0.y + f[1] * q1.y + f[2] * q2.y;
                            const double a1x = f[3] * q0.x + f[4] * q1.x + f[5] * q2.x, a1y = f[3] * q0.y + f[4] * q1.y + f[5] * q2.y;
                            const double a2x = f[6] * q0.x + f[7] * q1.x + f[8] * q2.x, a2y = f[6] * q0.y + f[7] * q1.y + f[8] * q2.y;
                            *reinterpret_cast<double2 *>(dst + 16 * j) = make_double2(a0x, a0y);
                            *reinterpret_cast<double2 *>(dst + ld + 16 * j) = make_double2(a1x, a1y);
                            *reinterpret_cast<double2 *>(dst + 2 * ld + 16 * j) = make_double2(a2x, a2y);
                            bacc[2 * j] = fma(a0x, f[9], fma(a1x, f[10], fma(a2x, f[11], bacc[2 * j])));
                            bacc[2 * j + 1] = fma(a0y, f[9], fma(a1y, f[10], fma(a2y, f[11], bacc[2 * j + 1])));
                        }
                    }
                }
                if (sub == ppc - 1) {
                    if (buf == 0) named_bar_arrive<1>(nthreads); else named_bar_arrive<2>(nthreads);
                }
            }
        } else {
        for (int ch = 0; ch < nchunks; ch++) {
                const int buf = ch & 1;
    #pragma unroll 1
                for (int pass = 0; pass < kObsChunk / 8; pass++) {
                    const int lo = pass * 8 + ob;            // observation slot within the chunk
                    const int gi = ch * kObsChunk + lo;
                    int v = -1;
                    double f[9], yy[3];
                    if (gi < nrows) v = vid_staged ? svid[gi] : __ldg(&vid[gi]);
                    if (v >= 0) {
    #pragma unroll
                        for (int k = 0; k < 9; k++) f[k] = __ldg(F + (size_t)gi * 9 + k);
    #pragma unroll
                        for (int k = 0; k < 3; k++) yy[k] = __ldg(y + (size_t)gi * 3 + k);
                    } else {
    #pragma unroll
                        for (int k = 0; k < 9; k++) f[k] = 0.0;
                        yy[0] = yy[1] = yy[2] = 0.0;
                    }
                    const double *q = m.Q + (size_t)3 * (v >= 0 ? v : 0) * Kp + cg;
                    double q0[NBMAX], q1[NBMAX], q2[NBMAX];
    #pragma unroll
                    for (int i = 0; i < NBMAX; i++) {
                        if (i < NB) { q0[i] = __ldg(q + 8 * i); q1[i] = __ldg(q + Kp + 8 * i); q2[i] = __ldg(q + 2 * Kp + 8 * i); }
                    }
                    if (pass == 0) {  // consumers are done with this buffer
                        if (buf == 0) named_bar_sync<3>(nthreads); else named_bar_sync<4>(nthreads);
                    }
                    double *dst = sA + buf * bufsz + (RPO * lo) * ld + cg;
    #pragma unroll
                    for (int i = 0; i < NBMAX; i++) {
                        if (i < NB) {
                            double a0 = f[0] * q0[i] + f[1] * q1[i] + f[2] * q2[i];
                            double a1 = f[3] * q0[i] + f[4] * q1[i] + f[5] * q2[i];
                            double a2 = f[6] * q0[i] + f[7] * q1[i] + f[8] * q2[i];
                            if (RPO == 3) { dst[8 * i] = a0; dst[ld + 8 * i] = a1; dst[2 * ld + 8 * i] = a2; }
                            else dst[8 * i] = a0 * row_scale;
                            bacc[i] = fma(a0, yy[0], fma(a1, yy[1], fma(a2, yy[2], bacc[i])));
                        }
                    }
                }
                if (buf == 0) named_bar_arrive<1>(nthreads); else named_bar_arrive<2>(nthreads);
            }
        }
        ICP_FT(if (pt == 0 && c < 8192) { g_ft[kFtStride * c + 3] = ftw; g_ft[kFtStride * c + 4] = ftw2; g_ft[kFtStride * c + 5] = clock64() - ft0; })
        // reduce b over the 8 observation slots (fixed order: deterministic)
        named_bar_sync<5>(kProdWarps * 32);      // producers only
        // the last two buffers may still be read by consumers: use the tail of the shared allocation
        double *sb = sm + 2 * bufsz;             // [8][Kp]
        if (vid_staged) {
#pragma unroll
            for (int j = 0; j < kNJ; j++)
                if (2 * cg + 16 * j < Kp) { sb[ob * Kp + 2 * cg + 16 * j] = bacc[2 * j]; sb[ob * Kp + 2 * cg + 16 * j + 1] = bacc[2 * j + 1]; }
        } else {
#pragma unroll
            for (int i = 0; i < NBMAX; i++)
                if (i < NB) sb[ob * Kp + cg + 8 * i] = bacc[i];
        }
        named_bar_sync<5>(kProdWarps * 32);
        double bval[(8 * NBMAX + kProdWarps * 32 - 1) / (kProdWarps * 32)];
#pragma unroll
        for (int u = 0; u < (8 * NBMAX + kProdWarps * 32 - 1) / (kProdWarps * 32); u++) {
            int j = pt + u * kProdWarps * 32;
            double t = 0.0;
            if (j < Kp) {
#pragma unroll
                for (int r = 0; r < 8; r++) t += sb[r * Kp + j];
            }
            bval[u] = t;
        }
        if (!CHOL) {
#pragma unroll
            for (int u = 0; u < (8 * NBMAX + kProdWarps * 32 - 1) / (kProdWarps * 32); u++) {
                int j = pt + u * kProdWarps * 32;
                if (j < Kp) mu[(size_t)ent * Kp + j] = bval[u];
            }
            ICP_FT(if (pt == 0 && c < 8192) {
                unsigned smid;
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                g_ft[kFtStride * c] = ft0; g_ft[kFtStride * c + 6] = clock64() - ft0; g_ft[kFtStride * c + 7] = ((clock64() - ft0) << 8) | smid;
            })
            return;
        }
        named_bar_sync<6>(nthreads);
        // right-hand side = block row NB of the factorisation (row Kp real, 7 zero rows)
        for (int e = pt; e < 8 * ld; e += kProdWarps * 32) sA[(size_t)Kp * ld + e] = 0.0;
        named_bar_sync<5>(kProdWarps * 32);
#pragma unroll
        for (int u = 0; u < (8 * NBMAX + kProdWarps * 32 - 1) / (kProdWarps * 32); u++) {
            int j = pt + u * kProdWarps * 32;
            if (j < Kp) sA[(size_t)Kp * ld + j] = bval[u];
        }
    }
    if (!CHOL) return;
    __syncthreads();
    if (M_out) {   // only the primitive API (icp_posterior) asks for M
        double *Mc = M_out + (size_t)c * Kp * Kp;
        for (int e = tid; e < Kp * Kp; e += nthreads) {
            int i = e / Kp, j = e - i * Kp;
            Mc[e] = j <= i ? sA[(size_t)i * ld + j] : sA[(size_t)j * ld + i];
        }
    }
    const int oc = out_slot ? out_slot[c] : c;
    ICP_FT(long long ftc = clock64();)
    chol_factor_solve_store<nthreads>(sA, Kp, &bad, L + (size_t)oc * Kp * Kp, mu + (size_t)oc * Kp, status ? status + c : nullptr, ymean);
    ICP_FT(if (tid == 0 && c < 8192) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        g_ft[kFtStride * c] = ft0; g_ft[kFtStride * c + 6] = ftc - ft0; g_ft[kFtStride * c + 7] = ((clock64() - ft0) << 8) | smid;
    })
}

#ifdef ICP_FUSED_TIMING
extern "C" int icp_debug_fused_timing(long long *out, int n) {
    return (int)cudaMemcpyFromSymbol(out, g_ft, sizeof(long long) * (size_t)n);
}
#endif

template <int NBLK, int NBMAX, int NWC>
static void launch_fused(const ModelDev &m, int C, const ObsDev &o, double *d_M, int total, const GramFast *gf, double *d_L,
                         double *d_mu, const int *d_out_slot, int *d_status, double *d_Mp, double *d_b, cudaStream_t s,
                         const QuadArgs *qa, bool *quad_done, bool ymean) {
    const int Kp = m.Kp, ld = Kp + 4;
    size_t stage = (size_t)2 * kMmaRows * ld + 8 * Kp + (std::min(o.n, kMaxStagedIds) + 3) / 4 * 2 + (size_t)kRawStages * kProdWarps * 32 * 3 * ((NBMAX + 1) / 2) * 2;
    size_t fact = (size_t)(Kp + 8) * ld + 3 * Kp;
    const unsigned nthr = (NWC + kProdWarps) * 32;
    if (d_Mp) {
        // rank update (block-packed M and b to global memory), then the high-occupancy factorisation
        size_t smem = sizeof(double) * stage;
        {
            ProfScope _ps(ST_POSTERIOR_BUILD, s);
            if (gf) {
                ICP_CUDA(cudaFuncSetAttribute(k_posterior_fused<NBLK, NBMAX, NWC, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_posterior_fused<NBLK, NBMAX, NWC, 1, false><<<C, nthr, smem, s>>>(m, o, d_Mp, total, gf->Gs, gf->gs_scale, gf->row_scale, nullptr, d_b, nullptr, nullptr, false);
            } else {
                ICP_CUDA(cudaFuncSetAttribute(k_posterior_fused<NBLK, NBMAX, NWC, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_posterior_fused<NBLK, NBMAX, NWC, 3, false><<<C, nthr, smem, s>>>(m, o, d_Mp, total, nullptr, 0.0, 1.0, nullptr, d_b, nullptr, nullptr, false);
            }
            ICP_CUDA(cudaGetLastError());
        }
        ProfScope _ps(ST_CHOLESKY, s);
        size_t smem_c = sizeof(double) * ((size_t)total * 64 + 4 * Kp);
        run_cholesky_packed(C, Kp, smem_c, d_Mp, d_b, d_M, d_L, d_mu, d_out_slot, d_status, qa, ymean, o.list, o.count, s);
        if (quad_done) *quad_done = qa != nullptr;
        return;
    }
    ProfScope _ps(ST_POSTERIOR_BUILD, s);
    size_t smem = sizeof(double) * std::max(stage, fact);
    if (gf) {
        ICP_CUDA(cudaFuncSetAttribute(k_posterior_fused<NBLK, NBMAX, NWC, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_posterior_fused<NBLK, NBMAX, NWC, 1, true><<<C, nthr, smem, s>>>(m, o, d_M, total, gf->Gs, gf->gs_scale, gf->row_scale, d_L, d_mu, d_out_slot, d_status, ymean);
    } else {
        ICP_CUDA(cudaFuncSetAttribute(k_posterior_fused<NBLK, NBMAX, NWC, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_posterior_fused<NBLK, NBMAX, NWC, 3, true><<<C, nthr, smem, s>>>(m, o, d_M, total, nullptr, 0.0, 1.0, d_L, d_mu, d_out_slot, d_status, ymean);
    }
}

void launch_cholesky_packed(int C, int Kp, const double *d_Mp, const double *d_b, double *d_M_or_null, double *d_L, double *d_mu,
                            const int *d_out_slot, int *d_status, const QuadArgs *qa, bool ymean, cudaStream_t s,
                            const int *d_list, const int *d_count) {
    ProfScope _ps(ST_CHOLESKY, s);
    const int NB = Kp / 8, total = NB * (NB + 1) / 2;
    size_t smem_c = sizeof(double) * ((size_t)total * 64 + 4 * Kp);
    run_cholesky_packed(C, Kp, smem_c, d_Mp, d_b, d_M_or_null, d_L, d_mu, d_out_slot, d_status, qa, ymean, d_list, d_count, s);
    ICP_CUDA(cudaGetLastError());
}

// posterior build + Cholesky + solve; returns false when the shape is outside the DMMA kernels' range (the caller then
// runs launch_posterior_build + launch_cholesky_solve). Default: two launches - the rank update writes M block-packed
// (d_Mp, C x NB (NB + 1) / 2 x 64 doubles) and b (d_b), k_cholesky_packed factorises at four chains per SM.
// ICPCUDA_FUSE=1 (or d_Mp == nullptr): the single-launch variant, whose factorisation runs at two chains per SM.
static bool fused_off() {
    static const bool off = (getenv("ICPCUDA_NO_DMMA") && getenv("ICPCUDA_NO_DMMA")[0] == '1') ||
                            (getenv("ICPCUDA_NO_FUSE") && getenv("ICPCUDA_NO_FUSE")[0] == '1');
    return off;
}
static bool fused_one_launch() {
    static const bool one_launch = getenv("ICPCUDA_FUSE") && getenv("ICPCUDA_FUSE")[0] == '1';
    return one_launch;
}

bool posterior_packed_path(int Kp) { return !fused_off() && !fused_one_launch() && Kp / 8 <= 13; }

bool launch_posterior_fused(const ModelDev &m, int C, const ObsDev &o, const GramFast *gf, double *d_M_or_null, double *d_L,
                            double *d_mu, const int *d_out_slot, int *d_status, double *d_Mp, double *d_b, cudaStream_t s,
                            const QuadArgs *qa, bool *quad_done, bool ymean) {
    if (quad_done) *quad_done = false;
    const int NB = m.Kp / 8, total = NB * (NB + 1) / 2;
    if (fused_off() || NB > 13 || C <= 0) return false;   // NB <= 13: the 192-thread variants; the fused matrix must fit 2 CTAs / SM
    if (fused_one_launch()) d_Mp = nullptr;
    if (NB <= 4) launch_fused<4, 4, 4>(m, C, o, d_M_or_null, total, gf, d_L, d_mu, d_out_slot, d_status, d_Mp, d_b, s, qa, quad_done, ymean);
    else if (NB <= 7) launch_fused<8, 7, 4>(m, C, o, d_M_or_null, total, gf, d_L, d_mu, d_out_slot, d_status, d_Mp, d_b, s, qa, quad_done, ymean);
    else launch_fused<24, 13, 4>(m, C, o, d_M_or_null, total, gf, d_L, d_mu, d_out_slot, d_status, d_Mp, d_b, s, qa, quad_done, ymean);
    ICP_CUDA(cudaGetLastError());
    return true;
}

// full square M -> the block-packed lower triangle k_cholesky_packed reads (row-major 8 x 8 blocks over the block triangle)
__global__ void __launch_bounds__(128) k_pack_lower(int Kp, const double *__restrict__ M, double *__restrict__ Mp) {
    const int NB = Kp >> 3, ntri = NB * (NB + 1) / 2, c = blockIdx.x;
    const double *Mc = M + (size_t)c * Kp * Kp;
    double *dst = Mp + (size_t)c * ntri * 64;
    for (int e = threadIdx.x; e < ntri * 64; e += blockDim.x) {
        int bi, bj;
        tri_index(e >> 6, bi, bj);
        dst[e] = Mc[(size_t)(8 * bi + ((e >> 3) & 7)) * Kp + 8 * bj + (e & 7)];
    }
}

// mu -> y = L^T mu in place, for the factorisation path that solves for mu only (k_cholesky_solve)
__global__ void __launch_bounds__(128) k_mean_to_ymean(int Kp, const double *__restrict__ L, double *__restrict__ mu,
                                                       const int *__restrict__ slot) {
    extern __shared__ double smu[];
    const int sl = slot ? slot[blockIdx.x] : blockIdx.x;
    const double *Lc = L + (size_t)sl * Kp * Kp;
    double *m = mu + (size_t)sl * Kp;
    for (int k = threadIdx.x; k < Kp; k += blockDim.x) smu[k] = m[k];
    __syncthreads();
    for (int j = threadIdx.x; j < Kp; j += blockDim.x) {
        double v = 0.0;
        for (int i = j; i < Kp; i++) v = fma(Lc[(size_t)i * Kp + j], smu[i], v);
        m[j] = v;
    }
}

void launch_cholesky_solve(int C, int K, int Kp, const double *d_M, const double *d_b, double *d_L, double *d_mu,
                           const int *d_out_slot, int *d_status, cudaStream_t s, double *d_Mp, const QuadArgs *qa, bool *quad_done,
                           bool ymean) {
    ProfScope _ps(ST_CHOLESKY, s);
    if (quad_done) *quad_done = false;
    if (C <= 0) return;
    static const bool no_mma = getenv("ICPCUDA_NO_DMMA") && getenv("ICPCUDA_NO_DMMA")[0] == '1';
    if (sizeof(double) * ((size_t)(Kp + 8) * (Kp + 4) + 3 * Kp) > 227 * 1024) {
        // 160 < Kp <= 224: the padded square does not fit shared memory, the block-packed lower triangle does (one CTA / SM)
        const int NB = Kp / 8, ntri = NB * (NB + 1) / 2;
        size_t smem_c = sizeof(double) * ((size_t)ntri * 64 + 4 * Kp);
        ICP_REQUIRE(d_Mp != nullptr && smem_c <= 227 * 1024 - 64, "rank too large for the shared-memory Cholesky (K <= 224)");
        k_pack_lower<<<C, 128, 0, s>>>(Kp, d_M, d_Mp);
        ICP_CUDA(cudaGetLastError());
        run_cholesky_packed(C, Kp, smem_c, d_Mp, d_b, nullptr, d_L, d_mu, d_out_slot, d_status, qa, ymean, nullptr, nullptr, s);
        ICP_CUDA(cudaGetLastError());
        if (quad_done) *quad_done = qa != nullptr;
        return;
    }
    if (!no_mma) {
        size_t smem2 = sizeof(double) * ((size_t)(Kp + 8) * (Kp + 4) + 3 * Kp);
        ICP_REQUIRE(smem2 <= 227 * 1024, "rank too large for the shared-memory Cholesky (K <= 160)");
        ICP_CUDA(cudaFuncSetAttribute(k_cholesky_solve_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
        k_cholesky_solve_mma<<<C, kCh2Threads, smem2, s>>>(K, Kp, d_M, d_b, d_L, d_mu, d_out_slot, d_status, ymean);
        ICP_CUDA(cudaGetLastError());
        return;
    }
    size_t smem = sizeof(double) * ((size_t)(Kp + 1) * (Kp + 1) + Kp);
    ICP_REQUIRE(smem <= 227 * 1024, "rank too large for the shared-memory Cholesky (K <= 160)");
    ICP_CUDA(cudaFuncSetAttribute(k_cholesky_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_cholesky_solve<<<C, kChThreads, smem, s>>>(K, Kp, d_M, d_b, d_L, d_mu, d_out_slot, d_status);
    ICP_CUDA(cudaGetLastError());
    if (ymean) {   // this path forms mu only: y = L^T mu
        k_mean_to_ymean<<<C, 128, sizeof(double) * Kp, s>>>(Kp, d_L, d_mu, d_out_slot);
        ICP_CUDA(cudaGetLastError());
    }
}

// ---------------------------------------------------------------------------------------------------
// propose / log-transition
// ---------------------------------------------------------------------------------------------------
// w = L^-T z by a single warp (registers + shuffles), L rows read from global memory (L2 resident).
// Requires Kp <= 32 * 8.
__device__ void warp_backsolve_LT(const double *__restrict__ Lc, int Kp, const double *z_sm, double *w_sm) {
    int lane = threadIdx.x & 31;
    double zr[8];
#pragma unroll
    for (int q = 0; q < 8; q++) { int k = lane + 32 * q; zr[q] = k < Kp ? z_sm[k] : 0.0; }
    for (int i = Kp - 1; i >= 0; i--) {
        int owner = i & 31, slot = i >> 5;
        double zi = 0.0;
#pragma unroll
        for (int q = 0; q < 8; q++) if (q == slot) zi = zr[q];
        double wi = __shfl_sync(0xffffffffu, zi, owner) / __ldg(&Lc[(size_t)i * Kp + i]);
        if (lane == 0) w_sm[i] = wi;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            int k = lane + 32 * q;
            if (k < i) zr[q] = fma(-__ldg(&Lc[(size_t)i * Kp + k]), wi, zr[q]);
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(128) k_propose(ModelDev m, double step, const double *__restrict__ theta,
                                                 const double *__restrict__ z, const double *__restrict__ L,
                                                 const double *__restrict__ mu, const int *__restrict__ slot,
                                                 double *__restrict__ theta_out, const double *__restrict__ W) {
    extern __shared__ double sm[];
    const int Kp = m.Kp, K = m.K, Lt = K + kTheta0;
    double *sz = sm, *sw = sm + Kp;
    int c = blockIdx.x;
    int sl = slot ? slot[c] : c;
    const double *Lc = L + (size_t)sl * Kp * Kp, *muc = mu + (size_t)sl * Kp;
    for (int k = threadIdx.x; k < Kp; k += blockDim.x) sz[k] = k < K ? z[(size_t)c * K + k] : 0.0;
    __syncthreads();
    if (W) block_matvec_rows(W + (size_t)sl * Kp * Kp, Kp, sz, sw);          // the reference's SVD factor (ICP_FACTOR_SVD)
    else if (threadIdx.x < 32) warp_backsolve_LT(Lc, Kp, sz, sw);
    __syncthreads();
    for (int k = threadIdx.x; k < Kp; k += blockDim.x) sz[k] = muc[k] + sw[k];   // v = mu + W z
    __syncthreads();
    const double *th = theta + (size_t)c * Lt;
    double *to = theta_out + (size_t)c * Lt;
    for (int j = threadIdx.x; j < Lt; j += blockDim.x) {
        if (j < kTheta0) { to[j] = th[j]; continue; }
        int jj = j - kTheta0;
        double acc = 0.0;  // (S v)_jj, S symmetric: read column-wise for coalescing
        for (int k = 0; k < Kp; k++) acc = fma(__ldg(&m.S[(size_t)k * Kp + jj]), sz[k], acc);
        to[j] = th[j] + (acc - th[j]) * step;                                       // :61-62
    }
}

void launch_propose(const ModelDev &m, int C, double step, const double *d_theta, const double *d_z,
                    const double *d_L, const double *d_mu, const int *d_slot, double *d_theta_out, cudaStream_t s,
                    const double *d_W) {
    if (C <= 0) return;
    ICP_REQUIRE(m.Kp <= 256, "rank too large for the propose kernel (K <= 256)");
    k_propose<<<C, 128, sizeof(double) * 2 * m.Kp, s>>>(m, step, d_theta, d_z, d_L, d_mu, d_slot, d_theta_out, d_W);
    ICP_CUDA(cudaGetLastError());
}

// |L^T d - y|^2 with d in shared memory (y nullable: |L^T d|^2); all threads of the block participate; red: >= 33 doubles
__device__ double block_quad_LT(const double *__restrict__ Lc, int Kp, const double *d_sm, double *red,
                                const double *__restrict__ y = nullptr) {
    double part = 0.0;
    for (int j = threadIdx.x; j < Kp; j += blockDim.x) {
        double v = 0.0;
        for (int i = j; i < Kp; i++) v = fma(__ldg(&Lc[(size_t)i * Kp + j]), d_sm[i], v);
        if (y) v -= y[j];
        part = fma(v, v, part);
    }
    return block_sum(part, red);
}

__global__ void __launch_bounds__(128) k_log_transition(int K, int Kp, double step, const double *__restrict__ from,
                                                        const double *__restrict__ to, const double *__restrict__ L,
                                                        const double *__restrict__ mu, const int *__restrict__ slot,
                                                        double *__restrict__ out) {
    extern __shared__ double sm[];
    double *sd = sm, *red = sm + Kp;
    __shared__ int differs;
    int c = blockIdx.x, Lt = K + kTheta0;
    int sl = slot ? slot[c] : c;
    const double *f = from + (size_t)c * Lt, *t = to + (size_t)c * Lt;
    if (threadIdx.x == 0) differs = 0;
    __syncthreads();
    if (threadIdx.x < kTheta0 && !(f[threadIdx.x] == t[threadIdx.x])) differs = 1;   // :72 only alpha may change
    for (int k = threadIdx.x; k < Kp; k += blockDim.x)
        sd[k] = k < K ? (f[kTheta0 + k] + ((t[kTheta0 + k] - f[kTheta0 + k]) / step)) - mu[(size_t)sl * Kp + k] : 0.0;  // :79
    __syncthreads();
    double q = block_quad_LT(L + (size_t)sl * Kp * Kp, Kp, sd, red);
    if (threadIdx.x == 0) out[c] = differs ? -INFINITY : -0.5 * (K * ICP_LOG_2PI + q);  // :83
}

// |L^T d|^2 with L / mu read back from global memory: the factorisation paths that do not form it in their epilogue
// ymean: the mean slot holds y = L^T mu, and the form is |L^T w - y|^2
__global__ void __launch_bounds__(128) k_quad_form(int Kp, const double *__restrict__ L, const double *__restrict__ mu,
                                                   const int *__restrict__ slot, QuadArgs qa, bool ymean) {
    extern __shared__ double sm[];
    double *sd = sm, *red = sm + Kp;
    const int c = blockIdx.x, Lt = qa.K + kTheta0;
    const int sl = slot ? slot[c] : c;
    const double *tp = qa.theta_post + (size_t)c * Lt + kTheta0, *to = qa.theta_other + (size_t)c * Lt + kTheta0;
    const double *mc = mu + (size_t)sl * Kp;
    for (int k = threadIdx.x; k < Kp; k += blockDim.x) {
        const double w = k < qa.K ? tp[k] + ((to[k] - tp[k]) / qa.step) : 0.0;
        sd[k] = ymean ? w : k < qa.K ? w - mc[k] : 0.0;
    }
    __syncthreads();
    const double q = block_quad_LT(L + (size_t)sl * Kp * Kp, Kp, sd, red, ymean ? mc : nullptr);
    if (threadIdx.x == 0) qa.out[c] = q;
}

void launch_quad_form(int C, int Kp, const double *d_L, const double *d_mu, const int *d_slot, const QuadArgs &qa, bool ymean,
                      cudaStream_t s) {
    if (C <= 0) return;
    k_quad_form<<<C, 128, sizeof(double) * (Kp + 40), s>>>(Kp, d_L, d_mu, d_slot, qa, ymean);
    ICP_CUDA(cudaGetLastError());
}

void launch_log_transition(int C, int K, int Kp, double step, const double *d_from, const double *d_to,
                           const double *d_L, const double *d_mu, const int *d_slot, double *d_out, cudaStream_t s) {
    if (C <= 0) return;
    k_log_transition<<<C, 128, sizeof(double) * (Kp + 40), s>>>(K, Kp, step, d_from, d_to, d_L, d_mu, d_slot, d_out);
    ICP_CUDA(cudaGetLastError());
}

}  // namespace icp

// Factorises C symmetric matrices M (host, C x K x K) with right-hand sides b (C x K) on the device path the posterior
// pipeline takes at this rank (Kp <= 104: k_cholesky_packed; above: launch_cholesky_solve), in the mu form (ymean = 0) or the
// chain runner's form (ymean = 1). Out: L (C x K x K, lower triangle; the upper triangle is left as passed in), mean (mu or
// y = L^-1 b), q (|L^T d|^2 of the transition theta_post -> theta_other, C x (K + 10) each; NULL: not formed), status.
extern "C" int32_t icp_debug_factor(icp_ctx ctx, int32_t C, int32_t K, const double *M, const double *b, const double *theta_post,
                                    const double *theta_other, double step, int32_t ymean, double *L, double *mean, double *q,
                                    int32_t *status) {
    using namespace icp;
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx && C > 0 && K > 0 && M && b && L && mean && status, "null or empty argument");
        // the ranks of icp_model_create: 225..232 would still fit the packed factorisation (Kp = 232), but no posterior
        // pipeline runs there, so a result at those ranks would describe nothing the library computes
        ICP_REQUIRE(K <= 224, "rank K must be in [1, 224]");
        ICP_REQUIRE(!q || (theta_post && theta_other), "q needs theta_post and theta_other");
        CtxLock lock(ctx);
        cudaStream_t s = ctx->stream;
        const int Kp = (K + 7) / 8 * 8, NB = Kp / 8, Lt = K + kTheta0;
        // padded exactly as the rank update pads: identity on the padded diagonal, zero right-hand side
        std::vector<double> hM((size_t)C * Kp * Kp, 0.0), hb((size_t)C * Kp, 0.0);
        for (int c = 0; c < C; c++) {
            for (int i = 0; i < Kp; i++)
                for (int j = 0; j < Kp; j++)
                    hM[((size_t)c * Kp + i) * Kp + j] = i < K && j < K ? M[((size_t)c * K + i) * K + j] : i == j ? 1.0 : 0.0;
            for (int i = 0; i < K; i++) hb[(size_t)c * Kp + i] = b[(size_t)c * K + i];
        }
        DevBuf<double> dM, db, dMp, dL, dmean, dtp, dto, dq;
        DevBuf<int> dst;
        dM.upload(hM.data(), hM.size(), s);
        db.upload(hb.data(), hb.size(), s);
        dMp.alloc((size_t)C * NB * (NB + 1) / 2 * 64);
        dL.alloc((size_t)C * Kp * Kp);
        ICP_CUDA(cudaMemsetAsync(dL.p, 0, sizeof(double) * dL.n, s));
        dmean.alloc((size_t)C * Kp);
        dst.alloc(C);
        QuadArgs qa{};
        if (q) {
            dtp.upload(theta_post, (size_t)C * Lt, s);
            dto.upload(theta_other, (size_t)C * Lt, s);
            dq.alloc(C);
            qa = QuadArgs{dtp.p, dto.p, step, K, dq.p};
        }
        bool quad_done = false;
        if (NB <= 13) {
            k_pack_lower<<<C, 128, 0, s>>>(Kp, dM.p, dMp.p);
            ICP_CUDA(cudaGetLastError());
            launch_cholesky_packed(C, Kp, dMp.p, db.p, nullptr, dL.p, dmean.p, nullptr, dst.p, q ? &qa : nullptr, ymean != 0, s);
            quad_done = q != nullptr;
        } else {
            launch_cholesky_solve(C, K, Kp, dM.p, db.p, dL.p, dmean.p, nullptr, dst.p, s, dMp.p, q ? &qa : nullptr, &quad_done, ymean != 0);
        }
        if (q && !quad_done) launch_quad_form(C, Kp, dL.p, dmean.p, nullptr, qa, ymean != 0, s);
        std::vector<double> hL((size_t)C * Kp * Kp), hm((size_t)C * Kp);
        ICP_CUDA(cudaMemcpyAsync(hL.data(), dL.p, sizeof(double) * hL.size(), cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaMemcpyAsync(hm.data(), dmean.p, sizeof(double) * hm.size(), cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaMemcpyAsync(status, dst.p, sizeof(int) * C, cudaMemcpyDeviceToHost, s));
        if (q) ICP_CUDA(cudaMemcpyAsync(q, dq.p, sizeof(double) * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        for (int c = 0; c < C; c++)
            for (int i = 0; i < K; i++) {
                for (int j = 0; j <= i; j++) L[((size_t)c * K + i) * K + j] = hL[((size_t)c * Kp + i) * Kp + j];
                mean[(size_t)c * K + i] = hm[(size_t)c * Kp + i];
            }
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}
