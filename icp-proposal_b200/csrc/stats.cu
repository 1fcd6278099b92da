// stats.cu - posterior variability maps accumulated inside the fused chain runner (icp_chain_set_statistics).
//
// apps/util/PosteriorVariability.scala:30-73 over the samples LogHelper.samplesFromLog (apps/util/LogHelper.scala:25-42)
// selects, without a chain log: every chain keeps FP64 accumulators - a count, and per vertex the mean, the centred
// second moment M2 (xx, yy, zz, xy, xz, yz) and the sum of unit vertex normals. The runner does not add a sample at every
// selected step: a chain counts the selected records at which its current state was current ("pending") and, when it
// accepts, hands (old state, pending) to launch_stats_flush - one weighted Welford / Chan update per flushed chain:
//   n' = n + w,  mean += (w / n') d,  M2 += (w n / n') d d^T,  normal_sum += w n^,   d = x - mean.
// The step-by-step runner, the look-ahead at any width and runs split by resume present the same sequence of (state, weight)
// updates to the same kernels, so their maps are bit-identical.
#include "icp_device.cuh"
#include "icp_internal.h"

namespace icp {

namespace {

constexpr int kStThreads = 128;   // thread = vertex
constexpr int kStCH = 8;          // flushed chains per CTA of the reconstruction (every basis entry read serves 8 chains)

// idx[0 .. *count) = the chains with w > 0, in chain order (one CTA, block-wide scan of the flags)
__global__ void __launch_bounds__(1024) k_stats_compact(int C, const long long *__restrict__ w, int *__restrict__ idx,
                                                        int *__restrict__ count) {
    __shared__ int wsum[32];
    __shared__ int base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int c0 = 0; c0 < C; c0 += blockDim.x) {
        const int c = c0 + threadIdx.x;
        const int f = (c < C && w[c] > 0) ? 1 : 0;
        const unsigned mask = __ballot_sync(0xffffffffu, f);
        const int pre = __popc(mask & ((1u << lane) - 1u));
        if (lane == 0) wsum[warp] = __popc(mask);
        __syncthreads();
        if (warp == 0) {
            int v = lane < nw ? wsum[lane] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, v, o);
                if (lane >= o) v += t;
            }
            wsum[lane] = v;   // inclusive prefix over the warps
        }
        __syncthreads();
        if (f) idx[base + (warp ? wsum[warp - 1] : 0) + pre] = c;
        __syncthreads();
        if (threadIdx.x == 0) base += wsum[nw - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

// X[j] = transformedMesh(theta[idx[j]]) for j < *count, the arithmetic of k_reconstruct (model.cu); a CTA takes 128 vertices
// of kStCH listed chains at a time
__global__ void __launch_bounds__(kStThreads) k_stats_reconstruct(ModelDev m, const double *__restrict__ theta,
                                                                  const int *__restrict__ idx, const int *__restrict__ count,
                                                                  double *__restrict__ X) {
    extern __shared__ double sm[];
    double *sa = sm;                              // [K][kStCH]
    double *sp = sm + (size_t)m.K * kStCH;        // [kStCH][16]: R(9) s t(3) c(3)
    const int n = *count, L = m.K + kTheta0;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    for (int g0 = blockIdx.y * kStCH; g0 < n; g0 += gridDim.y * kStCH) {
        const int nc = min(kStCH, n - g0);
        __syncthreads();   // the previous group's reads of sa / sp are done
        for (int e = threadIdx.x; e < m.K * kStCH; e += blockDim.x) {
            const int k = e / kStCH, cc = e % kStCH;
            sa[e] = cc < nc ? theta[(size_t)idx[g0 + cc] * L + kTheta0 + k] : 0.0;
        }
        if (threadIdx.x < nc) {
            const double *th = theta + (size_t)idx[g0 + threadIdx.x] * L;
            double *p = sp + threadIdx.x * 16;
            pose_matrix(th, p);
            p[9] = th[0];
            p[10] = th[1]; p[11] = th[2]; p[12] = th[3];
            p[13] = th[7]; p[14] = th[8]; p[15] = th[9];
        }
        __syncthreads();
        if (i >= m.N) continue;
        double acc[3][kStCH];
#pragma unroll
        for (int d = 0; d < 3; d++)
#pragma unroll
            for (int cc = 0; cc < kStCH; cc++) acc[d][cc] = 0.0;
        const size_t rows = (size_t)3 * m.N;
        const double *qt = m.QT + (size_t)3 * i;
#pragma unroll 4
        for (int k = 0; k < m.K; k++) {
            const double q0 = __ldg(qt + k * rows), q1 = __ldg(qt + k * rows + 1), q2 = __ldg(qt + k * rows + 2);
#pragma unroll
            for (int cc = 0; cc < kStCH; cc++) {
                const double a = sa[k * kStCH + cc];
                acc[0][cc] = fma(q0, a, acc[0][cc]);
                acc[1][cc] = fma(q1, a, acc[1][cc]);
                acc[2][cc] = fma(q2, a, acc[2][cc]);
            }
        }
        const double r0 = m.ref[3 * i], r1 = m.ref[3 * i + 1], r2 = m.ref[3 * i + 2];
        const double m0 = m.mean[3 * i], m1 = m.mean[3 * i + 1], m2 = m.mean[3 * i + 2];
#pragma unroll
        for (int cc = 0; cc < kStCH; cc++) {
            if (cc >= nc) break;
            const double *p = sp + cc * 16;
            const double px = r0 + (m0 + acc[0][cc]) - p[13], py = r1 + (m1 + acc[1][cc]) - p[14], pz = r2 + (m2 + acc[2][cc]) - p[15];
            double *o = X + ((size_t)(g0 + cc) * m.N + i) * 3;
            o[0] = p[9] * ((p[0] * px + p[1] * py + p[2] * pz) + p[13] + p[10]);
            o[1] = p[9] * ((p[3] * px + p[4] * py + p[5] * pz) + p[14] + p[11]);
            o[2] = p[9] * ((p[6] * px + p[7] * py + p[8] * pz) + p[15] + p[12]);
        }
    }
}

// weighted Welford / Chan update of the listed chains' accumulators with the meshes X[j] (weight w, previous count n_old)
__global__ void __launch_bounds__(kStThreads) k_stats_update(ModelDev m, const double *__restrict__ X, const int *__restrict__ idx,
                                                             const int *__restrict__ count, const long long *__restrict__ w,
                                                             const long long *__restrict__ n_old, double *__restrict__ mean,
                                                             double *__restrict__ m2, double *__restrict__ nsum) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= m.N) return;
    const int n = *count;
    for (int j = blockIdx.y; j < n; j += gridDim.y) {
        const int c = idx[j];
        const double wd = (double)w[c], na = (double)n_old[c], nb = na + wd;
        const double f = wd / nb, g = wd * na / nb;
        const double *x = X + ((size_t)j * m.N + v) * 3;
        double *mu = mean + ((size_t)c * m.N + v) * 3;
        double *q = m2 + ((size_t)c * m.N + v) * 6;
        const double dx = x[0] - mu[0], dy = x[1] - mu[1], dz = x[2] - mu[2];
        mu[0] += f * dx; mu[1] += f * dy; mu[2] += f * dz;
        q[0] += g * (dx * dx); q[1] += g * (dy * dy); q[2] += g * (dz * dz);
        q[3] += g * (dx * dy); q[4] += g * (dx * dz); q[5] += g * (dy * dz);
        if (nsum) {
            double nx, ny, nz;
            vertex_normal_dev(m, X + (size_t)j * m.N * 3, v, nx, ny, nz);
            double *s = nsum + ((size_t)c * m.N + v) * 3;
            s[0] += wd * nx; s[1] += wd * ny; s[2] += wd * nz;
        }
    }
}

// read-out: the chains' pending weight as one more flush, on copies of the counts
__global__ void k_stats_pending(int C, const long long *__restrict__ pending, long long *__restrict__ count,
                                long long *__restrict__ w, long long *__restrict__ n_old) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const long long p = pending[c];
    w[c] = p;
    n_old[c] = count[c];
    count[c] += p;
}

// Chan's merge of C per-chain partials in chain order (deterministic); C == 1 returns that chain's partial exactly
__global__ void __launch_bounds__(kStThreads) k_stats_pool(int C, int N, const long long *__restrict__ count,
                                                           const double *__restrict__ mean, const double *__restrict__ m2,
                                                           const double *__restrict__ nsum, double *__restrict__ omean,
                                                           double *__restrict__ om2, double *__restrict__ onsum) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    double mu[3] = {0, 0, 0}, q[6] = {0, 0, 0, 0, 0, 0}, s[3] = {0, 0, 0}, na = 0.0;
    for (int c = 0; c < C; c++) {
        const long long cb = count[c];
        if (cb == 0) continue;
        const double nb = (double)cb, nn = na + nb, f = nb / nn, g = na * nb / nn;
        const double *mb = mean + ((size_t)c * N + v) * 3, *qb = m2 + ((size_t)c * N + v) * 6;
        const double d[3] = {mb[0] - mu[0], mb[1] - mu[1], mb[2] - mu[2]};
#pragma unroll
        for (int k = 0; k < 3; k++) mu[k] += f * d[k];
        q[0] += qb[0] + g * (d[0] * d[0]); q[1] += qb[1] + g * (d[1] * d[1]); q[2] += qb[2] + g * (d[2] * d[2]);
        q[3] += qb[3] + g * (d[0] * d[1]); q[4] += qb[4] + g * (d[0] * d[2]); q[5] += qb[5] + g * (d[1] * d[2]);
        if (nsum) {
            const double *sb = nsum + ((size_t)c * N + v) * 3;
#pragma unroll
            for (int k = 0; k < 3; k++) s[k] += sb[k];
        }
        na = nn;
    }
#pragma unroll
    for (int k = 0; k < 3; k++) omean[3 * (size_t)v + k] = mu[k];
#pragma unroll
    for (int k = 0; k < 6; k++) om2[6 * (size_t)v + k] = q[k];
    if (onsum)
#pragma unroll
        for (int k = 0; k < 3; k++) onsum[3 * (size_t)v + k] = s[k];
}

// mean out; tot7 = the layout k_var_finish reads: M2 (xx, yy, zz, xy, xz, yz) and d^T M2 d with d the reference normal or
// the mean unit normal normal_sum / S (as k_var_means forms it)
__global__ void k_stats_moments(int N, long long S, const double *__restrict__ mean, const double *__restrict__ m2,
                                const double *__restrict__ nsum, const double *__restrict__ ref_normals,
                                double *__restrict__ mean_out, double *__restrict__ tot7) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N) return;
    const double inv = 1.0 / (double)S;
    double d[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        mean_out[3 * (size_t)v + k] = mean[3 * (size_t)v + k];
        d[k] = ref_normals ? ref_normals[3 * (size_t)v + k] : nsum[3 * (size_t)v + k] * inv;
    }
    const double *q = m2 + 6 * (size_t)v;
    double *o = tot7 + 7 * (size_t)v;
#pragma unroll
    for (int k = 0; k < 6; k++) o[k] = q[k];
    o[6] = q[0] * d[0] * d[0] + q[1] * d[1] * d[1] + q[2] * d[2] * d[2] +
           2.0 * (q[3] * d[0] * d[1] + q[4] * d[0] * d[2] + q[5] * d[1] * d[2]);
}

}  // namespace

void launch_stats_flush(const ModelDev &m, int C, const double *d_theta, const long long *d_w, const long long *d_n_old,
                        int *d_idx, int *d_count, double *d_X, const StatsAcc &acc, cudaStream_t s) {
    if (C <= 0) return;
    k_stats_compact<<<1, 1024, 0, s>>>(C, d_w, d_idx, d_count);
    ICP_CUDA(cudaGetLastError());
    // the grids cover every chain; a CTA leaves at once when the list is shorter (the host does not know its length)
    const int vb = (m.N + kStThreads - 1) / kStThreads;
    const int gy_rec = std::max(1, std::min((C + kStCH - 1) / kStCH, std::max(1, 4096 / vb)));
    const size_t smem = sizeof(double) * ((size_t)m.K * kStCH + kStCH * 16);
    k_stats_reconstruct<<<dim3(vb, gy_rec), kStThreads, smem, s>>>(m, d_theta, d_idx, d_count, d_X);
    ICP_CUDA(cudaGetLastError());
    const int gy_upd = std::max(1, std::min(C, std::max(1, 8192 / vb)));
    k_stats_update<<<dim3(vb, gy_upd), kStThreads, 0, s>>>(m, d_X, d_idx, d_count, d_w, d_n_old, acc.mean, acc.m2, acc.nsum);
    ICP_CUDA(cudaGetLastError());
}

void launch_stats_pending(int C, const long long *d_pending, long long *d_count, long long *d_w, long long *d_n_old, cudaStream_t s) {
    if (C <= 0) return;
    k_stats_pending<<<(C + 127) / 128, 128, 0, s>>>(C, d_pending, d_count, d_w, d_n_old);
    ICP_CUDA(cudaGetLastError());
}

void launch_stats_pool(int C, int N, const long long *d_count, const StatsAcc &acc, double *d_mean, double *d_m2, double *d_nsum,
                       cudaStream_t s) {
    k_stats_pool<<<(N + kStThreads - 1) / kStThreads, kStThreads, 0, s>>>(C, N, d_count, acc.mean, acc.m2, acc.nsum, d_mean, d_m2, d_nsum);
    ICP_CUDA(cudaGetLastError());
}

void launch_stats_moments(int N, long long S, const double *d_mean, const double *d_m2, const double *d_nsum, const double *d_ref_normals,
                          double *d_mean_out, double *d_tot7, cudaStream_t s) {
    k_stats_moments<<<(N + kStThreads - 1) / kStThreads, kStThreads, 0, s>>>(N, S, d_mean, d_m2, d_nsum, d_ref_normals, d_mean_out, d_tot7);
    ICP_CUDA(cudaGetLastError());
}

}  // namespace icp
