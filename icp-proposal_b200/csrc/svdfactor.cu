// svdfactor.cu - the reference's own covariance factor of the ICP posterior, batched over chains.
//
// NonRigidIcpProposal.propose draws `posterior.sample()` (NonRigidIcpProposal.scala:55): Scalismo's posterior GP carries
// the eigen-decomposition of Sigma' = D M^-1 D (D = diag(sqrt(lambda)), SURVEY Appendix A4), so a standard-normal
// vector z maps to coefficients alpha = mu + W z with
//     W = D^-1 Ubar diag(sqrt(lambda')),      Sigma' = Ubar diag(lambda') Ubar^T,  lambda' descending.
// Any W with W W^T = M^-1 gives the same proposal distribution (the default factor is L^-T, one back substitution);
// this kernel produces the reference's factor so that a caller passing its own z gets the reference's sample.
//
// Method: with M = L L^T,  Sigma'^-1 = D^-1 M D^-1 = H^T H,  H = L^T D^-1 (upper triangular, no inversion needed).
// One-sided (Hestenes) Jacobi on the columns of H: right rotations accumulate J until the columns of H J are orthogonal;
// then J = Ubar and |column j|^2 = 1 / lambda'_j. One CTA per posterior, H and J column-major in shared memory, a warp
// per column pair, the pairs of a round dealt by the round-robin tournament schedule (every pair once per sweep).
// Order: lambda' descending (ties: lower column index first). Sign: the entry of largest magnitude of every vector is
// positive (lowest index on ties) - a documented convention of this library (the test checkers adopt it); what LAPACK's
// dgesdd would return inside Breeze is not knowable without a JVM.
#include <cmath>
#include <vector>

#include "icp_device.cuh"
#include "icp_internal.h"

namespace icp {

constexpr int kSvdThreads = 256;
constexpr int kSvdMaxSweeps = 40;
// a pair rotates while |a.b| > kSvdTol |a| |b|; the femur-like posteriors of rank 31 to 224 stop after 8 or 9 sweeps
// (tests/test_gpu_posterior_ranks.py::test_svd_factor asserts that the cap is not reached)
constexpr double kSvdTol = 1e-15;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(kSvdThreads) k_svd_factor(int K, int Kp, const double *__restrict__ L,
                                                            const double *__restrict__ sqrt_var,
                                                            const int *__restrict__ slot, double *__restrict__ W,
                                                            double *__restrict__ scratch, int mats_in_smem, double tol,
                                                            int *__restrict__ sweeps) {
    extern __shared__ __align__(16) double sm[];
    __shared__ double s_n2[256];     // squared column norms (K <= 224)
    __shared__ int s_rank[256];
    __shared__ double s_sgn[256];
    const int c = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = kSvdThreads / 32;
    const int ld = Kp;
    const size_t KK = (size_t)Kp * Kp;
    // H and J: shared memory when they fit (both at Kp <= 112), else the per-chain scratch in global memory (the
    // __syncthreads between rounds orders the block's global accesses as well)
    double *G = mats_in_smem >= 1 ? sm : scratch + (size_t)c * 2 * KK;
    double *J = mats_in_smem >= 2 ? sm + KK : scratch + (size_t)c * 2 * KK + KK;
    const int sl = slot ? slot[c] : c;
    const double *Lc = L + (size_t)sl * KK;
    // H[i][j] = L[j][i] / sqrt(lambda_j) for i <= j (column j of H = row j of L, scaled); column-major: G[j * ld + i]
    for (int e = tid; e < Kp * Kp; e += kSvdThreads) {
        const int j = e / Kp, i = e - j * Kp;
        G[(size_t)j * ld + i] = (i <= j && j < K && i < K) ? Lc[(size_t)j * Kp + i] / sqrt_var[j] : 0.0;
        J[(size_t)j * ld + i] = i == j ? 1.0 : 0.0;
    }
    __syncthreads();
    const int n = (K + 1) & ~1;       // tournament size (even); an index >= K is a bye
    int sweep = 0;                    // sweeps that rotated; kSvdMaxSweeps: the cap ended the loop
    for (; sweep < kSvdMaxSweeps; sweep++) {
        int rotated = 0;
        for (int r = 0; r < n - 1; r++) {
            for (int k = warp; k < n / 2; k += nw) {
                int p, q;
                if (k == 0) { p = n - 1; q = r; }
                else { p = (r + k) % (n - 1); q = (r - k + (n - 1)) % (n - 1); }
                if (p >= K || q >= K) continue;
                if (p > q) { const int t = p; p = q; q = t; }
                double *a = G + (size_t)p * ld, *b = G + (size_t)q * ld;
                double aa = 0.0, bb = 0.0, ab = 0.0;
                for (int i = lane; i < K; i += 32) {
                    const double x = a[i], y = b[i];
                    aa = fma(x, x, aa); bb = fma(y, y, bb); ab = fma(x, y, ab);
                }
                aa = warp_sum(aa); bb = warp_sum(bb); ab = warp_sum(ab);
                if (fabs(ab) > tol * sqrt(aa * bb)) {
                    const double zeta = (bb - aa) / (2.0 * ab);
                    const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    const double cs = 1.0 / sqrt(1.0 + t * t), sn = cs * t;
                    double *ja = J + (size_t)p * ld, *jb = J + (size_t)q * ld;
                    for (int i = lane; i < K; i += 32) {
                        const double x = a[i], y = b[i];
                        a[i] = cs * x - sn * y; b[i] = sn * x + cs * y;
                        const double u = ja[i], v = jb[i];
                        ja[i] = cs * u - sn * v; jb[i] = sn * u + cs * v;
                    }
                    rotated = 1;
                }
            }
            __syncthreads();
        }
        if (!__syncthreads_or(rotated)) break;
    }
    if (sweeps && tid == 0) sweeps[c] = sweep;
    // column norms, sign of every vector
    for (int j = warp; j < K; j += nw) {
        const double *g = G + (size_t)j * ld, *u = J + (size_t)j * ld;
        double s = 0.0, vm = -1.0;
        int im = 0x7fffffff;
        for (int i = lane; i < K; i += 32) {
            s = fma(g[i], g[i], s);
            const double av = fabs(u[i]);
            if (av > vm) { vm = av; im = i; }     // ascending i: the first maximum of this lane
        }
        s = warp_sum(s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, vm, o);
            const int oi = __shfl_xor_sync(0xffffffffu, im, o);
            if (ov > vm || (ov == vm && oi < im)) { vm = ov; im = oi; }
        }
        if (lane == 0) { s_n2[j] = s; s_sgn[j] = (im < K && u[im] < 0.0) ? -1.0 : 1.0; }
    }
    __syncthreads();
    // lambda'_j = 1 / |g_j|^2 descending = |g_j|^2 ascending
    for (int j = tid; j < K; j += kSvdThreads) {
        const double v = s_n2[j];
        int rk = 0;
        for (int k = 0; k < K; k++) { const double o = s_n2[k]; rk += (o < v || (o == v && k < j)) ? 1 : 0; }
        s_rank[j] = rk;
    }
    __syncthreads();
    // W[i][rank_j] = sgn_j Ubar[i][j] sqrt(lambda'_j) / sqrt(lambda_i); zero on the padding
    double *Wc = W + (size_t)sl * KK;
    for (int e = tid; e < Kp * Kp; e += kSvdThreads) {
        const int j = e / Kp, i = e - j * Kp;
        if (j < K && i < K) Wc[(size_t)i * Kp + s_rank[j]] = s_sgn[j] * J[(size_t)j * ld + i] / (sqrt(s_n2[j]) * sqrt_var[i]);
        else Wc[(size_t)i * Kp + j] = 0.0;
    }
}

void launch_svd_factor(int C, int K, int Kp, const double *d_L, const double *d_sqrt_var, const int *d_slot, double *d_W,
                       DevBuf<double> &scratch, cudaStream_t s, double tol, int *d_sweeps) {
    if (C <= 0) return;
    ProfScope _ps(ST_OTHER, s);
    ICP_REQUIRE(K <= 256, "rank too large for the SVD factor kernel");
    const size_t KK = (size_t)Kp * Kp;
    int mats = 2;
    if (sizeof(double) * 2 * KK > 200 * 1024) mats = 1;
    if (sizeof(double) * KK > 200 * 1024) mats = 0;
    if (mats < 2) scratch.ensure((size_t)C * 2 * KK);
    const size_t smem = sizeof(double) * KK * mats;
    ICP_CUDA(cudaFuncSetAttribute(k_svd_factor, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_svd_factor<<<C, kSvdThreads, smem, s>>>(K, Kp, d_L, d_sqrt_var, d_slot, d_W, scratch.p, mats, tol > 0.0 ? tol : kSvdTol,
                                              d_sweeps);
    ICP_CUDA(cudaGetLastError());
}

}  // namespace icp

// The SVD factor of C posteriors from their Cholesky factors (host, C x K x K, lower triangle read) and the model variances:
// W (C x K x K) and the Jacobi sweeps that rotated per posterior (kSvdMaxSweeps: the cap ended the loop). tol <= 0: the
// pipeline's threshold.
extern "C" int32_t icp_debug_svd_factor(icp_ctx ctx, int32_t C, int32_t K, const double *L, const double *variance, double tol,
                                        double *W, int32_t *sweeps) {
    using namespace icp;
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx && C > 0 && K >= 1 && K <= 224 && L && variance && W && sweeps, "null or empty argument");
        for (int j = 0; j < K; j++) ICP_REQUIRE(variance[j] > 0.0 && std::isfinite(variance[j]), "variances must be finite and > 0");
        CtxLock lock(ctx);
        cudaStream_t s = ctx->stream;
        const int Kp = (K + 7) / 8 * 8;
        std::vector<double> hL((size_t)C * Kp * Kp, 0.0), hs(Kp, 1.0), hW((size_t)C * Kp * Kp);
        for (int c = 0; c < C; c++)
            for (int i = 0; i < K; i++)
                for (int j = 0; j <= i; j++) hL[((size_t)c * Kp + i) * Kp + j] = L[((size_t)c * K + i) * K + j];
        for (int j = 0; j < K; j++) hs[j] = std::sqrt(variance[j]);
        DevBuf<double> dL, ds, dW, scratch;
        DevBuf<int> dsw;
        dL.upload(hL.data(), hL.size(), s);
        ds.upload(hs.data(), hs.size(), s);
        dW.alloc(hW.size());
        dsw.alloc(C);
        launch_svd_factor(C, K, Kp, dL.p, ds.p, nullptr, dW.p, scratch, s, tol, dsw.p);
        ICP_CUDA(cudaMemcpyAsync(hW.data(), dW.p, sizeof(double) * hW.size(), cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaMemcpyAsync(sweeps, dsw.p, sizeof(int) * C, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        for (int c = 0; c < C; c++)
            for (int i = 0; i < K; i++)
                for (int j = 0; j < K; j++) W[((size_t)c * K + i) * K + j] = hW[((size_t)c * Kp + i) * Kp + j];
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}
