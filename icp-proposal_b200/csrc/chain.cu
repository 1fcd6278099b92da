// chain.cu - device-resident Metropolis-Hastings runner for C independent chains.
//
// Replaces the per-step work of Scalismo's MetropolisHastings.next + MixtureProposal as driven from
// api/sampling/SamplingRegistration.scala:52-85 (SURVEY.md section 3.1 and Appendix A8/A9):
//   currentP   = evaluator.logValue(current)          kept resident per chain (EvaluationCaching.scala:32-36)
//   proposal   = generator.propose(current)           k_chain_propose: mixture pick + component proposal
//   proposalP  = evaluator.logValue(proposal)         reconstruct + evaluator pipeline
//   t          = logTransitionRatio(current, proposal) ICP posteriors of the proposal + k_chain_accept
//   accept iff a > 0 or U < exp(a)                     k_chain_accept, chain log append
// The posterior of the current state of every ICP component stays resident per chain (the reference's
// Memoize(icpPosterior, 20), NonRigidIcpProposal.scala:49), so each step builds one new posterior per
// ICP component - for the proposed state.
#include <cmath>
#include <cstring>
#include <functional>
#include <map>
#include <unordered_map>

#include "icp_device.cuh"
#include "icp_internal.h"

using namespace icp;

namespace {

constexpr int kMaxComp = 16;
constexpr int kMaxNBc = 28;   // Kp <= 224 (icp_model_create enforces it)

struct CompDev {
    int kind, axis, icp_index;  // icp_index: which ICP posterior set (or -1)
    int factor;                 // ICP components: ICP_FACTOR_CHOLESKY | ICP_FACTOR_SVD
    double cdf, weight, sd, step;
};

struct ChainParams {
    int n_comp, n_icp, K, Kp, C;
    // Rejection look-ahead (see k_la_resolve): W > 1 lanes per chain. C then counts the lanes (C = Cr * W; lane-major: lane v is
    // lane v / Cr of chain v % Cr, so the first Cr * Wa entries are the lanes 0 .. Wa - 1 of every chain) and every per-chain
    // array of StateDev is per lane, except step / n_acc / status / theta_best / value_best. Wa <= W lanes are active in this
    // round (the kernels are launched over Cr * Wa lanes; C stays the stride of the per-lane arrays).
    int W, Cr, Wa;
    CompDev comp[kMaxComp];
};

struct RngDev {
    unsigned long long seed, chain_offset;
    const double *u_comp, *z, *u_acc;  // host-RNG mode when non-null: [step][C], [step][C][K], [step][C]
    int step_base;
};

struct LogDev {
    int *comp;
    uint8_t *accepted;
    double *values;  // [step][C][3]
    double *theta;   // [step][C][L]
    int step_base;   // record index = step - step_base (resumed runs keep counting steps for the RNG)
};

// posterior variability accumulated inside the run (icp_chain_set_statistics, stats.cu); every pointer is null when off.
// Per chain (look-ahead: per chain, not per lane): the selected records at which the current state was current and that
// are not in the accumulators yet, and what the current step / round flushed into them.
struct StatsDev {
    long long *pending;      // [Cr]
    long long *count;        // [Cr] samples in the accumulators
    long long *flush_w;      // [Cr] weight flushed by this step / round (0: none)
    long long *flush_n;      // [Cr] count before that flush
    double *flush_theta;     // [Cr][L] the flushed state
    long long burn_in, every, end;
};

__device__ __forceinline__ int stats_selected(const StatsDev &x, long long i) {
    return i >= x.burn_in && (x.end <= 0 || i < x.end) && (i - x.burn_in) % x.every == 0;
}

struct StateDev {
    double *theta_cur, *theta_prop;     // [C][L]
    double *values_cur, *values_prop;   // [C][3]
    int *cur_sel;                       // [C] which posterior state (0/1) is current
    int *slot_cur, *slot_prop;          // [C] = sel * C + c
    int *comp_sel;                      // [C] component picked this step
    double *u_acc;                      // [C]
    long long *n_acc;                   // [C]
    int *step;                          // [1] device step counter
    // [n_icp][2 C][Kp Kp], [n_icp][2 C][Kp]: L and the whitened mean y = L^-1 b = L^T mu of each posterior (ICP_FACTOR_SVD
    // components: mu itself, which their factor W needs)
    double *L, *ymean;
    double *W;                          // [n_icp][2 C][Kp Kp] the reference's SVD factor (ICP_FACTOR_SVD components; else null)
    int *status;                        // [C] sticky per-chain status bits (kSt*)
    double *theta_best, *value_best;    // [C][L], [C]: BestSampleLogger - the state with the largest product value so far
    // |L^T d|^2 of every ICP component's forward (posterior of the current state, formed by k_chain_propose while it holds
    // L_cur) and backward (posterior of the proposal, formed in the factorisation's epilogue) transition: [n_icp][C]
    double *qf, *qb;
    // look-ahead only: the lanes' accept decisions and status words of this round, the first step the run must not take
    int *lane_ok, *lane_status, *step_end;
    StatsDev sx;
};

// per-chain status bits of a run (icp_chain_io.status)
constexpr int kStEmptySet = 1;      // the collective evaluator's filtered distance list was empty (the reference throws)
constexpr int kStNotPD = 2;         // a posterior's M was not positive definite
constexpr int kStNanTransition = 4; // a mixture component returned a NaN transition density (Scalismo's mixture throws)
constexpr int kStNanValue = 8;      // the evaluator returned NaN for the initial state

// where the pipelines of the step leave their per-chain status words
struct StatusSrc {
    const int *eval;              // [C] ICP_OK | ICP_ERR_EMPTY_SET
    const int *post[kMaxComp];    // per ICP component [C], 0 = ok
    int n_post;
};

__device__ __forceinline__ int fold_status(const StatusSrc &ss, int c) {
    int st = 0;
    if (ss.eval && ss.eval[c] != 0) st |= kStEmptySet;
    for (int i = 0; i < ss.n_post; i++)
        if (ss.post[i] && ss.post[i][c] != 0) st |= kStNotPD;
    return st;
}

// status of the initial state (theta0): evaluator / posterior status words + a NaN log-value
__global__ void k_chain_status0(int C, int Lt, StateDev st, StatusSrc ss) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    int v = fold_status(ss, c);
    const double p = st.values_cur[3 * c];
    if (p != p) v |= kStNanValue;
    st.status[c] = v;
    // Scalismo's chain iterator yields the initial state first, so BestSampleLogger starts from it
    st.value_best[c] = p;
    for (int j = 0; j < Lt; j++) st.theta_best[(size_t)c * Lt + j] = st.theta_cur[(size_t)c * Lt + j];
}

__global__ void k_chain_init(int C, StateDev st) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0) *st.step = 0;
    if (c >= C) return;
    st.cur_sel[c] = 0;
    st.slot_cur[c] = c;
    st.slot_prop[c] = C + c;
    st.n_acc[c] = 0;
    st.status[c] = 0;
}

// standard normals of chain `chain` at step `step`: Philox block 1 + k/2 -> Box-Muller pair
__device__ __forceinline__ double chain_normal(unsigned long long seed, unsigned long long chain, unsigned int step, int k) {
    uint4 r = chain_philox(seed, chain, step, 1u + (unsigned int)(k >> 1));
    double u1 = 1.0 - u53(r.x, r.y);  // (0, 1]
    double u2 = u53(r.z, r.w);
    double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    return (k & 1) ? rad * sn : rad * cs;
}

// w = L^-T z, one warp, registers + shuffles; L staged in shared memory with
// the lower triangle packed row-major (row i at offset i (i + 1) / 2); the diagonal entries have been replaced
// by their reciprocals (one parallel division per row instead of a division on every step of the serial chain)
__device__ void warp_backsolve_packed(const double *sL, int Kp, const double *z_sm, double *w_sm) {
    int lane = threadIdx.x & 31;
    double zr[8];
#pragma unroll
    for (int q = 0; q < 8; q++) { int k = lane + 32 * q; zr[q] = k < Kp ? z_sm[k] : 0.0; }
    for (int i = Kp - 1; i >= 0; i--) {
        const double *row = sL + (i * (i + 1)) / 2;
        int owner = i & 31, slot = i >> 5;
        double zi = 0.0;
#pragma unroll
        for (int q = 0; q < 8; q++) if (q == slot) zi = zr[q];
        double wi = __shfl_sync(0xffffffffu, zi, owner) * row[i];
        if (lane == 0) w_sm[i] = wi;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            int k = lane + 32 * q;
            if (k < i) zr[q] = fma(-row[k], wi, zr[q]);
        }
    }
    __syncwarp();
}

// lower triangle of L (row-major Kp x Kp in global memory) -> packed row-major in shared memory (row i at i (i + 1) / 2):
// warps take rows, lanes take columns
__device__ __forceinline__ void stage_packed_L(const double *__restrict__ Lc, int Kp, double *sL) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int i0 = warp; i0 < Kp; i0 += 4 * nw) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
            int i = i0 + r * nw;
            if (i < Kp) {
                const double *src = Lc + (size_t)i * Kp;
                double *dst = sL + (i * (i + 1)) / 2;
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    int j = lane + 32 * q;
                    if (j <= i) dst[j] = __ldg(src + j);
                }
            }
        }
    }
}

// |L^T d - y|^2 (y nullable: |L^T d|^2) with the packed lower triangle and d in shared memory: thread j owns column j (for a
// fixed row the threads read consecutive words); result valid in every thread
__device__ __forceinline__ double block_quad_packed(const double *sL, int Kp, const double *d_sm, double *red,
                                                    const double *__restrict__ y) {
    double part = 0.0;
    for (int j = threadIdx.x; j < Kp; j += blockDim.x) {
        double v0 = 0.0, v1 = 0.0;
        int i = j;
        for (; i + 1 < Kp; i += 2) {
            v0 = fma(sL[(i * (i + 1)) / 2 + j], d_sm[i], v0);
            v1 = fma(sL[((i + 1) * (i + 2)) / 2 + j], d_sm[i + 1], v1);
        }
        if (i < Kp) v0 = fma(sL[(i * (i + 1)) / 2 + j], d_sm[i], v0);
        const double v = y ? (v0 + v1) - y[j] : v0 + v1;
        part = fma(v, v, part);
    }
    return block_sum(part, red);
}

// MixtureProposal.propose (pick the first component whose cumulative weight reaches r) + the component's propose, then the
// forward transition form |L_cur^T d|^2 of EVERY ICP component (MixtureProposal.logTransitionProbability sums over all of
// them): the factors of the current state are staged here anyway, so k_chain_accept never reads a factor back.
__global__ void __launch_bounds__(256) k_chain_propose(ChainParams P, ModelDev m, StateDev st, RngDev rng) {
    extern __shared__ double sm[];
    const int K = P.K, Kp = P.Kp, Lt = K + kTheta0, C = P.C;
    // sz: z (+ y) | sw: v = L^-T (y + z) (SVD factor: mu + W z) | sdl: alpha' - alpha | sd: transition argument |
    // sdg: diagonal of the staged factor |
    // part: 2 Kp partial sums of S v | red: block reduction | sL: packed lower triangle
    double *sz = sm, *sw = sm + Kp, *sdl = sm + 2 * Kp, *sd = sm + 3 * Kp, *sdg = sm + 4 * Kp, *part = sm + 5 * Kp, *red = sm + 7 * Kp,
           *sL = sm + 7 * Kp + 40;
    __shared__ int s_ci;
    int c = blockIdx.x;
    // look-ahead: lane c proposes step step[chain] + lane index of chain c / W from the chain's current state; the randomness
    // of a step is a function of (seed, chain, step) only, so this is the proposal the sequential chain makes at that step
    // if every step before it is rejected. Lanes past the end of the run repeat the last step (ignored by k_la_resolve).
    const int cr = P.W > 1 ? c % P.Cr : c, Cr = P.W > 1 ? P.Cr : C;
    unsigned int step = (unsigned int)*st.step;
    if (P.W > 1) {
        int sv = st.step[cr] + c / P.Cr;
        const int last = *st.step_end - 1;
        step = (unsigned int)(sv > last ? last : sv);
    }
    unsigned long long chain = rng.chain_offset + (unsigned long long)cr;
    if (threadIdx.x == 0) {
        double uc, ua;
        if (rng.u_comp) {
            uc = rng.u_comp[(size_t)(step - rng.step_base) * Cr + cr];
            ua = rng.u_acc[(size_t)(step - rng.step_base) * Cr + cr];
        } else {
            uint4 r = chain_philox(rng.seed, chain, step, 0u);
            uc = u53(r.x, r.y);
            ua = u53(r.z, r.w);
        }
        int ci = P.n_comp - 1;
        for (int i = 0; i < P.n_comp; i++)
            if (P.comp[i].cdf >= uc) { ci = i; break; }
        s_ci = ci;
        st.comp_sel[c] = ci;
        st.u_acc[c] = ua;
    }
    for (int k = threadIdx.x; k < Kp; k += blockDim.x) {
        double zz = 0.0;
        if (k < K) zz = rng.z ? rng.z[((size_t)(step - rng.step_base) * Cr + cr) * K + k] : chain_normal(rng.seed, chain, step, k);
        sz[k] = zz;
    }
    __syncthreads();
    const CompDev cd = P.comp[s_ci];
    const double *th = st.theta_cur + (size_t)c * Lt;
    double *to = st.theta_prop + (size_t)c * Lt;
    bool staged = false;   // sL holds the selected component's factor (diagonal inverted, true diagonal in sdg)
    if (cd.kind == ICP_PROP_ICP) {
        size_t pslot = (size_t)cd.icp_index * 2 * C + st.slot_cur[c];
        const double *Lc = st.L + pslot * Kp * Kp, *mean = st.ymean + pslot * Kp;
        if (cd.factor == ICP_FACTOR_SVD) {
            // the reference's factor W = D^-1 Ubar diag(sqrt(lambda')) of the current state's posterior (svdfactor.cu); the
            // mean slot of an SVD component holds mu: v = mu + W z
            block_matvec_rows(st.W + pslot * Kp * Kp, Kp, sz, sw);
            __syncthreads();
            for (int k = threadIdx.x; k < Kp; k += blockDim.x) sw[k] = mean[k] + sw[k];
        } else {
            // v = mu + L^-T z = L^-T (y + z): one back substitution
            for (int k = threadIdx.x; k < Kp; k += blockDim.x) sz[k] += mean[k];
            stage_packed_L(Lc, Kp, sL);
            __syncthreads();
            for (int i = threadIdx.x; i < Kp; i += blockDim.x) { double *d = sL + (i * (i + 1)) / 2 + i; sdg[i] = *d; *d = 1.0 / *d; }
            __syncthreads();
            if (threadIdx.x < 32) warp_backsolve_packed(sL, Kp, sz, sw);
            staged = true;
        }
        __syncthreads();
        // S v with S symmetric (read column-wise, coalesced); two halves of the k range per output
        for (int idx = threadIdx.x; idx < 2 * Kp; idx += blockDim.x) {
            int jj = idx % Kp, half = idx / Kp;
            int k0 = half * (Kp / 2), k1 = half ? Kp : Kp / 2;
            double acc = 0.0;
#pragma unroll 8
            for (int k = k0; k < k1; k++) acc = fma(__ldg(&m.S[(size_t)k * Kp + jj]), sw[k], acc);
            part[idx] = acc;
        }
        __syncthreads();
        for (int j = threadIdx.x; j < Lt; j += blockDim.x) {
            double v = th[j];
            if (j >= kTheta0) {
                int jj = j - kTheta0;
                double acc = part[jj] + part[Kp + jj];
                v = th[j] + (acc - th[j]) * cd.step;  // NonRigidIcpProposal.scala:61-62
                sdl[jj] = v - th[j];
            }
            to[j] = v;
        }
    } else {
        for (int j = threadIdx.x; j < Lt; j += blockDim.x) {
            double v = th[j];
            if (cd.kind == ICP_PROP_RANDOM_SHAPE) {
                if (j >= kTheta0) v = th[j] + cd.sd * sz[j - kTheta0];   // RandomShapeUpdateProposal.scala:34-35
            } else if (cd.kind == ICP_PROP_ROTATION) {
                if (j == 4 + cd.axis) v = th[j] + cd.sd * sz[0];         // PoseProposals.scala:36-44
            } else {
                if (j == 1 + cd.axis) v = th[j] + cd.sd * sz[0];         // PoseProposals.scala:70-78
            }
            to[j] = v;
            if (j >= kTheta0) sdl[j - kTheta0] = v - th[j];
        }
    }
    __syncthreads();
    // forward forms |L_cur,i^T d|^2, d = (alpha + (alpha' - alpha) / step_i) - mu_cur,i   (NonRigidIcpProposal.scala:79, :82-83),
    // formed as |L_cur,i^T s - y_cur,i|^2 with s = alpha + (alpha' - alpha) / step_i (SVD-factor components: d itself, from mu)
    // The selected component goes first when its factor is still staged: the other components stage theirs over it. (Taking
    // the components in index order formed the selected component's form from an overwritten factor whenever an ICP
    // component with a smaller index came before it - invisible next to a random-walk component, whose density dominates
    // the mixture's at these step sizes, and wrong in an ICP-only mixture: tools/check_forward_forms.py.)
    for (int pass = 0; pass < P.n_comp + 1; pass++) {
        const int i = pass == 0 ? s_ci : pass - 1;
        if (pass == 0 && !staged) continue;
        if (pass > 0 && staged && i == s_ci) continue;
        const CompDev ci = P.comp[i];
        if (ci.kind != ICP_PROP_ICP) continue;
        const size_t pslot = (size_t)ci.icp_index * 2 * C + st.slot_cur[c];
        if (pass == 0) {
            for (int k = threadIdx.x; k < Kp; k += blockDim.x) sL[(k * (k + 1)) / 2 + k] = sdg[k];   // the true diagonal again
        } else {
            stage_packed_L(st.L + pslot * Kp * Kp, Kp, sL);
        }
        const double *mean = st.ymean + pslot * Kp;
        const bool ym = ci.factor != ICP_FACTOR_SVD;
        for (int k = threadIdx.x; k < Kp; k += blockDim.x) {
            const double s = k < K ? th[kTheta0 + k] + (sdl[k] / ci.step) : 0.0;
            sd[k] = ym ? s : k < K ? s - mean[k] : 0.0;
        }
        __syncthreads();
        const double qf = block_quad_packed(sL, Kp, sd, red, ym ? mean : nullptr);
        if (threadIdx.x == 0) st.qf[(size_t)ci.icp_index * C + c] = qf;
        __syncthreads();
    }
}

__device__ __forceinline__ double gauss1_logpdf(double x, double sd) {
    return -(x * x) / (2.0 * sd * sd) - log(sd * sqrt(2.0 * 3.14159265358979323846));
}

// log transition densities of every mixture component in both directions, log-sum-exp, acceptance, log append
__global__ void __launch_bounds__(128) k_chain_accept(ChainParams P, StateDev st, LogDev lg, StatusSrc stsrc) {
    extern __shared__ double sm[];
    const int K = P.K, Kp = P.Kp, Lt = K + kTheta0, C = P.C;
    double *red = sm;
    __shared__ double s_fwd[kMaxComp], s_bwd[kMaxComp];
    __shared__ int s_flags[3];  // [0] any of theta[0..9] differs, [1] outside rotation group, [2] outside translation group
    int c = blockIdx.x;
    int step = *st.step;
    const double *cur = st.theta_cur + (size_t)c * Lt, *prp = st.theta_prop + (size_t)c * Lt;
    if (threadIdx.x < 3) s_flags[threadIdx.x] = 0;
    __syncthreads();
    // equality guards (ModelFittingParameters equality is element-wise on allParameters)
    for (int j = threadIdx.x; j < Lt; j += blockDim.x) {
        bool diff = !(cur[j] == prp[j]);
        if (diff) {
            if (j < kTheta0) s_flags[0] = 1;
            if (!(j >= 4 && j <= 6)) s_flags[1] = 1;
            if (!(j >= 1 && j <= 3)) s_flags[2] = 1;
        }
    }
    __syncthreads();
    double ss = 0.0;  // |alpha' - alpha|^2 for the random-walk components
    for (int k = threadIdx.x; k < K; k += blockDim.x) { double r = prp[kTheta0 + k] - cur[kTheta0 + k]; ss = fma(r, r, ss); }
    ss = block_sum(ss, red);
    for (int i = 0; i < P.n_comp; i++) {
        const CompDev cd = P.comp[i];
        double fwd, bwd;
        if (cd.kind == ICP_PROP_ICP) {
            if (s_flags[0]) { fwd = bwd = -INFINITY; }                          // NonRigidIcpProposal.scala:72-74
            else {
                // the two quadratic forms were formed where the factors were on chip: forward by k_chain_propose (L_cur),
                // backward by the factorisation of the proposal's posterior (L_prop)
                const double qf = st.qf[(size_t)cd.icp_index * C + c], qb = st.qb[(size_t)cd.icp_index * C + c];
                fwd = -0.5 * (K * ICP_LOG_2PI + qf);
                bwd = -0.5 * (K * ICP_LOG_2PI + qb);
            }
        } else if (cd.kind == ICP_PROP_RANDOM_SHAPE) {
            if (s_flags[0]) fwd = bwd = -INFINITY;                               // RandomShapeUpdateProposal.scala:39
            else fwd = bwd = -0.5 * (K * ICP_LOG_2PI + K * log(cd.sd * cd.sd) + ss / (cd.sd * cd.sd));
        } else if (cd.kind == ICP_PROP_ROTATION) {
            if (s_flags[1]) fwd = bwd = -INFINITY;                               // PoseProposals.scala:48
            else { double r = prp[4 + cd.axis] - cur[4 + cd.axis]; fwd = bwd = gauss1_logpdf(r, cd.sd); }
        } else {
            if (s_flags[2]) fwd = bwd = -INFINITY;                               // PoseProposals.scala:82
            else { double r = prp[1 + cd.axis] - cur[1 + cd.axis]; fwd = bwd = gauss1_logpdf(r, cd.sd); }
        }
        if (threadIdx.x == 0) { s_fwd[i] = fwd; s_bwd[i] = bwd; }
    }
    __syncthreads();
    __shared__ int s_acc;
    if (threadIdx.x == 0) {
        // MixtureProposal.logTransitionProbability: ln sum_i w_i exp(l_i)
        double mf = -INFINITY, mb = -INFINITY;
        bool nan = false;
        for (int i = 0; i < P.n_comp; i++) {
            mf = fmax(mf, s_fwd[i]); mb = fmax(mb, s_bwd[i]);
            if (s_fwd[i] != s_fwd[i] || s_bwd[i] != s_bwd[i]) nan = true;
        }
        double lf = -INFINITY, lb = -INFINITY;
        if (mf > -INFINITY) { double s = 0; for (int i = 0; i < P.n_comp; i++) s += P.comp[i].weight * exp(s_fwd[i] - mf); lf = log(s) + mf; }
        if (mb > -INFINITY) { double s = 0; for (int i = 0; i < P.n_comp; i++) s += P.comp[i].weight * exp(s_bwd[i] - mb); lb = log(s) + mb; }
        double t = lf - lb;
        double vp = st.values_prop[3 * c], vc = st.values_cur[3 * c];
        double a = vp - vc - t;                                                   // MetropolisHastings.next
        int ok = (!nan) && ((a > 0.0) || (st.u_acc[c] < exp(a)));
        s_acc = ok;
        // the reference throws where these happen (CollectiveAverage...Evaluator.scala:51,63; Scalismo's mixture on a NaN
        // transition); here the step is rejected and the chain's sticky status word records it
        const int stw = fold_status(stsrc, c) | (nan ? kStNanTransition : 0);
        if (P.W > 1) { st.lane_ok[c] = ok; st.lane_status[c] = stw; }   // k_la_resolve decides which lanes happened
        else if (stw) st.status[c] |= stw;
    }
    __syncthreads();
    if (P.W > 1) return;
    int ok = s_acc;
    if (st.sx.pending) {
        // statistics: an accepting chain flushes its old state with the selected records at which it was current; this
        // step's record belongs to the state that is current after it
        __shared__ int s_flush;
        if (threadIdx.x == 0) {
            const long long pend = st.sx.pending[c];
            const int sel = stats_selected(st.sx, step);
            const int flush = ok && pend > 0;
            st.sx.flush_w[c] = flush ? pend : 0;
            if (flush) { st.sx.flush_n[c] = st.sx.count[c]; st.sx.count[c] += pend; }
            st.sx.pending[c] = ok ? sel : pend + sel;
            s_flush = flush;
        }
        __syncthreads();
        if (s_flush)
            for (int j = threadIdx.x; j < Lt; j += blockDim.x) st.sx.flush_theta[(size_t)c * Lt + j] = cur[j];
        __syncthreads();
    }
    if (ok) {
        for (int j = threadIdx.x; j < Lt; j += blockDim.x) st.theta_cur[(size_t)c * Lt + j] = prp[j];
        if (threadIdx.x < 3) st.values_cur[3 * c + threadIdx.x] = st.values_prop[3 * c + threadIdx.x];
    }
    __syncthreads();
    // chain log: the state that is current after the step (JSONAcceptRejectLogger.scala:93-106)
    size_t rec = (size_t)(step - lg.step_base) * C + c;
    if (lg.theta)
        for (int j = threadIdx.x; j < Lt; j += blockDim.x) lg.theta[rec * Lt + j] = ok ? prp[j] : cur[j];
    // BestSampleLogger.logState on the state that is current after the step (a rejected step re-offers the retained state,
    // which cannot beat itself)
    if (ok && st.values_prop[3 * c] > st.value_best[c]) {
        for (int j = threadIdx.x; j < Lt; j += blockDim.x) st.theta_best[(size_t)c * Lt + j] = prp[j];
        __syncthreads();
        if (threadIdx.x == 0) st.value_best[c] = st.values_prop[3 * c];
    }
    if (threadIdx.x == 0) {
        if (ok) {
            int sel = 1 - st.cur_sel[c];
            st.cur_sel[c] = sel;
            st.slot_cur[c] = sel * C + c;
            st.slot_prop[c] = (1 - sel) * C + c;
            st.n_acc[c] += 1;
        }
        if (lg.comp) lg.comp[rec] = st.comp_sel[c];
        if (lg.accepted) lg.accepted[rec] = (uint8_t)ok;
        if (lg.values) {
            const double *v = ok ? st.values_prop + 3 * c : st.values_cur + 3 * c;
            lg.values[3 * rec] = v[0]; lg.values[3 * rec + 1] = v[1]; lg.values[3 * rec + 2] = v[2];
        }
    }
}

__global__ void k_step_increment(int *step) { *step += 1; }

// ---- rejection look-ahead ("prefetching" Metropolis-Hastings) ---------------------------------------------------------
// A single chain is a chain of dependent latencies (SamplingRegistration.scala:60-85 is sequential), but a REJECTED step leaves
// the state where it was, and the randomness of step s is a function of (seed, chain, s) alone. So W lanes evaluate the
// proposals of steps s, s + 1, .., s + W - 1 from the same current state in one batched round - exactly what the sequential
// chain computes at those steps as long as everything before is rejected. k_la_resolve then walks the lanes in step order:
// lanes before the first accepting one are the chain's rejected steps (logged as such), the first accepting lane is its next
// accepted step, the lanes after it are discarded (their steps are proposed again, from the new state, in the next round).
// The chain log is bit-identical to the sequential runner's; a round costs the latency of one step and consumes
// (1 - (1 - a)^W) / a steps at acceptance rate a (2.4 at a = 0.4, W = 8).
__global__ void k_la_init(int Cr, int W, int Lt, const double *__restrict__ theta0, StateDev st) {
    const int Cv = Cr * W;
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < Cr) { st.step[v] = 0; st.n_acc[v] = 0; st.status[v] = 0; }
    if (v >= Cv) return;
    st.cur_sel[v] = 0;
    st.slot_cur[v] = v;
    st.slot_prop[v] = Cv + v;
    const double *src = theta0 + (size_t)(v % Cr) * Lt;
    for (int j = 0; j < Lt; j++) st.theta_cur[(size_t)v * Lt + j] = src[j];
}

__global__ void k_la_set_end(int *step_end, int value) { *step_end = value; }

// status / best sample of the initial state from lane 0 of every chain (all lanes hold the same state)
__global__ void k_la_status0(int Cr, int W, int Lt, StateDev st, StatusSrc ss) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Cr) return;
    const int v = c;   // lane 0
    int s = fold_status(ss, v);
    const double p = st.values_cur[3 * v];
    if (p != p) s |= kStNanValue;
    st.status[c] = s;
    st.value_best[c] = p;
    for (int j = 0; j < Lt; j++) st.theta_best[(size_t)c * Lt + j] = st.theta_cur[(size_t)v * Lt + j];
}

__global__ void __launch_bounds__(128) k_la_resolve(ChainParams P, StateDev st, LogDev lg) {
    const int W = P.W, Cr = P.Cr, Cv = P.C, Lt = P.K + kTheta0;
    const int c = blockIdx.x, v0 = c;             // lane j of chain c is entry c + j * Cr
    const int s0 = st.step[c];
    int limit = *st.step_end - s0;
    if (limit > P.Wa) limit = P.Wa;               // lanes that ran in this round
    if (limit <= 0) {                             // this chain has taken all its steps
        if (st.sx.pending && threadIdx.x == 0) st.sx.flush_w[c] = 0;
        return;
    }
    int jstar = -1;
    for (int j = 0; j < limit; j++)
        if (st.lane_ok[v0 + j * Cr]) { jstar = j; break; }
    const int consumed = jstar >= 0 ? jstar + 1 : limit;
    // records of the consumed steps: the state that is current after each of them (JSONAcceptRejectLogger.scala:93-106)
    const double *cur = st.theta_cur + (size_t)v0 * Lt;
    for (int j = 0; j < consumed; j++) {
        const int v = v0 + j * Cr;
        const bool ok = j == jstar;
        const size_t rec = (size_t)(s0 + j - lg.step_base) * Cr + c;
        if (lg.theta) {
            const double *src = ok ? st.theta_prop + (size_t)v * Lt : cur;
            for (int k = threadIdx.x; k < Lt; k += blockDim.x) lg.theta[rec * Lt + k] = src[k];
        }
        if (threadIdx.x == 0) {
            if (lg.comp) lg.comp[rec] = st.comp_sel[v];
            if (lg.accepted) lg.accepted[rec] = (uint8_t)ok;
            if (lg.values) {
                const double *val = ok ? st.values_prop + 3 * v : st.values_cur + 3 * v0;
                lg.values[3 * rec] = val[0]; lg.values[3 * rec + 1] = val[1]; lg.values[3 * rec + 2] = val[2];
            }
            if (st.lane_status[v]) st.status[c] |= st.lane_status[v];
        }
    }
    if (st.sx.pending) {
        // statistics, as k_chain_accept does them step by step: the rejected steps' records belong to the old state, which
        // an accepting lane flushes; the accepting step's record belongs to the new state
        __shared__ int s_flush;
        if (threadIdx.x == 0) {
            long long pend = st.sx.pending[c];
            for (int j = 0; j < consumed; j++)
                if (j != jstar) pend += stats_selected(st.sx, (long long)s0 + j);
            const int flush = jstar >= 0 && pend > 0;
            st.sx.flush_w[c] = flush ? pend : 0;
            if (flush) { st.sx.flush_n[c] = st.sx.count[c]; st.sx.count[c] += pend; }
            st.sx.pending[c] = jstar >= 0 ? stats_selected(st.sx, (long long)s0 + jstar) : pend;
            s_flush = flush;
        }
        __syncthreads();
        if (s_flush)
            for (int k = threadIdx.x; k < Lt; k += blockDim.x) st.sx.flush_theta[(size_t)c * Lt + k] = cur[k];
    }
    __syncthreads();   // the log rows above read the old current state
    if (jstar >= 0) {
        const int w = v0 + jstar * Cr;
        const double *prp = st.theta_prop + (size_t)w * Lt;
        const double vp0 = st.values_prop[3 * w], vp1 = st.values_prop[3 * w + 1], vp2 = st.values_prop[3 * w + 2];
        // BestSampleLogger.logState
        if (vp0 > st.value_best[c])
            for (int k = threadIdx.x; k < Lt; k += blockDim.x) st.theta_best[(size_t)c * Lt + k] = prp[k];
        // the accepted proposal becomes the current state of every lane; its posteriors (the winner's proposal slot) become the
        // shared current posteriors, and the winner proposes into the other slot of its pair from now on
        for (int j = 0; j < W; j++)
            for (int k = threadIdx.x; k < Lt; k += blockDim.x) st.theta_cur[(size_t)(v0 + j * Cr) * Lt + k] = prp[k];
        __syncthreads();
        if (threadIdx.x == 0) {
            if (vp0 > st.value_best[c]) st.value_best[c] = vp0;
            const int newcur = st.slot_prop[w];
            for (int j = 0; j < W; j++) {
                const int v = v0 + j * Cr;
                st.slot_cur[v] = newcur;
                st.values_cur[3 * v] = vp0; st.values_cur[3 * v + 1] = vp1; st.values_cur[3 * v + 2] = vp2;
            }
            st.slot_prop[w] = newcur == w ? Cv + w : w;
            st.n_acc[c] += 1;
        }
    }
    if (threadIdx.x == 0) st.step[c] = s0 + consumed;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
struct icp_chain_s {
    icp_model model = nullptr;
    icp_target target = nullptr;
    icp_evaluator evaluator = nullptr;
    int max_chains = 0;
    ChainParams P{};
    std::vector<icp_proposal> icp_props;
    // state
    DevBuf<double> theta_cur, theta_prop, values_cur, values_prop, u_acc, L, ymean, X, W, theta_best, value_best, qf, qb;
    MetricsWork mwork;       // periodic RegistrationComparison of the best sample (icp_chain_io.metrics_interval)
    DevBuf<int> cur_sel, slot_cur, slot_prop, comp_sel, step, status;
    DevBuf<int> lane_ok, lane_status, step_end;   // rejection look-ahead (k_la_resolve)
    int lookahead = -1;      // lanes per chain: -1 automatic (lookahead_width) with the active width adapted while the run
                             // goes (chain_run_device), 0 / 1 off, else exactly that width
    int resident_W = 1;      // width the resident state was laid out with
    bool any_svd = false;    // some ICP component samples with the reference's SVD factor
    std::vector<int> h_status;   // per-chain status words of the last synchronous run
    DevBuf<long long> n_acc;
    std::vector<PosteriorWork> pwork;
    std::vector<DevBuf<int>> cp_map;     // per ICP component: index of its model points in the evaluator's list
    std::vector<char> cp_shared, on_side;
    bool use_streams = true;
    EvalWork ework;
    DevBuf<int> estatus;
    // staging for the host-buffer entry point
    DevBuf<double> h_u_comp, h_z, h_u_acc, h_log_values, h_log_theta, h_log_metrics;
    DevBuf<int> h_log_comp;
    DevBuf<uint8_t> h_log_acc;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaStream_t copy_stream = nullptr;   // host-buffer entry point: log rows leave for the host while later steps run
    cudaEvent_t copy_ev = nullptr;
    double last_ms = 0;
    int64_t last_launches = 0;
    int last_per_step = 0;
    int64_t last_rounds = 0;   // batched rounds of the last run (= steps without the look-ahead)
    bool use_graph = true;
    int resident_C = 0;      // chains whose state is resident from the last run (resume)
    int sized_C = 0;         // every workspace is allocated for this many chains (graph capture cannot allocate)
    cudaGraphExec_t exec = nullptr;   // cached step graph + the bytes of the kernel arguments it was captured with
    std::string exec_key;
    std::map<int, cudaGraphExec_t> exec_wa;   // look-ahead: the round graphs of the other active widths under the same key
    // what the adaptive look-ahead has learnt on this chain object (kept across runs of the same shape): ms per round of
    // every active width tried, the smoothed acceptance rate
    std::map<int, double> la_t_round;
    double la_a_hat = -1.0;
    int la_Cr = 0, la_W = 0;
    DevBuf<double> d_theta0, d_final;   // persistent staging of the host-buffer entry point
    DevBuf<long long> d_nacc;
    int steps_total = 0;     // value of the device step counter
    // posterior variability inside the run: requested parameters (icp_chain_set_statistics) and those of the resident run
    bool stats_req_on = false, stats_on = false;
    icp_chain_stats_params stats_req{}, stats_run{};
    DevBuf<long long> sx_pending, sx_count, sx_flush_w, sx_flush_n;   // StatsDev
    DevBuf<double> sx_flush_theta, sx_mean, sx_m2, sx_nsum;          // StatsDev.flush_theta, StatsAcc
    DevBuf<int> sx_idx, sx_nlist;                                    // launch_stats_flush's list of flushed chains
    // target set (icp_chain_create_targets). model / target / evaluator / icp_props above are those of entry 0, which every
    // entry shares except for its target; with one target nothing below is used and the runner is the single-target one.
    int n_targets = 1;
    std::vector<icp_target> all_targets;       // [G] (references held)
    std::vector<icp_evaluator> all_evals;      // [G]
    std::vector<icp_proposal> all_props;       // every entry's ICP proposals
    bool set_boundary = false;                 // OR of the targets' has_boundary
    DevBuf<TargetRec> trec;                    // [G]
    std::vector<DevBuf<double>> tp_all;        // per ICP component: [G][n_tp][3] the entries' target points (target sampling)
    DevBuf<double> etp_all;                    // [G][etp_n][3] the evaluators' target -> model lists, padded to the longest
    int etp_n = 0;
    std::vector<int> tidx_req;                 // icp_chain_set_target_index: the target of every chain of the next run from theta0
    DevBuf<int> tidx;                          // [C] target of every batch entry (look-ahead: lane v takes chain v % Cr's)
    std::vector<DevBuf<double>> tp_lane;       // per ICP component: [C][n_tp][3]
    DevBuf<double> etp_lane;                   // [C][etp_n][3]
};

namespace {

// first difference between two entries of a target set that may only differ in their target ("" when none)
std::string entry_difference(const icp_chain_target &a, const icp_chain_target &b, int n_components) {
    auto ids_of = [](const DevBuf<int> &d, int n) {
        std::vector<int> h(n);
        if (n) ICP_CUDA(cudaMemcpy(h.data(), d.p, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost));
        return h;
    };
    for (int i = 0; i < n_components; i++) {
        const icp_component &x = a.components[i], &y = b.components[i];
        const std::string c = "component " + std::to_string(i) + " ";
        if (x.kind != y.kind) return c + "kind";
        if (x.weight != y.weight) return c + "weight";
        if (x.sd != y.sd) return c + "sd";
        if (x.axis != y.axis) return c + "axis";
        if (x.kind != ICP_PROP_ICP) continue;
        if (!y.proposal) return c + "proposal (null)";
        const icp_proposal_s &p = *x.proposal, &q = *y.proposal;
        if (p.model != q.model) return c + "proposal model";
        if (p.prm.step_length != q.prm.step_length) return c + "proposal step_length";
        if (p.prm.tangential_noise != q.prm.tangential_noise) return c + "proposal tangential_noise";
        if (p.prm.noise_along_normal != q.prm.noise_along_normal) return c + "proposal noise_along_normal";
        if (p.prm.direction != q.prm.direction) return c + "proposal direction";
        if (p.prm.boundary_aware != q.prm.boundary_aware) return c + "proposal boundary_aware";
        if (p.prm.factor != q.prm.factor) return c + "proposal factor";
        if (p.prm.rank_update != q.prm.rank_update) return c + "proposal rank_update";
        if (p.n_ids != q.n_ids || ids_of(p.ids, p.n_ids) != ids_of(q.ids, q.n_ids)) return c + "proposal model point ids";
        if (p.n_tp != q.n_tp) return c + "proposal n_tp";
    }
    const icp_evaluator_s &e = *a.evaluator, &f = *b.evaluator;
    if (e.model != f.model) return "evaluator model";
    if (e.prm.kind != f.prm.kind) return "evaluator kind";
    if (e.prm.mode != f.prm.mode) return "evaluator mode";
    if (e.prm.use_prior != f.prm.use_prior) return "evaluator use_prior";
    if (e.prm.p0 != f.prm.p0) return "evaluator p0";
    if (e.prm.p1 != f.prm.p1) return "evaluator p1";
    if (e.prm.p2 != f.prm.p2) return "evaluator p2";
    if (e.n_ids != f.n_ids || ids_of(e.ids, e.n_ids) != ids_of(f.ids, f.n_ids)) return "evaluator model point ids";
    if (e.prm.kind != ICP_EVAL_HAUSDORFF && e.n_tp != f.n_tp) return "evaluator n_tp";   // Hausdorff: all of its target's vertices
    return "";
}

__global__ void k_gather_target_rows(long long total, int row, const int *__restrict__ tidx, const double *__restrict__ src,
                                     double *__restrict__ dst) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long c = i / row, k = i % row;
    dst[i] = src[(size_t)tidx[c] * row + k];
}

}  // namespace

extern "C" int32_t icp_chain_create_targets(icp_model m, int32_t n_targets, const icp_chain_target *targets, int32_t n_components,
                                            int32_t max_chains, icp_chain *out) {
    icp_chain ch = nullptr;
    icp_ctx _ctx = m ? m->ctx : nullptr;
    try {
        ICP_REQUIRE(m && targets && out && n_targets >= 1, "null argument");
        for (int g = 0; g < n_targets; g++) {
            const icp_chain_target &e = targets[g];
            ICP_REQUIRE(e.target && e.components && e.evaluator, "null argument (targets[" + std::to_string(g) + "])");
            ICP_REQUIRE(m->ctx == e.target->ctx, "model and target belong to different contexts");
            ICP_REQUIRE(e.evaluator->model == m && e.evaluator->target == e.target, "evaluator was built for another model / target");
        }
        ICP_REQUIRE(n_components >= 1 && n_components <= kMaxComp, "1..16 mixture components supported");
        ICP_REQUIRE(max_chains >= 1, "max_chains must be >= 1");
        CtxLock lock(_ctx);
        const icp_target t = targets[0].target;
        const icp_component *components = targets[0].components;
        const icp_evaluator evaluator = targets[0].evaluator;
        for (int g = 0; g < n_targets; g++)
            for (int i = 0; i < n_components; i++) {
                const icp_component &ci = targets[g].components[i];
                if (ci.kind == ICP_PROP_ICP)
                    ICP_REQUIRE(ci.proposal && ci.proposal->model == m && ci.proposal->target == targets[g].target,
                                "ICP component needs a proposal built for this model / target");
            }
        for (int g = 1; g < n_targets; g++) {
            const std::string d = entry_difference(targets[0], targets[g], n_components);
            ICP_REQUIRE(d.empty(), "targets[" + std::to_string(g) + "]: " + d + " differs from targets[0] (only the target may differ)");
        }
        ch = new icp_chain_s();
        ch->model = m; ch->target = t; ch->evaluator = evaluator; ch->max_chains = max_chains;
        ch->n_targets = n_targets;
        for (int g = 0; g < n_targets; g++) {
            ch->all_targets.push_back(targets[g].target);
            ch->all_evals.push_back(targets[g].evaluator);
            ch->set_boundary = ch->set_boundary || targets[g].target->has_boundary;
        }
        // with one target the boundary policy is that target's own
        const bool has_boundary = n_targets > 1 ? ch->set_boundary : t->has_boundary;
        ChainParams &P = ch->P;
        P.n_comp = n_components; P.K = m->K; P.Kp = m->Kp; P.n_icp = 0;
        double wsum = 0;
        for (int i = 0; i < n_components; i++) {
            ICP_REQUIRE(components[i].weight > 0 && std::isfinite(components[i].weight), "component weights must be > 0");
            wsum += components[i].weight;
        }
        double acc = 0;
        for (int i = 0; i < n_components; i++) {
            const icp_component &ci = components[i];
            CompDev &cd = P.comp[i];
            cd.kind = ci.kind; cd.axis = ci.axis; cd.sd = ci.sd; cd.icp_index = -1; cd.step = 1.0; cd.factor = ICP_FACTOR_CHOLESKY;
            cd.weight = ci.weight / wsum;
            acc += cd.weight;
            cd.cdf = i == n_components - 1 ? 1.0 : acc;
            switch (ci.kind) {
                case ICP_PROP_ICP:
                    cd.icp_index = P.n_icp++;
                    cd.step = ci.proposal->prm.step_length;
                    cd.factor = ci.proposal->prm.factor;
                    if (cd.factor == ICP_FACTOR_SVD) ch->any_svd = true;
                    ch->icp_props.push_back(ci.proposal);
                    break;
                case ICP_PROP_RANDOM_SHAPE:
                    ICP_REQUIRE(ci.sd > 0, "random-walk std-dev must be > 0");
                    break;
                case ICP_PROP_ROTATION:
                case ICP_PROP_TRANSLATION:
                    ICP_REQUIRE(ci.sd > 0 && ci.axis >= 0 && ci.axis < 3, "pose proposal needs sd > 0 and axis in 0..2");
                    break;
                default:
                    throw ArgError{"unknown component kind"};
            }
        }
        ch->pwork.resize(P.n_icp);
        // closest points shared with the evaluator: a model-sampling proposal whose point ids all occur in the
        // evaluator's model->target list reuses those traversals instead of repeating them
        ch->cp_map.resize(P.n_icp);
        ch->cp_shared.assign(P.n_icp, 0);
        ch->on_side.assign(P.n_icp, 0);
        { const char *e2 = getenv("ICPCUDA_NO_STREAMS"); ch->use_streams = !(e2 && e2[0] == '1'); }
        {
            const icp_evaluator_params &ep = evaluator->prm;
            bool ev_m2t = ep.kind == ICP_EVAL_HAUSDORFF || ((ep.kind == ICP_EVAL_INDEPENDENT || ep.kind == ICP_EVAL_COLLECTIVE) && ep.mode != ICP_TARGET_TO_MODEL);
            // not for the Hausdorff evaluator: its traversals stop every query that cannot raise the chain's maximum
            // (k_nearest, HDMAX), which is worth more than the shared queries and leaves most closest points unknown
            static const bool hd_prune_on = !(getenv("ICPCUDA_HAUSDORFF_PRUNE") && getenv("ICPCUDA_HAUSDORFF_PRUNE")[0] == '0');
            if (ev_m2t && evaluator->n_ids > 0 && !(ep.kind == ICP_EVAL_HAUSDORFF && hd_prune_on)) {
                std::vector<int> eids(evaluator->n_ids);
                ICP_CUDA(cudaMemcpy(eids.data(), evaluator->ids.p, sizeof(int) * eids.size(), cudaMemcpyDeviceToHost));
                std::unordered_map<int, int> pos;
                for (int i = (int)eids.size() - 1; i >= 0; i--) pos[eids[i]] = i;
                for (int k = 0; k < P.n_icp; k++) {
                    icp_proposal pr = ch->icp_props[k];
                    if (pr->prm.direction != ICP_MODEL_SAMPLING || pr->n_ids == 0) continue;
                    if (pr->prm.boundary_aware && has_boundary) continue;
                    std::vector<int> pids(pr->n_ids), map(pr->n_ids);
                    ICP_CUDA(cudaMemcpy(pids.data(), pr->ids.p, sizeof(int) * pids.size(), cudaMemcpyDeviceToHost));
                    bool ok = true;
                    for (int i = 0; i < pr->n_ids && ok; i++) {
                        auto it = pos.find(pids[i]);
                        if (it == pos.end()) ok = false; else map[i] = it->second;
                    }
                    if (!ok) continue;
                    ch->cp_map[k].upload(map.data(), map.size(), _ctx->stream);
                    ch->cp_shared[k] = 1;
                    ch->ework.force_cp_m2t = true;
                }
                ICP_CUDA(cudaStreamSynchronize(_ctx->stream));
            }
        }
        ICP_CUDA(cudaEventCreate(&ch->ev0));
        ICP_CUDA(cudaEventCreate(&ch->ev1));
        const char *env = getenv("ICPCUDA_NO_GRAPH");
        ch->use_graph = !(env && env[0] == '1');
        if (n_targets > 1) {
            // the device table of the targets and every entry's point lists, laid end to end in entry order
            cudaStream_t s = _ctx->stream;
            std::vector<TargetRec> rec(n_targets);
            for (int g = 0; g < n_targets; g++) {
                const icp_target tg = targets[g].target;
                rec[g] = TargetRec{{tg->tri_bvh.packed.p, tg->vert_bvh.packed.p}, {tg->tri_bvh.prim.p, tg->vert_bvh.prim.p},
                                   {tg->tri_data.p, tg->vert_data.p}, {tg->tri_bvh.n, tg->vert_bvh.n}, tg->boundary.p, tg->Nt};
            }
            ch->trec.upload(rec.data(), rec.size(), s);
            ch->tp_all.resize(P.n_icp);
            ch->tp_lane.resize(P.n_icp);
            for (int k = 0; k < P.n_icp; k++) {
                const int n_tp = ch->icp_props[k]->n_tp;
                if (ch->icp_props[k]->prm.direction != ICP_TARGET_SAMPLING || n_tp == 0) continue;
                ch->tp_all[k].alloc((size_t)n_targets * n_tp * 3);
                int j = 0;
                for (int i = 0; i < n_components; i++) {   // the k-th ICP component of entry g
                    if (components[i].kind != ICP_PROP_ICP || j++ != k) continue;
                    for (int g = 0; g < n_targets; g++)
                        ICP_CUDA(cudaMemcpyAsync(ch->tp_all[k].p + (size_t)g * n_tp * 3, targets[g].components[i].proposal->tp.p,
                                                 sizeof(double) * n_tp * 3, cudaMemcpyDeviceToDevice, s));
                }
            }
            for (int g = 0; g < n_targets; g++) ch->etp_n = std::max(ch->etp_n, targets[g].evaluator->n_tp);
            if (ch->etp_n > 0) {
                // Hausdorff targets may have different vertex counts: a shorter list is padded with repeats of its last
                // vertex, which leaves the largest distance, the only one the evaluator keeps, unchanged
                const int nm = ch->etp_n;
                ch->etp_all.alloc((size_t)n_targets * nm * 3);
                for (int g = 0; g < n_targets; g++) {
                    const icp_evaluator eg = targets[g].evaluator;
                    double *dst = ch->etp_all.p + (size_t)g * nm * 3;
                    ICP_CUDA(cudaMemcpyAsync(dst, eg->tp.p, sizeof(double) * eg->n_tp * 3, cudaMemcpyDeviceToDevice, s));
                    for (int r = eg->n_tp; r < nm; r++)
                        ICP_CUDA(cudaMemcpyAsync(dst + (size_t)r * 3, eg->tp.p + (size_t)(eg->n_tp - 1) * 3, sizeof(double) * 3,
                                                 cudaMemcpyDeviceToDevice, s));
                }
            }
            ICP_CUDA(cudaStreamSynchronize(s));
        }
        m->refs++;
        for (int g = 0; g < n_targets; g++) {
            targets[g].target->refs++;
            targets[g].evaluator->refs++;
            for (int i = 0; i < n_components; i++)
                if (targets[g].components[i].kind == ICP_PROP_ICP) {
                    targets[g].components[i].proposal->refs++;
                    ch->all_props.push_back(targets[g].components[i].proposal);
                }
        }
        *out = ch;
        return ICP_OK;
    } catch (...) {
        int32_t rc = translate_exception(_ctx);
        delete ch;
        return rc;
    }
}


extern "C" int32_t icp_chain_create(icp_model m, icp_target t, const icp_component *components, int32_t n_components,
                                    icp_evaluator evaluator, int32_t max_chains, icp_chain *out) {
    const icp_chain_target one{t, components, evaluator};
    return icp_chain_create_targets(m, 1, &one, n_components, max_chains, out);
}

extern "C" int32_t icp_chain_set_target_index(icp_chain c, int32_t C, const int32_t *target_index) {
    icp_ctx _ctx = c ? c->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr && target_index != nullptr, "null argument");
        CtxLock lock(_ctx);
        ICP_REQUIRE(C >= 1 && C <= c->max_chains, "C must be in [1, max_chains]");
        for (int i = 0; i < C; i++)
            ICP_REQUIRE(target_index[i] >= 0 && target_index[i] < c->n_targets,
                        "target_index[" + std::to_string(i) + "] = " + std::to_string(target_index[i]) + " is outside [0, n_targets)");
        c->tidx_req.assign(target_index, target_index + C);
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_chain_destroy(icp_chain c) {
    if (!c) return ICP_OK;
    icp_ctx _ctx = c->model->ctx;
    try {
        CtxLock lock(_ctx);
        ICP_CUDA(cudaStreamSynchronize(_ctx->stream));
        if (c->exec) cudaGraphExecDestroy(c->exec);
        for (auto &kv : c->exec_wa) if (kv.second) cudaGraphExecDestroy(kv.second);
        if (c->ev0) cudaEventDestroy(c->ev0);
        if (c->ev1) cudaEventDestroy(c->ev1);
        if (c->copy_ev) cudaEventDestroy(c->copy_ev);
        if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
        c->model->refs--;
        for (icp_target t : c->all_targets) t->refs--;
        for (icp_evaluator e : c->all_evals) e->refs--;
        for (icp_proposal pr : c->all_props) pr->refs--;
        delete c;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

namespace {

struct RunCtx {
    icp_chain ch;
    int C;            // stride of the per-chain arrays (lanes in look-ahead mode: Cr * W)
    int Cn = 0;       // entries the kernels of this step / round process (C, or Cr * Wa with Wa active lanes)
    int W = 1, Cr = 0, Wa = 1;
    StateDev st;
    RngDev rng;
    LogDev lg;
    cudaStream_t s;
    int64_t launches = 0;
};

// evaluator + ICP posteriors of the parameter vectors in `theta` (all chains), written to the
// posterior state selected by `slots`
// proposal: the state is the step's proposal, so every ICP posterior also leaves the backward transition form
// |L_prop^T d|^2 (theta_prop -> theta_cur) in st.qb while its factor is on chip
void enqueue_state_eval(RunCtx &r, const double *d_theta, double *d_values, const int *d_slots, bool proposal) {
    icp_chain ch = r.ch;
    icp_model m = ch->model;
    const int C = r.C, Cn = r.Cn, Kp = m->Kp;   // C: stride of the posterior / form arrays, Cn: entries to evaluate
    icp_ctx ctx = m->ctx;
    launch_reconstruct(m->dev(), Cn, d_theta, ch->X.p, r.s);
    // fork: ICP pipelines that do not consume the evaluator's closest points run on side streams, concurrently with
    // the evaluator and with each other (their Cholesky phases are latency bound and overlap the DMMA of the rest).
    // Profiling runs stay on one stream so that the per-kernel event times do not overlap.
    // (the model's vertex-BVH boxes are shared scratch: only fork when the nearest-vertex queries use the brute-force tile)
    const bool brute_ok = sizeof(double) * 3 * (size_t)((m->N + 1) & ~1) + sizeof(float4) * (size_t)m->N <= 100 * 1024;
    static const bool forced_bvh = getenv("ICPCUDA_NEAREST_VERTEX") && std::string(getenv("ICPCUDA_NEAREST_VERTEX")) == "bvh";
    const bool fork = !g_prof && ch->use_streams && brute_ok && !forced_bvh;
    int n_side = 0;
    // several targets: every consumer reads the batch entry's target from the table (TargetSet)
    const bool multi = ch->n_targets > 1;
    std::vector<TargetSet> tsv(ch->P.n_icp);
    if (multi)
        for (int i = 0; i < ch->P.n_icp; i++)
            tsv[i] = TargetSet{ch->trec.p, ch->tidx.p, ch->set_boundary, ch->tp_lane[i].p, ch->icp_props[i]->n_tp};
    const TargetSet ets{ch->trec.p, ch->tidx.p, ch->set_boundary, ch->etp_lane.p, ch->etp_n};
    if (fork) ICP_CUDA(cudaEventRecord(ctx->ev_fork, r.s));
    for (int i = 0; i < ch->P.n_icp; i++) {
        if (ch->cp_shared[i] || !fork || n_side >= icp_ctx_s::kAux) continue;
        cudaStream_t ss = ctx->aux[n_side];
        ICP_CUDA(cudaStreamWaitEvent(ss, ctx->ev_fork, 0));
        double *Lb = r.st.L + (size_t)i * 2 * C * Kp * Kp, *yb = r.st.ymean + (size_t)i * 2 * C * Kp;
        double *Wb = ch->icp_props[i]->prm.factor == ICP_FACTOR_SVD ? r.st.W + (size_t)i * 2 * C * Kp * Kp : nullptr;
        QuadArgs qa{r.st.theta_prop, r.st.theta_cur, ch->icp_props[i]->prm.step_length, m->K, r.st.qb + (size_t)i * C};
        posterior_pipeline(ch->icp_props[i], Cn, d_theta, ch->X.p, ch->pwork[i], Lb, yb, d_slots, ss, nullptr, Wb, proposal ? &qa : nullptr,
                           Wb == nullptr, multi ? &tsv[i] : nullptr);
        ICP_CUDA(cudaEventRecord(ctx->ev_join[n_side], ss));
        ch->on_side[i] = 1;
        n_side++;
    }
    evaluator_pipeline(ch->evaluator, ch->ework, Cn, d_theta, ch->X.p, d_values, ch->estatus.p, r.s, multi ? &ets : nullptr);
    for (int i = 0; i < ch->P.n_icp; i++) {
        if (ch->on_side[i]) { ch->on_side[i] = 0; continue; }
        double *Lb = r.st.L + (size_t)i * 2 * C * Kp * Kp, *yb = r.st.ymean + (size_t)i * 2 * C * Kp;
        SharedCp sh{ch->ework.cp_m2t.p, ch->evaluator->n_ids, ch->cp_map[i].p};
        double *Wb = ch->icp_props[i]->prm.factor == ICP_FACTOR_SVD ? r.st.W + (size_t)i * 2 * C * Kp * Kp : nullptr;
        QuadArgs qa{r.st.theta_prop, r.st.theta_cur, ch->icp_props[i]->prm.step_length, m->K, r.st.qb + (size_t)i * C};
        posterior_pipeline(ch->icp_props[i], Cn, d_theta, ch->X.p, ch->pwork[i], Lb, yb, d_slots, r.s, ch->cp_shared[i] ? &sh : nullptr, Wb,
                           proposal ? &qa : nullptr, Wb == nullptr, multi ? &tsv[i] : nullptr);
    }
    for (int k = 0; k < n_side; k++) ICP_CUDA(cudaStreamWaitEvent(r.s, ctx->ev_join[k], 0));   // join
}

StatusSrc status_sources(icp_chain ch) {
    StatusSrc ss{};
    ss.eval = ch->estatus.p;
    ss.n_post = ch->P.n_icp;
    for (int i = 0; i < ch->P.n_icp; i++) ss.post[i] = ch->pwork[i].status.p;
    return ss;
}

void enqueue_step(RunCtx &r) {
    icp_chain ch = r.ch;
    icp_model m = ch->model;
    const int C = r.C, Cn = r.Cn, Kp = m->Kp;
    ChainParams P = ch->P;
    P.C = C; P.W = r.W; P.Cr = r.Cr; P.Wa = r.Wa;
    size_t smem_p = sizeof(double) * ((size_t)7 * Kp + 40 + (size_t)Kp * (Kp + 1) / 2);
    {
        ProfScope ps(ST_PROPOSE, r.s);
        k_chain_propose<<<Cn, 256, smem_p, r.s>>>(P, m->dev(), r.st, r.rng);
        ICP_CUDA(cudaGetLastError());
    }
    enqueue_state_eval(r, r.st.theta_prop, r.st.values_prop, r.st.slot_prop, true);
    {
        ProfScope ps(ST_ACCEPT, r.s);
        k_chain_accept<<<Cn, 128, sizeof(double) * 40, r.s>>>(P, r.st, r.lg, status_sources(ch));
        ICP_CUDA(cudaGetLastError());
        if (r.W > 1) k_la_resolve<<<r.Cr, 128, 0, r.s>>>(P, r.st, r.lg);   // one round of the look-ahead: 1 .. W steps per chain
        else k_step_increment<<<1, 1, 0, r.s>>>(r.st.step);
        ICP_CUDA(cudaGetLastError());
    }
    if (r.st.sx.pending) {
        // statistics: the states the chains flushed in this step / round into their accumulators (stats.cu). ch->X, the
        // meshes of this step's proposals, is free until the next step reconstructs into it.
        ProfScope ps(ST_OTHER, r.s);
        const StatsDev &x = r.st.sx;
        launch_stats_flush(m->dev(), r.Cr, x.flush_theta, x.flush_w, x.flush_n, ch->sx_idx.p, ch->sx_nlist.p, ch->X.p,
                           StatsAcc{ch->sx_mean.p, ch->sx_m2.p, ch->stats_run.normals ? ch->sx_nsum.p : nullptr}, r.s);
    }
}

// Width of the rejection look-ahead a run of C chains will use (1 = the plain step-by-step runner). Off while profiling, with
// periodic metrics (they are defined per step), for asynchronous runs (the look-ahead reads the step counters back between
// batches of rounds) and for resumed runs of a state that was laid out without it.
int lookahead_width(icp_chain ch, int C, const icp_chain_io *io, bool resume, bool may_block) {
    if (resume) return ch->resident_W;
    static const int env = getenv("ICPCUDA_LOOKAHEAD") ? atoi(getenv("ICPCUDA_LOOKAHEAD")) : -1;
    int w = ch->lookahead >= 0 ? ch->lookahead : env;
    if (g_prof || !may_block || io->metrics_interval > 0) return 1;
    // automatic: as many lanes as still ride on latency rather than throughput (measured, tools/chains_sweep.py:
    // profiles/r2_session3.md section 9) - 8 up to 8 chains, 4 up to 32, 2 up to 148, none beyond
    if (w < 0) w = C <= 8 ? 8 : C <= 32 ? 4 : C <= 148 ? 2 : 1;
    if (w > 32) w = 32;
    return w < 2 ? 1 : w;
}

// on_step(k): called on the host right after step k (1-based) of this call has been enqueued on the library stream
// may_block: the call may synchronise with the device before it returns (the look-ahead needs that); async callers that
// synchronise themselves afterwards (icp_chain_run) pass true
void chain_run_device(icp_chain ch, int C, int n_steps, const double *theta0_dev, const icp_chain_io *io, bool async,
                      const std::function<void(int)> *on_step = nullptr, bool may_block = false) {
    may_block = may_block || !async;
    icp_model m = ch->model;
    icp_ctx ctx = m->ctx;
    cudaStream_t s = ctx->stream;
    const int K = m->K, Kp = m->Kp, Lt = K + kTheta0;
    ICP_REQUIRE(C >= 1 && C <= ch->max_chains, "C must be in [1, max_chains]");
    ICP_REQUIRE(n_steps >= 0, "n_steps must be >= 0");
    ICP_REQUIRE(io != nullptr, "null argument");
    const bool resume = theta0_dev == nullptr;
    if (resume) ICP_REQUIRE(ch->resident_C == C, "resume needs a previous run with the same number of chains");
    bool host_rng = io->u_comp || io->z || io->u_acc;
    if (host_rng) ICP_REQUIRE(io->u_comp && io->z && io->u_acc, "u_comp, z and u_acc must be given together");
    const int n_icp = ch->P.n_icp;
    // rejection look-ahead: W lanes per chain; from here on C counts lanes, Cr chains
    const int W = on_step ? 1 : lookahead_width(ch, C, io, resume, may_block), Cr = C;
    if (resume) ICP_REQUIRE(W == ch->resident_W, "this chain's resident state uses the rejection look-ahead: resume it without "
                            "a per-step hook, or restart it from theta0");
    if (W > 1) {
        ICP_REQUIRE(io->metrics_interval == 0 && may_block, "this chain's resident state uses the rejection look-ahead: "
                    "resume it without metrics_interval and synchronously, or restart it from theta0");
        C = Cr * W;
        ch->lane_ok.ensure(C); ch->lane_status.ensure(C); ch->step_end.ensure(1);
    }
    ch->theta_cur.ensure((size_t)C * Lt); ch->theta_prop.ensure((size_t)C * Lt);
    ch->values_cur.ensure((size_t)3 * C); ch->values_prop.ensure((size_t)3 * C);
    ch->u_acc.ensure(C); ch->cur_sel.ensure(C); ch->slot_cur.ensure(C); ch->slot_prop.ensure(C);
    ch->comp_sel.ensure(C); ch->step.ensure(Cr); ch->n_acc.ensure(C); ch->estatus.ensure(C); ch->status.ensure(C);
    if (ch->any_svd) ch->W.ensure((size_t)std::max(n_icp, 1) * 2 * C * Kp * Kp);
    ch->theta_best.ensure((size_t)C * Lt); ch->value_best.ensure(C);
    ch->qf.ensure((size_t)std::max(n_icp, 1) * C); ch->qb.ensure((size_t)std::max(n_icp, 1) * C);
    ICP_REQUIRE(io->metrics_interval >= 0, "metrics_interval must be >= 0");
    ICP_REQUIRE(io->metrics_interval == 0 || ch->n_targets == 1,
                "metrics_interval > 0 is not supported on a chain handle with several targets: measure each target's theta_best rows "
                "with icp_registration_metrics after the run");
    ICP_REQUIRE(io->metrics_interval == 0 || io->log_metrics != nullptr, "metrics_interval > 0 needs log_metrics");
    ch->L.ensure((size_t)std::max(n_icp, 1) * 2 * C * Kp * Kp); ch->ymean.ensure((size_t)std::max(n_icp, 1) * 2 * C * Kp);
    ch->X.ensure((size_t)C * m->N * 3);

    RunCtx r;
    r.ch = ch; r.C = C; r.Cn = C; r.s = s; r.W = W; r.Cr = Cr; r.Wa = W;
    r.st = StateDev{ch->theta_cur.p, ch->theta_prop.p, ch->values_cur.p, ch->values_prop.p, ch->cur_sel.p,
                    ch->slot_cur.p, ch->slot_prop.p, ch->comp_sel.p, ch->u_acc.p, ch->n_acc.p, ch->step.p, ch->L.p,
                    ch->ymean.p, ch->any_svd ? ch->W.p : nullptr, ch->status.p, ch->theta_best.p, ch->value_best.p,
                    ch->qf.p, ch->qb.p, ch->lane_ok.p, ch->lane_status.p, ch->step_end.p};
    if (!resume) { ch->stats_on = ch->stats_req_on; ch->stats_run = ch->stats_req; }
    r.st.sx = StatsDev{};
    if (ch->stats_on) {
        const size_t nv = (size_t)Cr * m->N;
        ch->sx_pending.ensure(Cr); ch->sx_count.ensure(Cr); ch->sx_flush_w.ensure(Cr); ch->sx_flush_n.ensure(Cr);
        ch->sx_flush_theta.ensure((size_t)Cr * Lt); ch->sx_idx.ensure(Cr); ch->sx_nlist.ensure(1);
        ch->sx_mean.ensure(nv * 3); ch->sx_m2.ensure(nv * 6);
        if (ch->stats_run.normals) ch->sx_nsum.ensure(nv * 3);
        if (!resume) {
            ICP_CUDA(cudaMemsetAsync(ch->sx_pending.p, 0, sizeof(long long) * Cr, s));
            ICP_CUDA(cudaMemsetAsync(ch->sx_count.p, 0, sizeof(long long) * Cr, s));
            ICP_CUDA(cudaMemsetAsync(ch->sx_flush_w.p, 0, sizeof(long long) * Cr, s));
            ICP_CUDA(cudaMemsetAsync(ch->sx_mean.p, 0, sizeof(double) * nv * 3, s));
            ICP_CUDA(cudaMemsetAsync(ch->sx_m2.p, 0, sizeof(double) * nv * 6, s));
            if (ch->stats_run.normals) ICP_CUDA(cudaMemsetAsync(ch->sx_nsum.p, 0, sizeof(double) * nv * 3, s));
        }
        r.st.sx = StatsDev{ch->sx_pending.p, ch->sx_count.p, ch->sx_flush_w.p, ch->sx_flush_n.p, ch->sx_flush_theta.p,
                           ch->stats_run.burn_in, ch->stats_run.take_every_n, ch->stats_run.end};
    } else if (!resume) {   // allocated only while statistics are on
        ch->sx_pending.release(); ch->sx_count.release(); ch->sx_flush_w.release(); ch->sx_flush_n.release();
        ch->sx_flush_theta.release(); ch->sx_idx.release(); ch->sx_nlist.release();
        ch->sx_mean.release(); ch->sx_m2.release(); ch->sx_nsum.release();
    }
    const int step_base = resume ? ch->steps_total : 0;
    r.rng = RngDev{io->seed, io->chain_id_offset, io->u_comp, io->z, io->u_acc, step_base};
    r.lg = LogDev{io->log_component, io->log_accepted, io->log_values, io->log_theta, step_base};

    if (ch->n_targets > 1 && !resume) {
        // the target of every batch entry (lane v of the look-ahead runs chain v % Cr) and the entries' own point lists
        ICP_REQUIRE((int)ch->tidx_req.size() == Cr, "a chain handle with several targets needs icp_chain_set_target_index with C = " +
                    std::to_string(Cr) + " entries before a run from theta0");
        std::vector<int> lane(C);
        for (int v = 0; v < C; v++) lane[v] = ch->tidx_req[v % Cr];
        ch->tidx.upload(lane.data(), lane.size(), s);
        auto gather = [&](const DevBuf<double> &all, DevBuf<double> &dst, int n) {
            if (!all.p || n == 0) return;
            const long long total = (long long)C * n * 3;
            dst.ensure((size_t)total);
            k_gather_target_rows<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(total, 3 * n, ch->tidx.p, all.p, dst.p);
            ICP_CUDA(cudaGetLastError());
        };
        for (int k = 0; k < n_icp; k++) gather(ch->tp_all[k], ch->tp_lane[k], ch->icp_props[k]->n_tp);
        gather(ch->etp_all, ch->etp_lane, ch->etp_n);
    }
    ICP_CUDA(cudaEventRecord(ch->ev0, s));
    if (!resume && W > 1) {
        k_la_init<<<(C + 127) / 128, 128, 0, s>>>(Cr, W, Lt, theta0_dev, r.st);
        ICP_CUDA(cudaGetLastError());
    } else if (!resume) {
        ICP_CUDA(cudaMemcpyAsync(ch->theta_cur.p, theta0_dev, sizeof(double) * (size_t)C * Lt, cudaMemcpyDeviceToDevice, s));
        k_chain_init<<<(C + 127) / 128, 128, 0, s>>>(C, r.st);
        ICP_CUDA(cudaGetLastError());
    }
    if (W > 1) {
        k_la_set_end<<<1, 1, 0, s>>>(ch->step_end.p, step_base + n_steps);
        ICP_CUDA(cudaGetLastError());
    }
    {
        size_t smem_p = sizeof(double) * ((size_t)7 * Kp + 40 + (size_t)Kp * (Kp + 1) / 2);
        ICP_REQUIRE(smem_p <= 227 * 1024, "rank too large for the propose kernel");
        ICP_CUDA(cudaFuncSetAttribute(k_chain_propose, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p));
    }
    // state of theta0: log-values + posteriors of every ICP component (state 0)
    if (!resume) {
        enqueue_state_eval(r, ch->theta_cur.p, ch->values_cur.p, ch->slot_cur.p, false);
        if (W > 1) k_la_status0<<<(Cr + 127) / 128, 128, 0, s>>>(Cr, W, Lt, r.st, status_sources(ch));
        else k_chain_status0<<<(C + 127) / 128, 128, 0, s>>>(C, Lt, r.st, status_sources(ch));
        ICP_CUDA(cudaGetLastError());
    }

    // SamplingRegistration.scala:75-82: every acceptInfoPrintInterval iterations (iterator index i % interval == 0, i != 0;
    // index 0 is the initial state, so index i is the state after step i) the boundary-aware registration measures of the
    // best sample so far. Enqueued between the steps on the same stream; row r - 1 belongs to step r * interval.
    int metrics_rows = 0;
    auto after_step = [&](int done) {
        if (io->metrics_interval > 0 && done % io->metrics_interval == 0) {
            registration_metrics_device(m, ch->target, C, ch->theta_best.p, io->log_metrics + (size_t)metrics_rows * C * 4, ch->mwork, s);
            metrics_rows++;
        }
        if (on_step) (*on_step)(done);
    };
    // The step graph is cached on the chain: its kernel arguments are the state / RNG / log descriptors by value, so it
    // can be replayed by any later call whose descriptors are byte-identical (same C, buffers, seed, offsets).
    int steps_done = 0;
    const bool sized = ch->sized_C == C;
    if (n_steps > 0 && (!sized || !ch->use_graph || g_prof)) {
        // first step eagerly: sizes every workspace (allocation is illegal during capture)
        enqueue_step(r);
        steps_done = 1;
        ch->sized_C = C;
        after_step(steps_done);
    }
    cudaGraphExec_t exec = nullptr;
    // captures the step / round r describes (r.Cn entries, r.Wa active lanes) as a graph; nullptr when that fails
    auto capture = [&](int *per_step_out) -> cudaGraphExec_t {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t ex = nullptr;
        if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        bool ok = true;
        try {
            enqueue_step(r);
        } catch (...) {
            ok = false;
        }
        cudaError_t e = cudaStreamEndCapture(s, &graph);
        if (!ok || e != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            return nullptr;
        }
        size_t nn = 0;
        int per_step = 0;
        cudaGraphGetNodes(graph, nullptr, &nn);
        std::vector<cudaGraphNode_t> nodes(nn);
        cudaGraphGetNodes(graph, nodes.data(), &nn);
        for (size_t i = 0; i < nn; i++) {
            cudaGraphNodeType ty;
            if (cudaGraphNodeGetType(nodes[i], &ty) == cudaSuccess && ty == cudaGraphNodeTypeKernel) per_step++;
        }
        if (cudaGraphInstantiate(&ex, graph, 0) != cudaSuccess) { ex = nullptr; cudaGetLastError(); }
        cudaGraphDestroy(graph);
        if (ex && per_step_out) *per_step_out = per_step;
        return ex;
    };
    const bool graphs = ch->use_graph && !g_prof && n_steps - steps_done >= 1;
    if (graphs) {
        ChainParams Pk = ch->P;
        Pk.C = C; Pk.W = W; Pk.Cr = Cr; Pk.Wa = W;
        std::string key;
        key.append((const char *)&Pk, sizeof Pk);
        key.append((const char *)&r.st, sizeof r.st);
        key.append((const char *)&r.rng, sizeof r.rng);
        key.append((const char *)&r.lg, sizeof r.lg);
        key.push_back(ch->stats_on ? 1 : 0);   // the flush kernels are part of the step graph while statistics are on
        if (ch->stats_on) {
            const void *sx[] = {ch->sx_mean.p, ch->sx_m2.p, ch->stats_run.normals ? ch->sx_nsum.p : nullptr, ch->sx_idx.p,
                                ch->sx_nlist.p, ch->X.p};
            key.append((const char *)sx, sizeof sx);
        }
        {   // buffers the captured kernels address that are not part of the descriptors above: the pipelines' status words
            // and the MODEL's BVH scratch, which other calls on the same model may reallocate (a replay would dangle)
            StatusSrc ss = status_sources(ch);
            key.append((const char *)&ss, sizeof ss);
            const void *shared[] = {m->tri_bvh.nodes.p, m->tri_bvh.nodebox.p, m->tri_bvh.counters.p,
                                    m->vert_bvh.nodes.p, m->vert_bvh.nodebox.p, m->vert_bvh.counters.p};
            key.append((const char *)shared, sizeof shared);
            // the target set: its table, the entries' target index and point lists
            std::vector<const void *> tsp{ch->trec.p, ch->tidx.p, ch->etp_lane.p};
            for (const DevBuf<double> &b : ch->tp_lane) tsp.push_back(b.p);
            key.append((const char *)tsp.data(), sizeof(const void *) * tsp.size());
        }
        if (!(ch->exec && ch->exec_key == key)) {
            if (ch->exec) { cudaGraphExecDestroy(ch->exec); ch->exec = nullptr; }
            for (auto &kv : ch->exec_wa)
                if (kv.second) cudaGraphExecDestroy(kv.second);
            ch->exec_wa.clear();
            ch->exec_key = key;
            int per_step = 0;
            ch->exec = capture(&per_step);      // full width (r.Wa == W)
            if (ch->exec) ch->last_per_step = per_step;
        }
        exec = ch->exec;
    }
    int64_t rounds_total = steps_done, launches_total = (int64_t)ch->last_per_step * steps_done;
    if (W > 1) {
        // Rounds instead of steps. A round of Wa active lanes consumes 1 .. Wa steps of every unfinished chain, so remaining / Wa
        // rounds can never overshoot; the step and acceptance counters are read back after each batch of rounds.
        // With the automatic width (ch->lookahead < 0) the ACTIVE width adapts while the run goes: the lanes are laid out lane
        // major, so a round over the first Cr * Wa entries runs the lanes 0 .. Wa - 1 of every chain. A batch is timed with
        // events; the next batch takes the width with the largest expected steps per millisecond,
        // (1 - (1 - a)^w) / (a t_w), from the measured acceptance rate a and the measured (or, for a width not tried yet, the
        // neighbour's) round time t_w. Wide rounds win when steps are rejected and lanes are cheap (few chains, small point
        // sets); a chain that accepts everything, or lanes that already fill the GPU, settle at one lane.
        const bool adaptive = ch->lookahead < 0 && graphs;
        std::vector<int> widths;
        for (int w = 1; w < W; w *= 2) widths.push_back(w);
        widths.push_back(W);
        if (ch->la_Cr != Cr || ch->la_W != W) { ch->la_t_round.clear(); ch->la_a_hat = -1.0; ch->la_Cr = Cr; ch->la_W = W; }
        std::map<int, double> &t_round = ch->la_t_round;       // measured ms per round at a width
        std::vector<int> h_step(Cr);
        std::vector<long long> h_acc(Cr);
        cudaEvent_t eb0 = nullptr, eb1 = nullptr;
        ICP_CUDA(cudaEventCreate(&eb0));
        ICP_CUDA(cudaEventCreate(&eb1));
        auto read_counters = [&](long long &steps_sum, long long &acc_sum, int &lo) {
            ICP_CUDA(cudaMemcpyAsync(h_step.data(), ch->step.p, sizeof(int) * (size_t)Cr, cudaMemcpyDeviceToHost, s));
            ICP_CUDA(cudaMemcpyAsync(h_acc.data(), ch->n_acc.p, sizeof(long long) * (size_t)Cr, cudaMemcpyDeviceToHost, s));
            ICP_CUDA(cudaStreamSynchronize(s));
            steps_sum = 0; acc_sum = 0; lo = h_step[0];
            for (int c = 0; c < Cr; c++) { steps_sum += h_step[c]; acc_sum += h_acc[c]; lo = std::min(lo, h_step[c]); }
        };
        long long steps0 = 0, acc0 = 0;
        int lo = 0;
        try {
            read_counters(steps0, acc0, lo);
            int remaining = step_base + n_steps - lo;
            double a_hat = ch->la_a_hat >= 0.0 ? ch->la_a_hat : 0.5;   // acceptance rate, smoothed over the batches
            int wa = adaptive ? 1 : W, batches = ch->la_a_hat >= 0.0 ? 1 : 0;
            // every width not timed yet is timed once (8 rounds each), narrowest first: a short run costs what the plain
            // step-by-step run costs
            std::vector<int> probe;
            for (int w : widths)
                if (!t_round.count(w)) probe.push_back(w);
            while (remaining > 0) {
                bool probing = false;
                if (adaptive && !probe.empty() && (t_round.empty() || remaining >= 64)) {   // no experiments at the end of a run
                    wa = probe.front();
                    probe.erase(probe.begin());
                    probing = true;
                } else if (adaptive) {
                    // expected steps per millisecond of every width; ties go to the narrower round
                    double best_rate = -1.0;
                    int best_w = wa;
                    const double a = std::min(std::max(a_hat, 1e-3), 1.0);
                    for (int w : widths) {
                        auto it = t_round.find(w);
                        if (it == t_round.end() || it->second <= 0.0) continue;
                        const double rate = (1.0 - std::pow(1.0 - a, w)) / a / it->second;
                        if (rate > best_rate * 1.02) { best_rate = rate; best_w = w; }
                    }
                    wa = best_w;
                }
                // a batch: at most 128 rounds (the acceptance rate drifts), never past the end of the run
                int rounds = std::max(1, std::min(remaining / wa, adaptive ? (probing ? 8 : 128) : (1 << 30)));
                r.Wa = wa; r.Cn = Cr * wa;
                cudaGraphExec_t ex = nullptr;
                if (graphs) {
                    if (wa == W) ex = exec;
                    else {
                        auto it = ch->exec_wa.find(wa);
                        if (it == ch->exec_wa.end()) it = ch->exec_wa.emplace(wa, capture(nullptr)).first;
                        ex = it->second;
                    }
                }
                ICP_CUDA(cudaEventRecord(eb0, s));
                for (int k = 0; k < rounds; k++) {
                    if (ex) ICP_CUDA(cudaGraphLaunch(ex, s));
                    else enqueue_step(r);
                }
                ICP_CUDA(cudaEventRecord(eb1, s));
                rounds_total += rounds;
                launches_total += (int64_t)ch->last_per_step * rounds;
                long long steps1 = 0, acc1 = 0;
                read_counters(steps1, acc1, lo);
                float ms = 0.f;
                cudaEventElapsedTime(&ms, eb0, eb1);
                const double t = ms / rounds;
                auto it = t_round.find(wa);
                if (it == t_round.end()) t_round[wa] = t; else it->second = 0.5 * it->second + 0.5 * t;
                if (steps1 > steps0) {
                    const double a = (double)(acc1 - acc0) / (double)(steps1 - steps0);
                    a_hat = batches == 0 ? a : 0.5 * a_hat + 0.5 * a;
                }
                steps0 = steps1; acc0 = acc1;
                remaining = step_base + n_steps - lo;
                batches++;
            }
            if (batches > 0) ch->la_a_hat = a_hat;
        } catch (...) {
            cudaEventDestroy(eb0); cudaEventDestroy(eb1);
            throw;
        }
        cudaEventDestroy(eb0); cudaEventDestroy(eb1);
        r.Wa = W; r.Cn = C;
    } else {
        for (; steps_done < n_steps; steps_done++) {
            if (exec) ICP_CUDA(cudaGraphLaunch(exec, s));
            else enqueue_step(r);
            after_step(steps_done + 1);
        }
        rounds_total = n_steps;
        launches_total = (int64_t)ch->last_per_step * n_steps;
    }
    if (io->theta_final)   // look-ahead: lane 0 of every chain = the first Cr entries (all lanes hold the chain's state)
        ICP_CUDA(cudaMemcpyAsync(io->theta_final, ch->theta_cur.p, sizeof(double) * (size_t)Cr * Lt, cudaMemcpyDeviceToDevice, s));
    if (io->n_accepted)
        ICP_CUDA(cudaMemcpyAsync(io->n_accepted, ch->n_acc.p, sizeof(long long) * (size_t)Cr, cudaMemcpyDeviceToDevice, s));
    if (io->status)
        ICP_CUDA(cudaMemcpyAsync(io->status, ch->status.p, sizeof(int) * (size_t)Cr, cudaMemcpyDeviceToDevice, s));
    if (io->theta_best)
        ICP_CUDA(cudaMemcpyAsync(io->theta_best, ch->theta_best.p, sizeof(double) * (size_t)Cr * Lt, cudaMemcpyDeviceToDevice, s));
    if (io->value_best)
        ICP_CUDA(cudaMemcpyAsync(io->value_best, ch->value_best.p, sizeof(double) * (size_t)Cr, cudaMemcpyDeviceToDevice, s));
    ICP_CUDA(cudaEventRecord(ch->ev1, s));
    ch->resident_C = Cr;
    ch->resident_W = W;
    ch->steps_total = step_base + n_steps;
    ch->last_launches = launches_total;
    ch->last_rounds = rounds_total;
    if (!async) {
        ch->h_status.resize(Cr);
        ICP_CUDA(cudaMemcpyAsync(ch->h_status.data(), ch->status.p, sizeof(int) * (size_t)Cr, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        float ms = 0;
        cudaEventElapsedTime(&ms, ch->ev0, ch->ev1);
        ch->last_ms = ms;
    }
}

// The reference throws where a chain's status word is set; the batched runner finishes the run (the step is rejected, the
// other chains are unaffected), writes every output and then reports the first such chain through the return code.
void throw_on_chain_status(const std::vector<int> &st) {
    for (size_t c = 0; c < st.size(); c++) {
        const int v = st[c];
        if (!v) continue;
        std::string where = "chain " + std::to_string(c) + " (icp_chain_io.status has the per-chain words; outputs were written)";
        if (v & kStEmptySet) throw StatusError{ICP_ERR_EMPTY_SET, "empty filtered distance list in the collective evaluator, " + where};
        if (v & kStNotPD) throw StatusError{ICP_ERR_NOT_POSITIVE_DEFINITE, "posterior matrix not positive definite, " + where};
        if (v & kStNanTransition) throw StatusError{ICP_ERR_NAN, "NaN transition probability, " + where};
        throw StatusError{ICP_ERR_NAN, "NaN log-value of the initial state, " + where};
    }
}

}  // namespace

extern "C" int32_t icp_chain_run_device(icp_chain c, int32_t C, int32_t n_steps, const double *theta0_dev,
                                        const icp_chain_io *io_dev, int32_t async) {
    icp_ctx _ctx = c ? c->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        CtxLock lock(_ctx);
        chain_run_device(c, C, n_steps, theta0_dev, io_dev, async != 0);
        if (!async) throw_on_chain_status(c->h_status);
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_chain_run(icp_chain c, int32_t C, int32_t n_steps, const double *theta0, const icp_chain_io *io) {
    icp_ctx _ctx = c ? c->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        ICP_REQUIRE(theta0 && io, "null argument");
        CtxLock lock(_ctx);
        icp_model m = c->model;
        cudaStream_t s = _ctx->stream;
        const int K = m->K, Lt = K + kTheta0;
        ICP_REQUIRE(C >= 1 && C <= c->max_chains, "C must be in [1, max_chains]");
        size_t rec = (size_t)n_steps * C;
        DevBuf<double> &d_theta0 = c->d_theta0, &d_final = c->d_final;
        DevBuf<long long> &d_nacc = c->d_nacc;
        d_theta0.upload(theta0, (size_t)C * Lt, s);
        icp_chain_io dio = *io;
        bool host_rng = io->u_comp || io->z || io->u_acc;
        if (host_rng) {
            ICP_REQUIRE(io->u_comp && io->z && io->u_acc, "u_comp, z and u_acc must be given together");
            c->h_u_comp.upload(io->u_comp, rec, s); dio.u_comp = c->h_u_comp.p;
            c->h_z.upload(io->z, rec * K, s); dio.z = c->h_z.p;
            c->h_u_acc.upload(io->u_acc, rec, s); dio.u_acc = c->h_u_acc.p;
        }
        if (io->log_component) { c->h_log_comp.ensure(rec); dio.log_component = c->h_log_comp.p; }
        if (io->log_accepted) { c->h_log_acc.ensure(rec); dio.log_accepted = c->h_log_acc.p; }
        if (io->log_values) { c->h_log_values.ensure(3 * rec); dio.log_values = c->h_log_values.p; }
        if (io->log_theta) { c->h_log_theta.ensure(rec * Lt); dio.log_theta = c->h_log_theta.p; }
        if (io->theta_final) { d_final.ensure((size_t)C * Lt); dio.theta_final = d_final.p; }
        if (io->n_accepted) { d_nacc.ensure(C); dio.n_accepted = (int64_t *)d_nacc.p; }
        dio.status = nullptr;   // read from the chain's own status words below
        dio.theta_best = nullptr; dio.value_best = nullptr;   // likewise (chain-resident)
        const int n_rows = io->metrics_interval > 0 ? n_steps / io->metrics_interval : 0;
        if (io->metrics_interval > 0) {
            ICP_REQUIRE(io->log_metrics != nullptr, "metrics_interval > 0 needs log_metrics");
            c->h_log_metrics.ensure((size_t)std::max(n_rows, 1) * C * 4);
            dio.log_metrics = c->h_log_metrics.p;
        }
        // The log is [step][chain]: rows of finished steps are contiguous. When the caller's log buffers are pinned, rows
        // leave on a copy stream in up to 16 slices while later steps run; pageable buffers (cudaMemcpyAsync would block
        // the enqueueing thread) are copied after the last step.
        auto pinned = [](const void *h) {
            if (!h) return true;
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, h) != cudaSuccess) { cudaGetLastError(); return false; }
            return at.type == cudaMemoryTypeHost;
        };
        // (not with the rejection look-ahead: its rounds finish a varying number of steps, the rows are copied at the end)
        const bool overlap = n_steps >= 2 && (io->log_component || io->log_accepted || io->log_values || io->log_theta) &&
                             pinned(io->log_component) && pinned(io->log_accepted) && pinned(io->log_values) && pinned(io->log_theta) &&
                             lookahead_width(c, C, &dio, false, true) == 1;
        int copied = 0;
        auto copy_rows = [&](cudaStream_t cs, int s0, int s1) {
            const size_t o = (size_t)s0 * C, nrow = (size_t)(s1 - s0) * C;
            auto dl = [&](void *h, const void *d, size_t elem) {
                if (h && nrow) ICP_CUDA(cudaMemcpyAsync((char *)h + o * elem, (const char *)d + o * elem, nrow * elem, cudaMemcpyDeviceToHost, cs));
            };
            dl(io->log_component, c->h_log_comp.p, sizeof(int));
            dl(io->log_accepted, c->h_log_acc.p, 1);
            dl(io->log_values, c->h_log_values.p, sizeof(double) * 3);
            dl(io->log_theta, c->h_log_theta.p, sizeof(double) * Lt);
        };
        if (overlap) {
            if (!c->copy_stream) {
                ICP_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
                ICP_CUDA(cudaEventCreateWithFlags(&c->copy_ev, cudaEventDisableTiming));
            }
            const int slice = (n_steps + 15) / 16;
            std::function<void(int)> hook = [&](int done) {
                if (done - copied >= slice && done < n_steps) {
                    ICP_CUDA(cudaEventRecord(c->copy_ev, s));
                    ICP_CUDA(cudaStreamWaitEvent(c->copy_stream, c->copy_ev, 0));
                    copy_rows(c->copy_stream, copied, done);
                    copied = done;
                }
            };
            chain_run_device(c, C, n_steps, d_theta0.p, &dio, true, &hook);
        } else {
            chain_run_device(c, C, n_steps, d_theta0.p, &dio, true, nullptr, true);
        }
        copy_rows(s, copied, n_steps);
        auto dl = [&](void *h, const void *d, size_t bytes) {
            if (h && bytes) ICP_CUDA(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s));
        };
        dl(io->theta_final, d_final.p, sizeof(double) * (size_t)C * Lt);
        dl(io->n_accepted, d_nacc.p, sizeof(long long) * (size_t)C);
        c->h_status.resize(C);
        dl(c->h_status.data(), c->status.p, sizeof(int) * (size_t)C);
        dl(io->theta_best, c->theta_best.p, sizeof(double) * (size_t)C * Lt);
        dl(io->value_best, c->value_best.p, sizeof(double) * (size_t)C);
        if (n_rows > 0) dl(io->log_metrics, c->h_log_metrics.p, sizeof(double) * (size_t)n_rows * C * 4);
        ICP_CUDA(cudaStreamSynchronize(s));
        if (overlap) ICP_CUDA(cudaStreamSynchronize(c->copy_stream));
        {   // the run was enqueued asynchronously: device time of the K steps, as chain_run_device records it when it waits
            float ms = 0;
            cudaEventElapsedTime(&ms, c->ev0, c->ev1);
            c->last_ms = ms;
        }
        if (io->status) memcpy(io->status, c->h_status.data(), sizeof(int) * (size_t)C);
        throw_on_chain_status(c->h_status);
        return ICP_OK;
    } catch (...) {
        if (c && c->copy_stream) cudaStreamSynchronize(c->copy_stream);   // no copy into the caller's buffers may outlive the call
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_chain_last_run_stats(icp_chain c, double *device_ms, int64_t *kernel_launches) {
    if (!c) return ICP_ERR_INVALID_ARGUMENT;
    if (device_ms) *device_ms = c->last_ms;
    if (kernel_launches) *kernel_launches = c->last_launches;
    return ICP_OK;
}

extern "C" int32_t icp_chain_set_lookahead(icp_chain c, int32_t width) {
    if (!c || width < -1 || width > 32) return ICP_ERR_INVALID_ARGUMENT;
    icp_ctx _ctx = c->model->ctx;
    try {
        CtxLock lock(_ctx);
        c->lookahead = width;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" int32_t icp_chain_last_run_rounds(icp_chain c, int64_t *rounds) {
    if (!c || !rounds) return ICP_ERR_INVALID_ARGUMENT;
    *rounds = c->last_rounds;
    return ICP_OK;
}

extern "C" int32_t icp_chain_set_statistics(icp_chain c, const icp_chain_stats_params *p) {
    icp_ctx _ctx = c ? c->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        CtxLock lock(_ctx);
        if (p) {
            ICP_REQUIRE(p->take_every_n >= 1, "take_every_n must be >= 1");
            ICP_REQUIRE(p->burn_in >= 0, "burn_in must be >= 0");
            ICP_REQUIRE(p->normals == 0 || p->normals == 1, "normals must be 0 or 1");
            c->stats_req = *p;
        }
        c->stats_req_on = p != nullptr;
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

// Reads the maps without changing the accumulators: copies of the chains' partials take their pending weight (the current
// state) as one more flush, the partials are merged in chain order and finished with the direction chosen here.
extern "C" int32_t icp_chain_statistics(icp_chain c, int32_t chain, int32_t sum_normals, const double *theta_ref,
                                        int64_t *n_samples, double *mean, double *cov, double *total_variance,
                                        double *normal_variance) {
    icp_ctx _ctx = c ? c->model->ctx : nullptr;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        CtxLock lock(_ctx);
        ICP_REQUIRE(c->stats_on && c->resident_C > 0,
                    "statistics were off for the resident run (icp_chain_set_statistics, then a run from theta0)");
        const int Cr = c->resident_C;
        ICP_REQUIRE(chain >= -1 && chain < Cr, "chain must be -1 (pooled) or in [0, C) of the resident run");
        ICP_REQUIRE(!sum_normals || c->stats_run.normals, "sum_normals needs statistics accumulated with normals = 1");
        icp_model m = c->model;
        cudaStream_t s = _ctx->stream;
        const int N = m->N, Lt = m->K + kTheta0;
        const int c0 = chain < 0 ? 0 : chain, n = chain < 0 ? Cr : 1;
        const size_t nv = (size_t)n * N;
        const bool nrm = c->stats_run.normals != 0;
        DevBuf<long long> cnt, w, n_old;
        DevBuf<double> mu, q, ns, pmu, pq, pns, refX, refN, d_mean, tot7, d_cov, d_total, d_along;
        DevBuf<int> idx, nlist;
        cnt.alloc(n); w.alloc(n); n_old.alloc(n); idx.alloc(n); nlist.alloc(1);
        mu.alloc(nv * 3); q.alloc(nv * 6);
        ICP_CUDA(cudaMemcpyAsync(cnt.p, c->sx_count.p + c0, sizeof(long long) * n, cudaMemcpyDeviceToDevice, s));
        ICP_CUDA(cudaMemcpyAsync(mu.p, c->sx_mean.p + (size_t)c0 * N * 3, sizeof(double) * nv * 3, cudaMemcpyDeviceToDevice, s));
        ICP_CUDA(cudaMemcpyAsync(q.p, c->sx_m2.p + (size_t)c0 * N * 6, sizeof(double) * nv * 6, cudaMemcpyDeviceToDevice, s));
        if (nrm) {
            ns.alloc(nv * 3);
            ICP_CUDA(cudaMemcpyAsync(ns.p, c->sx_nsum.p + (size_t)c0 * N * 3, sizeof(double) * nv * 3, cudaMemcpyDeviceToDevice, s));
        }
        const StatsAcc acc{mu.p, q.p, nrm ? ns.p : nullptr};
        // the current state of every chain (look-ahead: lane 0 = the first Cr entries) with its pending weight
        launch_stats_pending(n, c->sx_pending.p + c0, cnt.p, w.p, n_old.p, s);
        c->X.ensure(nv * 3);
        launch_stats_flush(m->dev(), n, c->theta_cur.p + (size_t)c0 * Lt, w.p, n_old.p, idx.p, nlist.p, c->X.p, acc, s);
        std::vector<long long> h_cnt(n);
        ICP_CUDA(cudaMemcpyAsync(h_cnt.data(), cnt.p, sizeof(long long) * n, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        long long S = 0;
        for (long long v : h_cnt) S += v;
        if (n_samples) *n_samples = S;
        ICP_REQUIRE(S >= 1, "no selected record: the run has not reached burn_in (or end <= burn_in)");
        ICP_REQUIRE(S <= 0x7fffffffLL, "more than 2^31 - 1 samples");
        pmu.alloc((size_t)N * 3); pq.alloc((size_t)N * 6);
        if (nrm) pns.alloc((size_t)N * 3);
        launch_stats_pool(n, N, cnt.p, acc, pmu.p, pq.p, nrm ? pns.p : nullptr, s);
        const double *ref_normals = nullptr;
        if (!sum_normals) {
            // normals of transformedMesh(theta_ref), or of the model's reference mesh when theta_ref is NULL
            refN.alloc((size_t)N * 3);
            const double *rx = m->ref.p;
            DevBuf<double> th;
            if (theta_ref) {
                th.upload(theta_ref, (size_t)Lt, s);
                refX.alloc((size_t)N * 3);
                launch_reconstruct(m->dev(), 1, th.p, refX.p, s);
                rx = refX.p;
                ICP_CUDA(cudaStreamSynchronize(s));   // th leaves scope
            }
            launch_vertex_normals(m->dev(), 1, rx, refN.p, s);
            ref_normals = refN.p;
        }
        d_mean.alloc((size_t)N * 3); tot7.alloc((size_t)N * 7); d_cov.alloc((size_t)N * 9); d_total.alloc(N); d_along.alloc(N);
        launch_stats_moments(N, S, pmu.p, pq.p, nrm ? pns.p : nullptr, ref_normals, d_mean.p, tot7.p, s);
        launch_var_finish((int)S, N, tot7.p, d_cov.p, d_total.p, d_along.p, s);
        auto dl = [&](double *h, const double *d, size_t cnt_) {
            if (h) ICP_CUDA(cudaMemcpyAsync(h, d, cnt_ * sizeof(double), cudaMemcpyDeviceToHost, s));
        };
        dl(mean, d_mean.p, (size_t)N * 3); dl(cov, d_cov.p, (size_t)N * 9); dl(total_variance, d_total.p, N);
        dl(normal_variance, d_along.p, N);
        ICP_CUDA(cudaStreamSynchronize(s));
        return ICP_OK;
    } catch (...) {
        if (_ctx) cudaStreamSynchronize(_ctx->stream);   // no copy may outlive the call's buffers
        return translate_exception(_ctx);
    }
}

// Philox block exactly as the chain runner draws it (integer-exact check against the oracle)
__global__ void k_debug_philox(unsigned long long seed, unsigned long long chain, unsigned int step, unsigned int block,
                               unsigned int *out) {
    uint4 r = chain_philox(seed, chain, step, block);
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

extern "C" int32_t icp_debug_philox(icp_ctx ctx, uint64_t seed, uint64_t chain, uint32_t step, uint32_t block,
                                    uint32_t out[4]) {
    icp_ctx _ctx = ctx;
    try {
        ICP_REQUIRE(ctx && out, "null argument");
        CtxLock lock(ctx);
        DevBuf<unsigned int> d;
        d.alloc(4);
        k_debug_philox<<<1, 1, 0, ctx->stream>>>(seed, chain, step, block, d.p);
        ICP_CUDA(cudaGetLastError());
        ICP_CUDA(cudaMemcpyAsync(out, d.p, 16, cudaMemcpyDeviceToHost, ctx->stream));
        ICP_CUDA(cudaStreamSynchronize(ctx->stream));
        return ICP_OK;
    } catch (...) {
        return translate_exception(_ctx);
    }
}

extern "C" const char *icp_stage_name(int32_t stage) {
    static const char *names[ST_COUNT] = {"propose", "reconstruct", "closest_point_static", "bvh_refit",
                                          "nearest_dynamic", "observations", "posterior_build", "cholesky_solve",
                                          "eval_reduce", "accept", "other"};
    return (stage >= 0 && stage < ST_COUNT) ? names[stage] : "";
}

extern "C" int32_t icp_chain_profile(icp_chain c, int32_t C, int32_t n_steps, const double *theta0, uint64_t seed,
                                     double *stage_ms, int64_t *stage_launches) {
    icp_ctx _ctx = c ? c->model->ctx : nullptr;
    Profiler prof;
    try {
        ICP_REQUIRE(_ctx != nullptr, "null handle");
        ICP_REQUIRE(theta0 && stage_ms && stage_launches, "null argument");
        static_assert(ST_COUNT == ICP_N_STAGES, "stage table out of sync with the header");
        CtxLock lock(_ctx);
        cudaStream_t s = _ctx->stream;
        const int Lt = c->model->K + kTheta0;
        DevBuf<double> d_theta0;
        d_theta0.upload(theta0, (size_t)C * Lt, s);
        icp_chain_io io{};
        io.seed = seed;
        // warm-up (sizes the workspaces), then the profiled run
        chain_run_device(c, C, n_steps > 2 ? 2 : n_steps, d_theta0.p, &io, false);
        g_prof = &prof;
        chain_run_device(c, C, n_steps, d_theta0.p, &io, false);
        g_prof = nullptr;
        ICP_CUDA(cudaStreamSynchronize(s));
        prof.collect();
        for (int i = 0; i < ST_COUNT; i++) { stage_ms[i] = prof.ms[i]; stage_launches[i] = prof.launches[i]; }
        return ICP_OK;
    } catch (...) {
        g_prof = nullptr;
        prof.collect();
        return translate_exception(_ctx);
    }
}
