// icp_internal.h - internal structures and kernel launchers of libicpcuda.so (not part of the C ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/icpcuda.h"
#include "../../include/icpcuda_debug.h"

namespace icp {

constexpr int kTheta0 = 10;  // theta = [s, t3, rot3, c3, alpha_K]

inline int pad8(int k) { return (k + 7) & ~7; }

// ---- error plumbing ---------------------------------------------------------------------------
struct CudaError {
    cudaError_t e;
    const char *file;
    int line;
};
#define ICP_CUDA(x)                                                          \
    do {                                                                     \
        cudaError_t _e = (x);                                                \
        if (_e != cudaSuccess) throw icp::CudaError{_e, __FILE__, __LINE__}; \
    } while (0)

struct ArgError {
    std::string msg;
};
#define ICP_REQUIRE(cond, msg)                 \
    do {                                       \
        if (!(cond)) throw icp::ArgError{msg}; \
    } while (0)

struct StatusError {
    int32_t code;
    std::string msg;
};

// RAII device buffer (cudaMalloc on the current device)
uint64_t next_alloc_id();   // api.cu: process-wide counter, never 0

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    uint64_t id = 0;   // unique per allocation (next_alloc_id): a cached graph compares ids, not addresses, so an allocation
                       // that comes back at the same address after a free is still seen as new
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n), id(o.id) { o.p = nullptr; o.n = 0; o.id = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; id = o.id; o.p = nullptr; o.n = 0; o.id = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        id = 0;
    }
    void alloc(size_t count) {
        release();
        if (count == 0) count = 1;
        cudaError_t e = cudaMalloc((void **)&p, count * sizeof(T));
        if (e != cudaSuccess) {
            p = nullptr;
            throw CudaError{e, __FILE__, __LINE__};
        }
        n = count;
        id = next_alloc_id();
    }
    void ensure(size_t count) {
        if (count > n) alloc(count);
    }
    void upload(const T *h, size_t count, cudaStream_t s) {
        ensure(count);
        if (count) ICP_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s));
    }
};

// ---- per-stage device timing (CUDA events on the launching stream; enabled by icp_chain_profile) ----
enum Stage {
    ST_PROPOSE = 0, ST_RECONSTRUCT, ST_NEAREST_STATIC, ST_REFIT, ST_NEAREST_DYNAMIC, ST_OBSERVATIONS, ST_POSTERIOR_BUILD,
    ST_CHOLESKY, ST_EVAL_REDUCE, ST_ACCEPT, ST_OTHER, ST_COUNT
};
struct Profiler {
    struct Rec { int stage; cudaEvent_t e0, e1; };
    std::vector<Rec> recs;
    double ms[ST_COUNT] = {0};
    long long launches[ST_COUNT] = {0};
    void collect();  // after a stream synchronise: accumulates and frees the events
};
extern thread_local Profiler *g_prof;
struct ProfScope {
    int idx = -1;
    cudaStream_t s;
    ProfScope(int stage, cudaStream_t stream);
    ~ProfScope();
};

// Bounding-volume hierarchy: static topology (LBVH, Karras 2012) + one set of child boxes per
// instance. Internal nodes 0..n-2 (root 0); a child c >= 0 is an internal node, c < 0 is the
// leaf slot ~c in Morton order; prim[slot] is the original primitive id.
struct Bvh {
    int n = 0;               // leaves (>= 2; a single primitive is duplicated)
    int prim_kind = 0;       // 0 triangles, 1 points
    DevBuf<int2> children;   // [n-1]
    DevBuf<int> parent;      // [2n-1]: internal nodes then leaves (n-1+slot)
    DevBuf<int> prim;        // [n]
    DevBuf<float4> nodes;    // [instances][n-1][3] child boxes
    DevBuf<float4> packed;   // [n-1][4] boxes of the build-time positions + child links in one 64-byte record (static queries)
    DevBuf<float4> nodebox;  // scratch [instances][2n-1][2] full boxes (lo, hi)
    DevBuf<int> counters;    // scratch [instances][n-1] (atomic refit)
    DevBuf<int> order, level_off;  // internal nodes by increasing height + level boundaries (level-synchronous refit)
    int n_levels = 0;
    int instances = 0;
    float slack = 0.f;
};

// builds the topology from reference positions (verts N x 3 on the device; tris T x 3 or nullptr for
// a point BVH) and refits instance 0
void bvh_build(Bvh &b, int prim_kind, int n_prims, const double *d_verts, const int *d_tris, double scale,
               cudaStream_t s);
// refits `instances` sets of boxes from vertex positions X[instance][N][3]
void bvh_refit(Bvh &b, int instances, const double *d_X, int N, const int *d_tris, cudaStream_t s);

// L-ary collapse of a static triangle LBVH for the warp-cooperative traversal (bvh_wide.cu): n_nodes wide nodes in
// breadth-first order, each L child records of two float4 {lo.x, lo.y, lo.z, hi.x}, {hi.y, hi.z, reference, -}; a
// reference >= 0 is a wide node, < 0 encodes a leaf cluster ~((first slot << 3) | (count - 1)) of Morton-contiguous triangles
struct WideBvh {
    int L = 0, n_nodes = 0, n_leaves = 0;
    DevBuf<float4> nodes;
};
void wide_build(const Bvh &b, WideBvh &w, int L, cudaStream_t s);

// One target of a chain handle's target set (icp_chain_create_targets) as the device reads it: the static triangle BVH
// ([0]) and vertex BVH ([1]) of the target - packed nodes, leaf-slot -> primitive ids, Morton-ordered leaf data, leaf
// count - and its boundary table. The chain runner uploads one record per target and a target index per batch entry.
struct TargetRec {
    const float4 *nodes[2];
    const int *prim[2];
    const double *data[2];
    int n[2];
    const uint8_t *boundary;   // [Nt]
    int Nt;
};

struct NearestArgs {
    // structure
    const Bvh *bvh = nullptr;
    const WideBvh *wide = nullptr;      // static triangle structures: take the warp-cooperative kernel when set
    int sm_count = 148;
    const double *prim_data = nullptr;  // static: tri_data [slot][10] / vert_data [slot][4]; nullptr => dynamic
    const double *X = nullptr;          // dynamic: vertex positions [instance][N][3]
    const int *tris = nullptr;          // dynamic triangles
    int N = 0;                          // vertices per instance (dynamic) / per query mesh (gather)
    // queries: C x nq. Either gathered from a per-chain mesh (Xq + q_ids) or points (per chain or shared)
    int C = 1;
    int64_t nq = 0;
    const double *q = nullptr;      // [nq][3] shared, or [C][nq][3] when q_per_chain
    int q_per_chain = 0;
    const double *Xq = nullptr;     // [C][Nq][3]
    const int *q_ids = nullptr;     // [nq]
    int Nq = 0;
    const int *perm = nullptr;      // optional processing order (C == 1): thread g handles query perm[g]
    // optional [C][nq], read and rewritten: leaf slot of the query's previous answer (any value; out of range = none).
    // The traversal starts from the exact distance to that primitive, which prunes most of the tree when the query
    // moved little since (successive MH states of a chain). The result does not depend on it.
    int *seed_slot = nullptr;
    // optional [C], Hausdorff evaluator only (distance-only triangle queries): running maximum of the exact squared
    // distances of the chain (bits of a non-negative double, zeroed by the caller); queries that cannot raise it stop early
    // and write an upper bound instead of the exact distance (see k_nearest)
    unsigned long long *chain_max = nullptr;
    // outputs [C][nq]
    int *out_prim = nullptr;
    int *out_feat = nullptr;
    double *out_cp = nullptr;
    double *out_d2 = nullptr;
    // several static targets in one launch: query row c walks the structure of record mt_rec[mt_idx[c]] (the triangle BVH
    // for triangle queries, the vertex BVH for point queries) instead of bvh / prim_data, which then only give the
    // primitive kind. Never takes the warp-cooperative kernel.
    const TargetRec *mt_rec = nullptr;
    const int *mt_idx = nullptr;
};
void launch_nearest(const NearestArgs &a, cudaStream_t s);
// false: the arguments are outside the wide kernel's domain (nothing launched)
bool launch_nearest_wide(const NearestArgs &a, int sm_count, cudaStream_t s);
// scratch of the query-ordering pass of large point batches
struct QuerySort {
    DevBuf<unsigned int> keys, keys2;
    DevBuf<int> vals, perm;
    DevBuf<unsigned char> tmp;
};
// like launch_nearest for free query points; batches >= 16384 are processed in Morton order (lo / hi: bounding box of
// the structure). Results are written in the caller's order either way.
void launch_nearest_sorted(NearestArgs a, QuerySort &qs, const double lo[3], const double hi[3], cudaStream_t s);
// nearest vertex of C per-chain meshes X[C][N][3] through the model's vertex BVH refitted in shared memory (one CTA per
// chain); d_seed (nullable) [C][nq] carries each query's previous leaf slot. false: does not fit, nothing launched
bool launch_nearest_vertex_tree(const Bvh &b, int N, int C, const double *d_X, int64_t nq, const double *d_q, int q_per_chain,
                                int *d_seed, int *d_prim, double *d_d2, cudaStream_t s);
// brute-force nearest vertex of C small meshes X[C][N][3] (FP32 screening + exact FP64); returns false (nothing
// launched) when N is too large for the shared-memory tile, in which case the caller uses the vertex BVH
// the domains of the two kernels above (what launch_* checks before launching)
bool nearest_vertex_tree_fits(const Bvh &b, int N);
bool nearest_vertex_brute_fits(int N);
bool launch_nearest_vertex_brute(int N, int C, const double *d_X, int64_t nq, const double *d_q, int q_per_chain, double scale,
                                 int *d_prim, double *d_d2, cudaStream_t s);

// ---- model kernels ---------------------------------------------------------------------------------
struct ModelDev {  // plain device view, passed by value to kernels
    int N, T, K, Kp;
    const double *ref, *mean, *Q, *QT, *S;  // mean: mean deformation (3N)
    const int *tris, *adj_off, *adj;
    const uint8_t *boundary;
};
void launch_reconstruct(const ModelDev &m, int C, const double *d_theta, double *d_X, cudaStream_t s);
void launch_vertex_normals(const ModelDev &m, int C, const double *d_X, double *d_normals, cudaStream_t s);
void launch_gram(const ModelDev &m, double *d_G /*Kp x Kp*/, cudaStream_t s);

// ---- posterior variability accumulated inside the chain runner (stats.cu) ------------------------------------------
struct StatsAcc {   // per-chain accumulators: mean [C][N][3], centred second moment [C][N][6] (xx yy zz xy xz yz), unit-normal sum
    double *mean, *m2, *nsum;   // [C][N][3] (nullable)
};
// one weighted Welford / Chan update of every chain c with d_w[c] > 0: the mesh of d_theta[c] (and its unit vertex normals)
// with weight d_w[c] into accumulators that held d_n_old[c] samples. d_idx [C] / d_count [1]: scratch for the list of those
// chains; d_X: [C][N][3] scratch for their meshes.
void launch_stats_flush(const ModelDev &m, int C, const double *d_theta, const long long *d_w, const long long *d_n_old,
                        int *d_idx, int *d_count, double *d_X, const StatsAcc &acc, cudaStream_t s);
// w = pending, n_old = count, count += pending (the read-out merges the chains' pending weight into copies)
void launch_stats_pending(int C, const long long *d_pending, long long *d_count, long long *d_w, long long *d_n_old, cudaStream_t s);
// Chan's merge of the C chains' partials in chain order into [N] arrays (d_nsum / acc.nsum nullable together)
void launch_stats_pool(int C, int N, const long long *d_count, const StatsAcc &acc, double *d_mean, double *d_m2, double *d_nsum,
                       cudaStream_t s);
// mean out and the [N][7] moments k_var_finish reads, along the reference normals or (NULL) the mean unit normal d_nsum / S
void launch_stats_moments(int N, long long S, const double *d_mean, const double *d_m2, const double *d_nsum, const double *d_ref_normals,
                          double *d_mean_out, double *d_tot7, cudaStream_t s);
// k_var_finish (comm.cu): [N][7] moments of S samples -> cov [N][9], total [N], along [N]
void launch_var_finish(int S, int N, const double *d_tot7, double *d_cov, double *d_total, double *d_along, cudaStream_t s);
void launch_scale_basis(int rows, int K, int Kp, const double *d_U, const double *d_var, double *d_Q, double *d_QT,
                        cudaStream_t s);

// ---- posterior / proposal kernels -------------------------------------------------------------------
struct ObsDev {  // observation list of one ICP proposal for C chains, stride n per chain
    int n;       // slots per chain (n_ids or n_tp)
    int *vid;    // [C][n] reference vertex id (-1: filtered out)
    double *F;   // [C][n][9] rows n/sd_n, t1/sd_t, t2/sd_t of the whitening frame
    double *y;   // [C][n][3] F (y_i - mean_i)
    int *nobs;   // [C] observations kept
    int *nrows = nullptr;  // [C] leading slots in use (<= n; observations of one vertex may share a slot); null: n
};
struct ObsArgs {
    ModelDev m;
    icp_proposal_params prm;
    int C;
    const double *theta;   // [C][K+10]
    const double *X;       // [C][N][3]
    // model sampling: closest points of the sampled vertices on the target
    const int *ids;        // [n]
    const double *cp;      // [C][cp_stride][3]; observation i reads entry cp_map[i] (or i when cp_map is null)
    int cp_stride;
    const int *cp_map;
    const uint8_t *cp_on_boundary;  // [C][n] or nullptr
    // target sampling: nearest current-mesh vertex per target point
    const double *tp;      // [n][3], or [C][n][3] when tp_per_chain
    int tp_per_chain;
    const int *near_vid;   // [C][n]
    int iso;               // 1: isotropic noise sigma2 (deterministic ICP), frame = I / sqrt(sigma2)
    double iso_sigma2;
    int world_frame;       // 1: the observation is target point - reference point as it is, NOT pulled back through the inverse
                           // pose (IcpBasedSurfaceFitting.scala:81 regresses the untransformed model on world-frame targets)
};
void launch_observations(const ObsArgs &a, const ObsDev &o, cudaStream_t s);
// M = I + sum_i (F_i Q_i)^T (F_i Q_i) (lower + upper, Kp x Kp, identity on the padding), b = sum (F_i Q_i)^T y_i
// constant-Gram fast path of the posterior build (see k_posterior_build_mma): Gs = sum_i Q_i^T Q_i over the
// proposal's model points, gs_scale = 1 / sd_t^2, row_scale = sqrt(1 - sd_n^2 / sd_t^2)
struct GramFast {
    const double *Gs;
    double gs_scale, row_scale;
};
void launch_posterior_build(const ModelDev &m, int C, const ObsDev &o, double *d_M, double *d_b, cudaStream_t s,
                            const GramFast *gf = nullptr);
void launch_gram_rows(const ModelDev &m, int n_ids, const int *d_ids, double *d_G, cudaStream_t s);
// Transition density of the chain runner that belongs to the posterior being built, formed while the factor is still in
// shared memory: out[c] = |L_c^T d|^2, d = (theta_post + (theta_other - theta_post) / step)[alpha] - mu_c
// (logTransitionProbability(theta_post -> theta_other), NonRigidIcpProposal.scala:76-83)
struct QuadArgs {
    const double *theta_post;    // [C][K+10] the state the posterior belongs to
    const double *theta_other;   // [C][K+10] the other end of the transition
    double step;
    int K;
    double *out;                 // [C]
};
// qa (nullable): also the quadratic form above; *quad_done tells whether the launched path formed it (the caller runs
// launch_quad_form otherwise)
// ymean (every factorisation entry below): d_mu receives y = L^-1 b instead of mu = L^-T y, and the quadratic form is
// |L^T w - y|^2 with w = theta_post + (theta_other - theta_post) / step - the chain runner's mean slot (it needs neither mu
// nor the back substitution that forms it)
bool launch_posterior_fused(const ModelDev &m, int C, const ObsDev &o, const GramFast *gf, double *d_M_or_null, double *d_L,
                            double *d_mu, const int *d_out_slot, int *d_status, double *d_Mp, double *d_b, cudaStream_t s,
                            const QuadArgs *qa = nullptr, bool *quad_done = nullptr, bool ymean = false);
// rank update on the INT8 tensor cores (tc_i8.cu): block-packed M and b like the DMMA rank update.
// I8Model: the basis with every column divided by its bound (max over the vertices of |Q_v[:, j]|) and the bounds;
// I8Scale: frame multiplier that brings the whitened rows into |x| <= 2^30 and the factors that undo it.
// false: shape outside the kernel's domain, nothing launched
struct I8Model { const double *Qhat, *colnorm, *Qsub; };   // Qsub (nullable): the proposal's rows packed by launch_pack_obs_rows
struct I8Scale { double fmul, w2, bscale; };
bool launch_rank_update_i8(const ModelDev &m, int C, const ObsDev &o, const GramFast *gf, const I8Model &im, const I8Scale &sc,
                           double *d_Mp, double *d_b, int n_sm, cudaStream_t s);
void launch_unit_basis(int rows, int Kp, const double *d_Q, const double *d_colnorm, double *d_Qhat, cudaStream_t s);
void launch_pack_obs_rows(int n, int Kp, const int *d_ids, const double *d_Qhat, double *d_Qsub /* [n][3 Kp + 2] */, cudaStream_t s);
// k_cholesky_packed on a block-packed M (the second half of launch_posterior_fused's default path)
void launch_cholesky_packed(int C, int Kp, const double *d_Mp, const double *d_b, double *d_M_or_null, double *d_L, double *d_mu,
                            const int *d_out_slot, int *d_status, const QuadArgs *qa, bool ymean, cudaStream_t s);
// the same quadratic form from L / mu (ymean: y) in global memory (paths whose factorisation kernel does not form it)
void launch_quad_form(int C, int Kp, const double *d_L, const double *d_mu, const int *d_slot, const QuadArgs &qa, bool ymean,
                      cudaStream_t s);
// in: M (C x Kp x Kp), b (C x Kp). out: L (lower Cholesky factor, C x Kp x Kp), mu = M^-1 b, status (0 ok)
// out_slot (nullable): chain c writes L / mu at index out_slot[c] instead of c
// d_Mp: scratch for the block-packed lower triangle (C x NB (NB + 1) / 2 x 64 doubles), needed when Kp > 160
void launch_cholesky_solve(int C, int K, int Kp, const double *d_M, const double *d_b, double *d_L, double *d_mu,
                           const int *d_out_slot, int *d_status, cudaStream_t s, double *d_Mp = nullptr,
                           const QuadArgs *qa = nullptr, bool *quad_done = nullptr, bool ymean = false);
// alpha' = alpha + step (S (mu + L^-T z) - alpha); L/mu addressed through per-chain slot indices
// d_W (nullable): explicit factor [slot][Kp][Kp] (ICP_FACTOR_SVD); alpha' then uses W z instead of L^-T z
void launch_propose(const ModelDev &m, int C, double step, const double *d_theta, const double *d_z,
                    const double *d_L, const double *d_mu, const int *d_slot, double *d_theta_out, cudaStream_t s,
                    const double *d_W = nullptr);
// the reference's covariance factor W = D^-1 Ubar diag(sqrt(lambda')) of C posteriors from their Cholesky factors
// (svdfactor.cu); L / W addressed through d_slot (nullable); scratch is grown when the matrices do not fit shared memory
void launch_svd_factor(int C, int K, int Kp, const double *d_L, const double *d_sqrt_var, const int *d_slot, double *d_W,
                       DevBuf<double> &scratch, cudaStream_t s);
// -1/2 (K ln 2pi + |L^T (alpha_c - mu)|^2), -inf unless only alpha changed
void launch_log_transition(int C, int K, int Kp, double step, const double *d_from, const double *d_to,
                           const double *d_L, const double *d_mu, const int *d_slot, double *d_out, cudaStream_t s);

// ---- evaluator kernels ------------------------------------------------------------------------------
struct EvalReduceArgs {
    icp_evaluator_params prm;
    int C, K;
    const double *theta;        // [C][K+10]
    // model -> target distances (squared) [C][n_m2t], optional boundary flags of the hit
    int n_m2t;
    const double *d2_m2t;
    const uint8_t *skip_m2t;
    // target -> model
    int n_t2m;
    const double *d2_t2m;
    const uint8_t *skip_t2m;
    double *values;             // [C][3] product, prior, distance
    int *status;                // [C] or nullptr
};
void launch_eval_reduce(const EvalReduceArgs &a, cudaStream_t s);
void launch_prior(int C, int K, const double *d_theta, double *d_out, cudaStream_t s);
// flags[c][i] = table[prim[c][i]]; with rec / tidx (several targets) the table of row c is rec[tidx[c]].boundary, rows of
// `per` entries
void launch_lookup_flags(int64_t n, const int *d_prim, const uint8_t *d_table, int table_n, uint8_t *d_flags,
                         cudaStream_t s, const TargetRec *rec = nullptr, const int *tidx = nullptr, int64_t per = 1);

}  // namespace icp

// ---- handles ------------------------------------------------------------------------------------
struct icp_ctx_s {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    static constexpr int kAux = 3;          // side streams: independent pipelines of one MH step run concurrently
    cudaStream_t aux[kAux] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[kAux] = {nullptr, nullptr, nullptr};
    std::mutex mu;                          // serialises calls on ctx->stream and on the scratch shared through models / targets
    std::mutex err_mu;                      // guards err (calls on different handles run concurrently)
    std::string err;
    std::string device_name;
};

struct icp_model_s {
    std::mutex props_mu;
    std::vector<icp_proposal> proposals;   // live proposals built on this model (siblings for the speculative posterior)
    icp_ctx ctx = nullptr;
    int refs = 0;                     // proposals / evaluators / chains built on this handle (destroy refuses while > 0)
    int N = 0, T = 0, K = 0, Kp = 0;  // Kp = K padded to a multiple of 8
    icp::DevBuf<double> ref;          // N x 3
    icp::DevBuf<double> mean;         // 3N: mean deformation
    icp::DevBuf<double> Q;            // 3N x Kp row-major, scaled basis, zero padded
    icp::DevBuf<double> QT;           // Kp x 3N
    icp::DevBuf<double> S;            // Kp x Kp, Appendix A5 constant (identity on the padding)
    icp::DevBuf<double> sqrt_var;     // Kp: sqrt(lambda) (1 on the padding)
    icp::DevBuf<double> Qhat, col_norm;  // INT8 rank update (tc_i8.cu): Q with unit column bounds (3N x Kp), the bounds (Kp)
    std::vector<double> h_col_norm;   // Kp: max over the vertices of |Q_v[:, j]|_2 (column bound of the INT8 rank update)
    std::vector<double> h_var;        // K
    icp::DevBuf<int> tris;            // T x 3
    icp::DevBuf<int> adj_off, adj;    // vertex -> triangles CSR (ascending triangle id)
    icp::DevBuf<uint8_t> boundary;    // N
    bool has_boundary = false;
    std::vector<uint8_t> h_boundary;
    std::vector<double> h_mean_def;
    std::vector<double> h_ref;        // reference vertices (host copy: spatial ordering of query lists)
    double scale = 1.0;               // max |coordinate| of the reference mesh (box slack)
    icp::Bvh tri_bvh, vert_bvh;       // topology from the reference mesh, boxes refit per chain
    icp::ModelDev dev() const {
        return icp::ModelDev{N, T, K, Kp, ref.p, mean.p, Q.p, QT.p, S.p, tris.p, adj_off.p, adj.p, boundary.p};
    }
    // scratch for primitive calls (guarded by mu)
    icp::DevBuf<double> s_theta, s_X, s_q, s_d;
    icp::DevBuf<int> s_i;
};

struct icp_target_s {
    icp_ctx ctx = nullptr;
    int refs = 0;
    int Nt = 0, Tt = 0;
    icp::DevBuf<double> verts;      // Nt x 3
    icp::DevBuf<int> tris;          // Tt x 3
    icp::DevBuf<double> tri_data;   // [leaf slot][10]: a b c (9 doubles) + pad, Morton order
    icp::DevBuf<double> vert_data;  // [leaf slot][4]: xyz + pad, Morton order
    icp::DevBuf<uint8_t> boundary;  // Nt
    icp::DevBuf<double> vnormals;   // Nt x 3 vertex normals (Scalismo vertexNormals; inside test of the Dice coefficient)
    bool has_boundary = false;
    std::vector<uint8_t> h_boundary;
    icp::Bvh tri_bvh, vert_bvh;
    icp::WideBvh tri_wide;          // L-ary collapse of tri_bvh (empty when ICPCUDA_WIDE=0)
    const icp::WideBvh *wide() const { return tri_wide.n_nodes > 0 ? &tri_wide : nullptr; }
    icp::QuerySort qsort;
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};   // bounding box of the vertices
    icp::DevBuf<double> s_q, s_d;
    icp::DevBuf<int> s_i;
};

namespace icp {

// per-batch workspace of the correspondence + posterior pipeline of one ICP proposal
struct PosteriorWork {
    int C = 0;
    DevBuf<double> X;        // [C][N][3]
    DevBuf<double> cp, d2;   // [C][n][3], [C][n]
    DevBuf<int> prim;        // [C][n]
    DevBuf<int> seed;        // [C][n] traversal seeds (NearestArgs::seed_slot)
    DevBuf<uint8_t> flags;   // [C][n]
    DevBuf<int> vid;
    DevBuf<double> F, y;
    DevBuf<int> nobs;
    DevBuf<double> M, b;     // [C][Kp*Kp], [C][Kp]
    DevBuf<double> Mp;       // [C][NB (NB + 1) / 2][64] block-packed lower triangle of M (rank update -> factorisation)
    bool want_M = false;     // the primitive API returns M; the chain runner never needs it in global memory
    DevBuf<int> status;
    DevBuf<double> svd_scratch;   // ICP_FACTOR_SVD at ranks whose matrices do not fit shared memory
};

}  // namespace icp

namespace icp {
// One in-flight per-call entry (icp_propose / icp_log_transition / icp_posterior / icp_eval_log_value) on a handle: its own
// stream and scratch. The reference shares ONE proposal and ONE evaluator object between its ten fitting threads
// (RunMHRandomInitComparison.scala:59-86); a handle whose pipeline touches no scratch of its model (proposal_self_contained /
// evaluator_self_contained in api.cu) keeps a small pool of these, so concurrent calls on the same handle overlap on the GPU.
// page-locked host staging of a call slot: inputs and outputs of a per-call entry travel through it, so the copies are
// plain asynchronous copies (and graph nodes with fixed addresses)
struct PinnedBuf {
    char *p = nullptr;
    size_t n = 0;
    uint64_t id = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf &) = delete;
    PinnedBuf &operator=(const PinnedBuf &) = delete;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    void ensure(size_t bytes) {
        if (bytes <= n) return;
        bytes = (std::max(bytes, 2 * n) + 4095) & ~(size_t)4095;   // grow geometrically: every growth invalidates the slot's graphs
        if (p) cudaFreeHost(p);
        p = nullptr; n = 0; id = 0;
        cudaError_t e = cudaHostAlloc((void **)&p, bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) { p = nullptr; throw CudaError{e, __FILE__, __LINE__}; }
        n = bytes;
        id = next_alloc_id();
    }
};
struct CallSlotBase {
    std::mutex mu;                // held for the duration of one call
    cudaStream_t stream = nullptr;
    PinnedBuf h_in, h_out, h_aux;
    // The work of one entry point at one batch size, captured once as a CUDA graph (host -> device copies out of h_in, the
    // kernels, device -> host copies into h_out) and replayed: one graph launch + one synchronise per call instead of
    // 10 - 20 runtime calls, which is what bounds C = 1 calls from several host threads (they serialise in the driver).
    // The first call with a key runs eagerly (it sizes the scratch), the second is captured; a graph is dropped when any
    // allocation it baked in has been replaced since (ids).
    struct Graph {
        cudaGraphExec_t exec = nullptr;
        std::vector<uint64_t> ids;
        bool seen = false, eager_only = false;
    };
    std::unordered_map<uint64_t, Graph> graphs;
    ~CallSlotBase() {
        for (auto &g : graphs)
            if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
        if (stream) cudaStreamDestroy(stream);
    }
};
// body() enqueues the work on s. graph = false: just that. Otherwise replay / capture as described above.
template <class F>
void run_call_graph(CallSlotBase &cs, bool graph, uint64_t key, const std::vector<uint64_t> &ids, cudaStream_t s, F &&body) {
    if (!graph) { body(); return; }
    CallSlotBase::Graph &g = cs.graphs[key];
    if (g.eager_only) { body(); return; }
    if (g.exec && g.ids != ids) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; g.seen = false; }
    if (g.exec) { ICP_CUDA(cudaGraphLaunch(g.exec, s)); return; }
    if (!g.seen) { body(); g.seen = true; return; }   // sizes every buffer the body touches
    cudaGraph_t graph_obj = nullptr;
    if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); body(); return; }
    bool ok = true;
    try { body(); } catch (...) { ok = false; }
    cudaError_t e = cudaStreamEndCapture(s, &graph_obj);
    cudaGraphExec_t exec = nullptr;
    if (ok && e == cudaSuccess && graph_obj && cudaGraphInstantiate(&exec, graph_obj, 0) != cudaSuccess) exec = nullptr;
    if (graph_obj) cudaGraphDestroy(graph_obj);
    if (!exec) {            // not capturable in this configuration: stay eager for this key
        cudaGetLastError();
        g.eager_only = true;
        body();
        return;
    }
    g.exec = exec;
    g.ids = ids;
    ICP_CUDA(cudaGraphLaunch(exec, s));
}
constexpr int kMaxCallSlots = 16;
}  // namespace icp

struct icp_proposal_s {
    int refs = 0;             // chains using this proposal
    icp_model model = nullptr;
    icp_target target = nullptr;
    icp_proposal_params prm{};
    int n_ids = 0, n_tp = 0;
    icp::DevBuf<int> ids;     // n_ids
    icp::DevBuf<double> tp;   // n_tp x 3
    icp::DevBuf<int> qperm;   // processing order of the model points (Morton order of their reference positions)
    icp::DevBuf<double> Gs;   // Kp x Kp: sum of Q_i^T Q_i over the model points (constant-Gram fast path), empty if unused
    icp::DevBuf<double> Qsub; // [n_ids][3 Kp + 2]: the model points' unit-bound basis rows in slot order (INT8 rank update of the constant-Gram path)
    bool gram_fast = false;
    // posterior cache (the reference's Memoize(icpPosterior, 20)): theta bytes -> slot
    int cache_slots = 0;
    std::unordered_map<std::string, int> cache_map;
    std::vector<std::string> slot_key;
    std::vector<int> slot_nobs, slot_status;
    int cache_next = 0;
    icp::DevBuf<double> cache_L, cache_mu, cache_M;  // [slots][Kp*Kp], [slots][Kp], [slots][Kp*Kp]
    icp::DevBuf<double> cache_W;                     // [slots][Kp*Kp] (ICP_FACTOR_SVD only)
    // the cache is shared by the concurrent calls: cache_rw is held shared for the length of a call and exclusively while the
    // slot arrays are (re)allocated; cache_lock guards the map and the per-slot state; a slot is pinned while a call uses it and
    // not ready while the call that missed on it is still computing it (other calls with the same key wait on cache_cv)
    std::shared_mutex cache_rw;
    std::mutex cache_lock;
    std::condition_variable cache_cv;
    std::vector<int> slot_pin;
    std::vector<char> slot_ready;
    icp::PosteriorWork work;  // scratch of icp_std_icp_iteration's temporary proposal
    struct Call : icp::CallSlotBase {
        icp::PosteriorWork work;
        icp::DevBuf<double> s_theta, s_theta2, s_z, s_out, s_L, s_mu;
        icp::DevBuf<int> s_slot, s_qslot;
    };
    std::mutex pool_mu;
    std::vector<std::unique_ptr<Call>> calls;
    unsigned next_call = 0;
    // Speculative posterior of the state a proposal just produced (api.cu: prefetch_posterior): a Metropolis-Hastings host asks
    // every ICP component for logTransitionProbability(theta', theta) right after propose(theta) returned theta', which needs
    // the posterior AT theta'. icp_propose therefore starts that posterior on every self-contained proposal of the same model
    // and target in the background (own call slot, no synchronisation) - a pure cache fill: the later call finds the entry "in
    // flight" and waits for the rest of it instead of starting it. One computation in flight per proposal.
    std::mutex bg_mu;                 // guards the fields below; lock order: cache_rw -> bg_mu -> cache_lock
    std::unique_ptr<Call> bg_call;
    cudaEvent_t bg_ev = nullptr;
    bool bg_busy = false;
    std::vector<int> bg_slots;        // cache slots the computation in flight fills (pinned, not ready)
    std::vector<std::string> bg_keys;
    std::vector<char> slot_bg;        // [cache_slots] 1: being filled by the background computation
    ~icp_proposal_s() { if (bg_ev) cudaEventDestroy(bg_ev); }
};

namespace icp {
struct EvalWork {
    DevBuf<unsigned long long> hd_max;   // [C] running maxima of the Hausdorff evaluator's two traversals (NearestArgs::chain_max)
    DevBuf<double> X, cp_m2t, d2_m2t, cp_t2m, d2_t2m;
    DevBuf<int> prim, seed_m2t, seed_t2m;   // seed_*: traversal seeds (NearestArgs::seed_slot)
    DevBuf<uint8_t> skip_m2t, skip_t2m;
    bool force_cp_m2t = false;  // also keep the model->target closest points (shared with ICP proposals)
};
}  // namespace icp

struct icp_evaluator_s {
    int refs = 0;
    icp_model model = nullptr;
    icp_target target = nullptr;
    icp_evaluator_params prm{};
    int n_ids = 0, n_tp = 0;
    icp::DevBuf<int> ids;
    icp::DevBuf<int> qperm;   // processing order of the model points (Morton order of their reference positions)
    icp::DevBuf<double> tp;
    struct Call : icp::CallSlotBase {
        icp::EvalWork work;
        icp::DevBuf<double> s_theta, s_values;
        icp::DevBuf<int> s_status;
    };
    std::mutex pool_mu;
    std::vector<std::unique_ptr<Call>> calls;
    unsigned next_call = 0;
};

namespace icp {
// workspace of registration_metrics_device
struct MetricsWork {
    DevBuf<double> X, d2a, cpa, d2b;
    DevBuf<int> prim;
    DevBuf<uint8_t> skip;
};
// RegistrationComparison measures of C parameter vectors on the device: d_out [C][4] = {avg, hausdorff,
// avg_boundary_aware, max_boundary_aware}
void registration_metrics_device(icp_model m, icp_target t, int C, const double *d_theta, double *d_out, MetricsWork &w,
                                 cudaStream_t s);
void nearest_model_vertex(icp_model m, int C, const double *d_X, int64_t nq, const double *d_q, int q_per_chain, int *d_seed,
                          int *d_prim, cudaStream_t s);
// correspondence + posterior pipeline: L / mu (at out_slot[c] or c) for C parameter vectors on the device.
// d_X: transformed meshes [C][N][3] if the caller already has them, else nullptr.
// shared: closest points another consumer already computed for a superset of this proposal's model points
// (the evaluator's model->target queries in the chain runner); nullptr = run the traversal here.
struct SharedCp {
    const double *cp;   // [C][stride][3]
    int stride;
    const int *map;     // [n_ids] index into the shared list
};
// Several targets in one batch (the chain runner of a target set): entry c of the batch fits target rec[tidx[c]], and a
// consumer whose point list belongs to the target reads the entry's own copy tp [C][n_tp][3]. has_boundary is the OR over
// the targets: it decides the boundary path (no closest-point sharing, no constant-Gram path) for every entry.
struct TargetSet {
    const TargetRec *rec;   // [G]
    const int *tidx;        // [C]
    bool has_boundary;
    const double *tp;       // [C][n_tp][3] (target sampling / the evaluator's target -> model queries), else null
    int n_tp;               // entries per row of tp (the Hausdorff evaluator: the largest Nt, shorter lists padded)
};
// d_W (nullable, [slot][Kp][Kp]): also the reference's SVD-based covariance factor (ICP_FACTOR_SVD)
// ymean: d_mu receives y = L^-1 b instead of mu (see launch_posterior_fused); only the chain runner asks for it
void posterior_pipeline(icp_proposal p, int C, const double *d_theta, const double *d_X, PosteriorWork &w, double *d_L,
                        double *d_mu, const int *d_out_slot, cudaStream_t s, const SharedCp *shared = nullptr,
                        double *d_W = nullptr, const QuadArgs *qa = nullptr, bool ymean = false, const TargetSet *ts = nullptr);
// distance evaluator pipeline: values [C][3] = {product, prior, distance}; ts: see TargetSet
void evaluator_pipeline(icp_evaluator e, EvalWork &w, int C, const double *d_theta, const double *d_X, double *d_values,
                        int *d_status, cudaStream_t s, const TargetSet *ts = nullptr);
// RAII: selects the context device, serialises calls on the context
struct CtxLock {
    std::unique_lock<std::mutex> lk;
    explicit CtxLock(icp_ctx c);
};
// RAII of a per-call entry point on a proposal / evaluator handle: selects the device and leases one of the handle's call
// slots (a free one, a new one while the pool is below kMaxCallSlots, else it waits for one). A handle that is not
// self-contained takes the context lock first (lock order: context, then slot) and runs on ctx->stream like every other call.
template <class Handle>
struct CallLease {
    std::unique_lock<std::mutex> ctx_lk, lk;
    typename Handle::Call *call = nullptr;
    cudaStream_t stream = nullptr;
    CallLease(icp_ctx c, Handle *h, bool self_contained) {
        if (!self_contained) ctx_lk = std::unique_lock<std::mutex>(c->mu);
        cudaError_t e = cudaSetDevice(c->device);
        if (e != cudaSuccess) throw CudaError{e, __FILE__, __LINE__};
        {
            std::unique_lock<std::mutex> pool(h->pool_mu);
            for (auto &cs : h->calls) {
                std::unique_lock<std::mutex> t(cs->mu, std::try_to_lock);
                if (t.owns_lock()) { call = cs.get(); lk = std::move(t); break; }
            }
            if (!call && (int)h->calls.size() < kMaxCallSlots) {
                std::unique_ptr<typename Handle::Call> cs(new typename Handle::Call());
                e = cudaStreamCreateWithFlags(&cs->stream, cudaStreamNonBlocking);
                if (e != cudaSuccess) throw CudaError{e, __FILE__, __LINE__};
                call = cs.get();
                lk = std::unique_lock<std::mutex>(cs->mu);
                h->calls.push_back(std::move(cs));
            }
            if (!call) call = h->calls[h->next_call++ % h->calls.size()].get();
        }
        if (!lk.owns_lock()) lk = std::unique_lock<std::mutex>(call->mu);   // every slot busy: queue on one
        stream = ctx_lk.owns_lock() ? c->stream : call->stream;
    }
};
// waits for the calls in flight on a handle (destroy; the context lock is held)
template <class Handle>
void drain_calls(Handle *h) {
    std::unique_lock<std::mutex> pool(h->pool_mu);
    for (auto &cs : h->calls) {
        std::lock_guard<std::mutex> in_flight(cs->mu);
        cudaStreamSynchronize(cs->stream);
    }
}
int32_t translate_exception(icp_ctx ctx);  // call inside catch (...)
void set_error(icp_ctx ctx, const std::string &msg);
}  // namespace icp
