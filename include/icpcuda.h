/*
 * icpcuda.h - C ABI of libicpcuda.so, the B200-native (sm_100a) hot path of
 * unibas-gravis/icp-proposal: closest-point ICP proposal + likelihood evaluators inside the
 * Metropolis-Hastings registration loop.
 *
 * This is the drop-in boundary: the entry points below are what a Scala/Panama (or JNI) binding of
 * the reference's L2 classes would bind. Each group cites the reference interface it replaces;
 * paths are relative to src/main/scala of the reference. INTEGRATION.md shows the Scala side.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, opaque handles, no exceptions, no callbacks.
 *  - every function returns int32_t: 0 = ICP_OK, negative = error (icp_last_error gives the text).
 *  - -inf / NaN in outputs are VALUES, not errors (logTransitionProbability legitimately returns
 *    -inf, NonRigidIcpProposal.scala:73).
 *  - all floating-point data is FP64, row-major. Host buffers unless the name ends in _device.
 *    The library copies what it keeps; caller buffers are only read/written during the call.
 *  - theta (ModelFittingParameters.allParameters, ModelFittingParameters.scala:64):
 *        [ s | tx ty tz | phi theta psi | cx cy cz | alpha_0 .. alpha_{K-1} ]     length K + 10
 *  - "C" is the number of chains (parameter vectors) in a batched call.
 *  - There is no CPU fallback: every compute entry point runs CUDA kernels on the context's device
 *    and fails with ICP_ERR_CUDA when that is impossible.
 *  - Handles are safe to use from several host threads. The per-call entries of a proposal or evaluator (icp_propose,
 *    icp_log_transition, icp_posterior, icp_eval_log_value) run concurrently, also on ONE shared handle - the reference shares its
 *    proposal mixture and evaluator between ten fitting threads (apps/femur/RunMHRandomInitComparison.scala:59-86): every call
 *    leases a call slot of the handle (own stream and scratch, at most 16 in flight), the posterior cache of a proposal is shared.
 *    Handles whose pipeline refits scratch of the model (evaluators that measure target -> model distances) and every other entry
 *    point serialise on the context.
 */
#ifndef ICPCUDA_H
#define ICPCUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICP_OK 0
#define ICP_ERR_INVALID_ARGUMENT (-1)
#define ICP_ERR_CUDA (-2)
#define ICP_ERR_OUT_OF_MEMORY (-3)
#define ICP_ERR_EMPTY_SET (-4)   /* CollectiveAverage...Evaluator.scala:51,63 `filteredDists.max` on an empty list */
#define ICP_ERR_NOT_POSITIVE_DEFINITE (-5)
#define ICP_ERR_NAN (-6)         /* a NaN transition probability (Scalismo's MixtureProposal throws) or a NaN initial log-value */

typedef struct icp_ctx_s *icp_ctx;
typedef struct icp_model_s *icp_model;
typedef struct icp_target_s *icp_target;
typedef struct icp_proposal_s *icp_proposal;
typedef struct icp_evaluator_s *icp_evaluator;
typedef struct icp_chain_s *icp_chain;
typedef struct icp_comm_s *icp_comm;
typedef struct icp_jsonlog_s *icp_jsonlog;

/* ---- (1) context --------------------------------------------------------------------------- */
int32_t icp_ctx_create(int32_t device, icp_ctx *out);
int32_t icp_ctx_destroy(icp_ctx ctx);
/* copies the last error text of this context (or of the calling thread when ctx == NULL) */
int32_t icp_last_error(icp_ctx ctx, char *buf, size_t n);
/* library / device identification for logs: "icpcuda 0.1 sm_100a <device name>" */
int32_t icp_version(icp_ctx ctx, char *buf, size_t n);

/* ---- (2) model: StatisticalMeshModel (read at apps/femur/LoadTestData.scala:34-35) ---------- */
/* ref_xyz N x 3, mean_def 3N (NULL = zero mean deformation), basis 3N x K unscaled U,
 * variance K, tris T x 3. Q = U diag(sqrt(variance)) is formed on the device. 1 <= K <= 224 (the reference ships
 * ranks 51, 101 and 201); larger ranks are ICP_ERR_INVALID_ARGUMENT. */
int32_t icp_model_create(icp_ctx ctx, int32_t N, int32_t T, int32_t K, const double *ref_xyz,
                         const double *mean_def, const double *basis, const double *variance,
                         const int32_t *tris, icp_model *out);
int32_t icp_model_destroy(icp_model m);
int32_t icp_model_rank(icp_model m, int32_t *K);

/* ---- (3) target: TriangleMesh3D + its lazily built query structures ------------------------- */
/* builds on the device: triangle BVH (operations.closestPointOnSurface), vertex BVH
 * (pointSet.findClosestPoint), boundary table (operations.pointIsOnBoundary) */
int32_t icp_target_create(icp_ctx ctx, int32_t Nt, int32_t Tt, const double *xyz, const int32_t *tris,
                          icp_target *out);
int32_t icp_target_destroy(icp_target t);

/* ---- (4) primitives ------------------------------------------------------------------------- */
/* target.operations.closestPointOnSurface(q).point (NonRigidIcpProposal.scala:97,
 * IndependentPointDistanceEvaluator.scala:43, CollectiveAverage...:45, IcpBasedSurfaceFitting.scala:73,
 * RegistrationComparison.scala:35). tri: closest triangle (ties: lowest index), feature: 0 vertex,
 * 1 edge, 2 face interior, cp nq x 3, d2 squared distance. Any output may be NULL. */
int32_t icp_closest_point_surface(icp_target t, int64_t nq, const double *q, int32_t *tri,
                                  int32_t *feature, double *cp, double *d2);
/* same with q / outputs in device memory (bench "value": inputs resident in HBM) */
int32_t icp_closest_point_surface_device(icp_target t, int64_t nq, const double *q_dev, int32_t *tri_dev,
                                         double *cp_dev, double *d2_dev);
/* target.pointSet.findClosestPoint(q).id (NonRigidIcpProposal.scala:98, CollectiveAverage...:46) */
int32_t icp_closest_vertex(icp_target t, int64_t nq, const double *q, int32_t *id, double *d2);
/* target.operations.pointIsOnBoundary for every vertex (NonRigidIcpProposal.scala:99) */
int32_t icp_target_boundary_flags(icp_target t, uint8_t *flags /* Nt */);
/* ModelFittingParameters.transformedMesh (ModelFittingParameters.scala:108-110): xyz C x N x 3 */
int32_t icp_reconstruct(icp_model m, int32_t C, const double *theta, double *xyz);
/* transformedMesh(theta).vertexNormals (NonRigidIcpProposal.scala:100,120): normals C x N x 3 */
int32_t icp_vertex_normals(icp_model m, int32_t C, const double *theta, double *normals);
/* modelSample.operations.closestPointOnSurface (IndependentPointDistanceEvaluator.scala:51,
 * CollectiveAverage...:57, MeshMetrics.hausdorffDistance): the same nq query points against each
 * of the C transformed model meshes. Outputs C x nq (x 3). */
int32_t icp_model_closest_point_surface(icp_model m, int32_t C, const double *theta, int64_t nq,
                                        const double *q, int32_t *tri, int32_t *feature, double *cp,
                                        double *d2);
/* currentMesh.pointSet.findClosestPoint (NonRigidIcpProposal.scala:118): ids C x nq */
int32_t icp_model_closest_vertex(icp_model m, int32_t C, const double *theta, int64_t nq, const double *q,
                                 int32_t *id, double *d2);
/* model.referenceMesh boundary table (currentMesh.operations.pointIsOnBoundary, :119) */
int32_t icp_model_boundary_flags(icp_model m, uint8_t *flags /* N */);

/* ---- (5) NonRigidIcpProposal (api/sampling/proposals/NonRigidIcpProposal.scala:30-153) ------ */
#define ICP_MODEL_SAMPLING 0    /* api/other/IcpProjectionDirection.scala */
#define ICP_TARGET_SAMPLING 1

/* Covariance factor W (W W^T = M^-1) that maps the caller's standard normals z to a posterior sample (:55):
 *   ICP_FACTOR_CHOLESKY  W = L^-T, M = L L^T: one back substitution per proposal (default of the fused runner; the
 *                        same proposal DISTRIBUTION as the reference, different values for the same z)
 *   ICP_FACTOR_SVD       W = D^-1 Ubar diag(sqrt(lambda')), Ubar diag(lambda') Ubar^T = D M^-1 D, lambda' descending,
 *                        largest-magnitude entry of every vector positive: the factor Scalismo's posterior GP samples
 *                        with (SURVEY Appendix A4/A6), i.e. the reference's VALUE for the caller's z. Costs one K x K
 *                        eigen-decomposition per posterior (batched one-sided Jacobi on the device); needs variance > 0. */
#define ICP_FACTOR_CHOLESKY 0
#define ICP_FACTOR_SVD 1
/* Arithmetic of the posterior's rank update M = I + sum Q_i^T Sigma_i^-1 Q_i (:152), the dominant kernel of an MH step:
 *   ICP_RANK_UPDATE_FP64  FP64 tensor pipe (mma.sync m8n8k4 f64): M to ~1e-15, posterior mean to ~1e-12 (default)
 *   ICP_RANK_UPDATE_INT8  5th-generation tensor cores (tcgen05.mma kind::i8, INT32 accumulators in TMEM) through a
 *                         split-integer (Ozaki) emulation of the FP64 product with four base-255 digits: M to 2e-9,
 *                         posterior mean to ~1e-8 relative - inside the 1e-5 contract of BASELINE.json, several times
 *                         faster. Ranks up to 112; other shapes fall back to FP64.
 * The environment variable ICPCUDA_RANK_UPDATE=int8|fp64 overrides the field for every proposal of the process. */
#define ICP_RANK_UPDATE_FP64 0
#define ICP_RANK_UPDATE_INT8 1

typedef struct {
    double step_length;         /* stepLength */
    double tangential_noise;    /* tangentialNoise: std-dev in the tangent plane */
    double noise_along_normal;  /* noiseAlongNormal: std-dev along the vertex normal */
    int32_t direction;          /* ICP_MODEL_SAMPLING | ICP_TARGET_SAMPLING */
    int32_t boundary_aware;     /* boundaryAware */
    int32_t factor;             /* ICP_FACTOR_CHOLESKY | ICP_FACTOR_SVD */
    int32_t rank_update;        /* ICP_RANK_UPDATE_FP64 | ICP_RANK_UPDATE_INT8 */
} icp_proposal_params;

/* model_point_ids: decimatedModel.referenceMesh.pointSet.pointIds (:94; they index the FULL mesh,
 * SURVEY Appendix B1). target_points: decimatedTarget.pointSet.points (:117). The host passes the
 * lists it got from Scalismo's (VTK) decimation, so parity does not depend on VTK. */
int32_t icp_proposal_create(icp_model m, icp_target t, const icp_proposal_params *params,
                            const int32_t *model_point_ids, int32_t n_ids, const double *target_points,
                            int32_t n_tp, icp_proposal *out);
int32_t icp_proposal_destroy(icp_proposal p);

/* icpPosterior (:88-153): posterior of the GP given the closest-point correspondences of theta.
 * mu C x K posterior mean coefficients; M C x K x K (= I + sum Q_i^T Sigma_i^-1 Q_i, the inverse
 * coefficient-space covariance; NULL to skip); n_obs C (observations that survived the boundary
 * filter; NULL to skip). */
int32_t icp_posterior(icp_proposal p, int32_t C, const double *theta, double *mu, double *M, int32_t *n_obs);
/* propose (:53-68). z: C x K standard normals drawn by the caller's RNG (posterior.sample(), :55).
 * theta_out C x (K+10). alpha' = alpha + step (S (mu + W z) - alpha), W W^T = M^-1 (W as selected by params.factor). */
int32_t icp_propose(icp_proposal p, int32_t C, const double *theta, const double *z, double *theta_out);
/* logTransitionProbability(from, to) (:71-85): out C. -inf unless only alpha changed (:72-74). */
int32_t icp_log_transition(icp_proposal p, int32_t C, const double *from, const double *to, double *out);
/* drops the per-handle posterior cache (the reference's Memoize(icpPosterior, 20), :49) */
int32_t icp_proposal_clear_cache(icp_proposal p);

/* RandomShapeUpdateProposal.logTransitionProbability (proposals/RandomShapeUpdateProposal.scala:38-45)
 * and GaussianAxis{Rotation,Translation}Proposal (proposals/PoseProposals.scala:47-62,81-89) are
 * O(K) host arithmetic in the reference; they exist on the device inside icp_chain_run only. */

/* model.posterior(corr, sigma2).mean + model.coefficients + step of the deterministic ICP
 * (api/other/IcpBasedSurfaceFitting.scala:55-92), identity pose (what IcpRegistration.scala:40-43 passes): alpha C x K -> alpha_out C x K.
 * direction per call (the reference flips an unseeded coin, :67, so the caller supplies it). */
int32_t icp_std_icp_iteration(icp_model m, icp_target t, int32_t direction, const int32_t *model_point_ids,
                              int32_t n_ids, const double *target_points, int32_t n_tp, double sigma2,
                              double step_length, int32_t C, const double *alpha, double *alpha_out);

/* the same iteration under a rigid transform (currentTrans, :61 `model.transform(currentTrans).instance(params)`): theta
 * C x (K+10) carries the transform and the coefficients. As in the reference the correspondences are found on the
 * transformed instance while the posterior (:81) is that of the untransformed model on the target points as they are. */
int32_t icp_std_icp_iteration_theta(icp_model m, icp_target t, int32_t direction, const int32_t *model_point_ids,
                                    int32_t n_ids, const double *target_points, int32_t n_tp, double sigma2,
                                    double step_length, int32_t C, const double *theta, double *alpha_out);

/* ---- (5b) IcpBasedSurfaceFitting.runfitting on the device (api/other/IcpBasedSurfaceFitting.scala:46-126) ----------- */
/* The whole deterministic-ICP loop for C independent fits: every sigma2 of iterationSeq runs num_iterations + 1 iterations
 * (:55-109), each one the icp_std_icp_iteration_theta of its fit, with the rigid transform of theta0 (currentTrans, :61) fixed
 * and only the coefficients moving. Iterations are replayed CUDA graphs; a run synchronises once. */
#define ICP_MODEL_AND_TARGET_SAMPLING 2   /* IcpProjectionDirection.scala: a coin per iteration (:67); icp_std_icp only */
typedef struct icp_std_icp_s *icp_std_icp;
/* model_point_ids / target_points as for icp_std_icp_iteration (uploaded once; n_ids, n_tp >= 1). direction: the direction
 * of every iteration unless a run supplies its own: ICP_MODEL_SAMPLING, ICP_TARGET_SAMPLING or ICP_MODEL_AND_TARGET_SAMPLING
 * (a Philox coin, see icp_std_icp_io). The handle holds references on the model and the target. */
int32_t icp_std_icp_create(icp_model m, icp_target t, const int32_t *model_point_ids, int32_t n_ids, const double *target_points,
                           int32_t n_tp, double step_length, int32_t direction, int32_t max_fits, icp_std_icp *out);
int32_t icp_std_icp_destroy(icp_std_icp h);
/* per-fit status words (icp_std_icp_io.status): where the reference catches an exception and returns the last coefficients
 * (:94-104), that fit stops: it keeps its coefficients for the rest of the run, its later log rows repeat them and
 * iterations_done stops counting. The other fits are unaffected and the run returns ICP_OK. */
#define ICP_STD_ICP_NON_FINITE 1             /* theta0 or the new coefficients were not finite */
#define ICP_STD_ICP_NOT_POSITIVE_DEFINITE 2  /* the posterior's factorisation failed */
typedef struct {
    /* directions == NULL with ICP_MODEL_AND_TARGET_SAMPLING: fit c flips a coin in iteration i with Philox4x32-10 keyed by seed,
     * counter (fit_id_offset + c, i, block 0) as in icp_chain_io: u = 53-bit uniform of words x (high) and y (low), model
     * sampling when u < 0.5. Results do not depend on how fits are batched or sharded over GPUs. */
    uint64_t seed;
    uint64_t fit_id_offset;
    const int32_t *directions;  /* [iters][C] ICP_MODEL_SAMPLING | ICP_TARGET_SAMPLING, or NULL; iters = n_sigma (num_iterations + 1) */
    /* outputs, any may be NULL */
    double *alpha_final;        /* [C][K] */
    double *log_alpha;          /* [iters][C][K] coefficients after every iteration */
    int32_t *log_direction;     /* [iters][C] */
    int32_t *status;            /* [C] OR of ICP_STD_ICP_* */
    int32_t *iterations_done;   /* [C] iterations completed before the fit stopped (iters when it never did) */
} icp_std_icp_io;
/* theta0 C x (K+10), sigma2 n_sigma values > 0 (iterationSeq), 1 <= C <= max_fits. Host buffers. */
int32_t icp_std_icp_run(icp_std_icp h, int32_t C, const double *theta0, int32_t n_sigma, const double *sigma2,
                        int32_t num_iterations, const icp_std_icp_io *io);
/* the same with theta0_dev and every io pointer in DEVICE memory (sigma2 stays a host array). Caller directions are read
 * back to the host before the run is enqueued (the split of every iteration is planned there); the run is synchronised before
 * returning unless async != 0. */
int32_t icp_std_icp_run_device(icp_std_icp h, int32_t C, const double *theta0_dev, int32_t n_sigma, const double *sigma2,
                               int32_t num_iterations, const icp_std_icp_io *io_dev, int32_t async);
/* device time in milliseconds of the last run (CUDA events on the library stream) and the kernels + memsets it launched */
int32_t icp_std_icp_last_run_stats(icp_std_icp h, double *device_ms, int64_t *launches);

/* ---- (6) evaluators (api/sampling/evaluators/<Name>.scala, ProductEvaluators.scala) -------------- */
#define ICP_EVAL_ACCEPT_ALL 0     /* AcceptAllEvaluator.scala:22-28 */
#define ICP_EVAL_INDEPENDENT 1    /* IndependentPointDistanceEvaluator.scala:27-67, Gaussian(p0 = mean, p1 = sd) */
#define ICP_EVAL_HAUSDORFF 2      /* HausdorffDistanceEvaluator.scala:25-36, Exponential(p0 = rate) */
#define ICP_EVAL_COLLECTIVE 3     /* CollectiveAverageHausdorffDistanceBoundaryAwareEvaluator.scala:27-79,
                                     Gaussian(p0 = mean, p1 = sd) on the average + Exponential(p2) on the max */
#define ICP_MODEL_TO_TARGET 0     /* EvaluationModeType.scala */
#define ICP_TARGET_TO_MODEL 1
#define ICP_SYMMETRIC 2

typedef struct {
    int32_t kind;       /* ICP_EVAL_* */
    int32_t mode;       /* ICP_MODEL_TO_TARGET | ICP_TARGET_TO_MODEL | ICP_SYMMETRIC */
    int32_t use_prior;  /* 1: ProductEvaluator(ModelPriorEvaluator, distance) (ProductEvaluators.scala:44-47) */
    int32_t reserved;
    double p0, p1, p2;
} icp_evaluator_params;

/* model_point_ids = randomPointIdsOnModel, target_points = randomPointsOnTarget
 * (IndependentPointDistanceEvaluator.scala:37-38); ignored by the Hausdorff evaluator, which uses
 * every vertex of both meshes (MeshMetrics.hausdorffDistance). */
int32_t icp_evaluator_create(icp_model m, icp_target t, const icp_evaluator_params *params,
                             const int32_t *model_point_ids, int32_t n_ids, const double *target_points,
                             int32_t n_tp, icp_evaluator *out);
int32_t icp_evaluator_destroy(icp_evaluator e);
/* computeLogValue / logValue for C parameter vectors. values: C x 3 = {product, prior, distance}
 * (the keys of the evaluator map, ProductEvaluators.scala:49-53; prior = 0 when use_prior == 0).
 * status: C (NULL to skip), ICP_OK or ICP_ERR_EMPTY_SET per chain (value is NaN then). */
int32_t icp_eval_log_value(icp_evaluator e, int32_t C, const double *theta, double *values, int32_t *status);
/* ModelPriorEvaluator.logValue (ModelPriorEvaluator.scala:28-30): out C */
int32_t icp_eval_prior(icp_model m, int32_t C, const double *theta, double *out);
/* RegistrationComparison.evaluateReconstruction2GroundTruth[BoundaryAware]
 * (api/other/RegistrationComparison.scala:24-49): per chain {avg, hausdorff, avg_boundary_aware,
 * max_boundary_aware} between transformedMesh(theta) and the target; out C x 4. */
int32_t icp_registration_metrics(icp_model m, icp_target t, int32_t C, const double *theta, double *out);
/* MeshMetrics.diceCoefficient(transformedMesh(theta), target) (apps/femur/StdIcpVsChainICPrandomInitComparisonAll.scala:46):
 * Monte-Carlo overlap 2 |A and B| / (|A| + |B|) over n_samples points drawn uniformly in the union of the two bounding
 * boxes; a point is inside a mesh when vertexNormal(v) . (v - p) > 0 for the mesh vertex v nearest to p (Scalismo
 * toBinaryImage). The reference draws 10 000 points from an unseeded RNG; here the caller supplies them as unit-cube
 * samples (unit_samples, n_samples x 3 in [0, 1], scaled into each chain's evaluation region) or passes NULL for
 * device-generated Philox samples keyed by `seed` (the same set for every chain). out: C. */
int32_t icp_dice_coefficient(icp_model m, icp_target t, int32_t C, const double *theta, int32_t n_samples,
                             const double *unit_samples, uint64_t seed, double *out);
/* PosteriorVariability.computeDistanceMapFromMeshesTotal / ...Normal (apps/util/PosteriorVariability.scala:30-73)
 * over the shapes LogHelper.logSamples2shapes reconstructs from S logged parameter vectors
 * (apps/util/LogHelper.scala:39-41): per model vertex the sample mean (mean: N x 3), the sample covariance with
 * divisor S - 1 (cov: N x 9 row-major), its trace (total_variance: N, the "Total" colour map) and the variance of
 * the samples along a direction n (normal_variance: N, the "Normal" map). sum_normals != 0: n = mean over the
 * samples of their unit vertex normals, not re-normalised (:59-60); sum_normals == 0: n = vertex normal of `ref`
 * = transformedMesh(theta_ref), or of the model's reference mesh when theta_ref is NULL (:62-63). Any output pointer
 * may be NULL. S == 1 yields NaN variances like the reference (0 * 1/0). */
int32_t icp_posterior_variability(icp_model m, int32_t S, const double *theta, int32_t sum_normals,
                                  const double *theta_ref, double *mean, double *cov, double *total_variance,
                                  double *normal_variance);

/* ---- (7) fused Metropolis-Hastings runner ---------------------------------------------------- */
/* Scalismo MetropolisHastings.next + MixtureProposal, driven from
 * api/sampling/SamplingRegistration.scala:52-85, as a device-resident loop over n_steps for C
 * independent chains. */
#define ICP_PROP_ICP 0
#define ICP_PROP_RANDOM_SHAPE 1     /* RandomShapeUpdateProposal(sd) */
#define ICP_PROP_ROTATION 2         /* GaussianAxisRotationProposal(sd, axis 0 roll/phi, 1 pitch/theta, 2 yaw/psi) */
#define ICP_PROP_TRANSLATION 3      /* GaussianAxisTranslationProposal(sd, axis) */

typedef struct {
    int32_t kind;            /* ICP_PROP_* */
    int32_t axis;            /* pose proposals */
    double weight;           /* effective (flattened) mixture weight; normalised by the library */
    double sd;               /* random-walk / pose std-dev */
    icp_proposal proposal;   /* kind == ICP_PROP_ICP */
} icp_component;

int32_t icp_chain_create(icp_model m, icp_target t, const icp_component *components, int32_t n_components,
                         icp_evaluator evaluator, int32_t max_chains, icp_chain *out);
int32_t icp_chain_destroy(icp_chain c);

/* Several targets in one chain handle: every chain names its own target, and the chains of all targets run in the same
 * batched launches (icp_chain_create is the one-target case). Entry g holds a target, the mixture built for it and its
 * evaluator. Only the targets may differ: every entry has the same component kinds, weights, sd and axes; the ICP
 * proposals share the model, every icp_proposal_params field, the model point ids and n_tp; the evaluators share kind,
 * mode, use_prior, p0 - p2, the model point ids and n_tp (not the Hausdorff evaluator, whose list is all vertices of its
 * target: shorter lists are padded with repeats of their last vertex, which does not change the maximum). Any other
 * difference is refused with ICP_ERR_INVALID_ARGUMENT and a message naming the field. The handle holds references on
 * every target, proposal and evaluator.
 * Boundary policy: the boundary path (no closest-point sharing with the evaluator, no constant-Gram posterior) is taken
 * for every chain when any target has a boundary, so a chain on a closed target of such a set agrees with its
 * single-target run to rounding, not bit for bit. Runs with metrics_interval > 0 are refused when n_targets > 1
 * (icp_registration_metrics on each target's rows of theta_best afterwards gives the same measures). */
typedef struct {
    icp_target target;
    const icp_component *components;  /* n_components entries */
    icp_evaluator evaluator;          /* built for (model, target) */
} icp_chain_target;
int32_t icp_chain_create_targets(icp_model m, int32_t n_targets, const icp_chain_target *targets, int32_t n_components,
                                 int32_t max_chains, icp_chain *out);
/* target_index [C] (host): chain c runs on targets[target_index[c]]. Takes effect at the next run from theta0; resumed runs
 * keep the assignment. Required before the first run of a handle with n_targets > 1 (and again whenever a run from theta0
 * has a different C). Sharded runs pass the indices of their own chains. */
int32_t icp_chain_set_target_index(icp_chain c, int32_t C, const int32_t *target_index);

typedef struct {
    /* randomness: either counter-based on the device (Philox4x32-10 keyed by seed and the global
     * chain id chain_id_offset + c, so results do not depend on how chains are sharded over GPUs)
     * or supplied by the caller's RNG (all three non-NULL): u_comp [n_steps][C] picks the mixture
     * component, z [n_steps][C][K] are the proposal's standard normals, u_acc [n_steps][C] is the
     * acceptance uniform. */
    uint64_t seed;
    uint64_t chain_id_offset;
    const double *u_comp;
    const double *z;
    const double *u_acc;
    /* chain log, one record per step and chain in the layout of jsonLogFormat
     * (api/sampling/loggers/JSONAcceptRejectLogger.scala:35,93-106); any pointer may be NULL.
     * log_values: {product, prior, distance} of the state that is current after the step. */
    int32_t *log_component;   /* [n_steps][C]   proposal index (-> generatedBy name) */
    uint8_t *log_accepted;    /* [n_steps][C]   status */
    double *log_values;       /* [n_steps][C][3] */
    double *log_theta;        /* [n_steps][C][K+10] parameters of the current state after the step */
    double *theta_final;      /* [C][K+10] */
    int64_t *n_accepted;      /* [C] */
    /* [C] per-chain status words, OR of the ICP_CHAIN_* bits below, sticky over the run (and over resumed runs). Where the
     * reference would throw, the batched runner rejects that step, lets every chain finish, writes all outputs and then
     * returns ICP_ERR_EMPTY_SET / ICP_ERR_NOT_POSITIVE_DEFINITE / ICP_ERR_NAN for the first flagged chain. */
    int32_t *status;
    /* BestSampleLogger(evaluator) (api/sampling/SamplingRegistration.scala:58,87): the state with the largest product
     * log-value among theta0 and the states current after every step. */
    double *theta_best;       /* [C][K+10] */
    double *value_best;       /* [C] */
    /* RegistrationComparison.evaluateReconstruction2GroundTruthBoundaryAware of the best sample so far, every
     * metrics_interval steps (SamplingRegistration.scala:75-82, acceptInfoPrintInterval; 0 = off): row r - 1 is taken after
     * step r * metrics_interval of this call; layout of icp_registration_metrics. */
    int32_t metrics_interval;
    int32_t reserved;
    double *log_metrics;      /* [n_steps / metrics_interval][C][4] */
} icp_chain_io;
#define ICP_CHAIN_EMPTY_SET 1        /* CollectiveAverage...Evaluator.scala:51,63: filtered distance list empty */
#define ICP_CHAIN_NOT_POSITIVE_DEFINITE 2
#define ICP_CHAIN_NAN_TRANSITION 4   /* a mixture component's transition density was NaN */
#define ICP_CHAIN_NAN_VALUE 8        /* the evaluator returned NaN for theta0 */

/* theta0 C x (K+10) (host). io buffers are host memory. When the log buffers are page-locked (cudaHostAlloc /
 * cudaHostRegister), finished log rows are copied out on a second stream while later steps run; pageable buffers are
 * copied after the last step. */
int32_t icp_chain_run(icp_chain c, int32_t C, int32_t n_steps, const double *theta0, const icp_chain_io *io);
/* same with theta0 and every non-NULL io pointer in DEVICE memory; the run is enqueued on the
 * context stream and synchronised before returning unless `async` != 0.
 * theta0_dev == NULL resumes the C chains of the previous run from their resident state (current
 * parameters, log-values and posteriors stay on the device; the step counter - hence the Philox
 * stream - continues, the log pointers of this call start at record 0). */
int32_t icp_chain_run_device(icp_chain c, int32_t C, int32_t n_steps, const double *theta0_dev,
                             const icp_chain_io *io_dev, int32_t async);
int32_t icp_ctx_synchronize(icp_ctx ctx);
/* device time in milliseconds of the last icp_chain_run* on this chain (CUDA events on the
 * library stream) and the number of kernels it launched */
int32_t icp_chain_last_run_stats(icp_chain c, double *device_ms, int64_t *kernel_launches);
/* Rejection look-ahead of the fused runner ("prefetching" Metropolis-Hastings). The loop of
 * api/sampling/SamplingRegistration.scala:60-85 is sequential, and with few chains every step is a chain of dependent kernel
 * latencies. A rejected step leaves the state where it was and the randomness of step s depends on (seed, chain, s) only, so
 * `width` lanes per chain evaluate the proposals of steps s .. s + width - 1 from the same current state in ONE batched
 * round; the lanes before the first accepting one are the chain's rejected steps, that lane is its next accepted step, the
 * rest is discarded. The chain log is bit-identical to the step-by-step runner's (also with caller-supplied u_comp / z /
 * u_acc); a round costs the latency of one step and takes (1 - (1 - a)^width) / a steps at acceptance rate a.
 * width: -1 automatic (the default; ICPCUDA_LOOKAHEAD overrides it): up to 8 lanes for up to 8 chains, 4 up to 32, 2 up to 148, none
 * beyond, and the number of lanes that are ACTIVE in a round adapts while the run goes - every active width is timed once, then
 * each batch of rounds takes the width with the most expected steps per millisecond at the measured acceptance rate, so a chain
 * that accepts everything, or lanes that already fill the GPU, run at one lane; 0 or 1 off; 2 .. 32 exactly that many lanes. Not used by runs with metrics_interval > 0, asynchronous icp_chain_run_device calls or
 * icp_chain_profile. rounds (nullable): batched rounds of the last run (= its steps when the look-ahead was off). */
int32_t icp_chain_set_lookahead(icp_chain c, int32_t width);
int32_t icp_chain_last_run_rounds(icp_chain c, int64_t *rounds);

/* Posterior variability maps accumulated inside the run: icp_posterior_variability over the states LogHelper.samplesFromLog
 * (apps/util/LogHelper.scala:25-42) would select from the chain log, without a chain log, per chain or pooled.
 * Record i of a chain is its i-th step since theta0 (resumed runs keep counting); it is selected when
 * burn_in <= i < end (end <= 0: no limit) and (i - burn_in) % take_every_n == 0, and its sample is the state current after
 * that step (row i of log_theta). Unlike LogHelper, which fails there, a selected record before the chain's first acceptance
 * counts theta0. Each chain keeps FP64 accumulators on the device: a count and per vertex the mean, the centred second
 * moment and (normals = 1) the sum of unit vertex normals - 12 N doubles per chain. They are updated when a chain accepts,
 * once per accepted state with the number of selected records at which that state was current, so the step-by-step
 * runner, the rejection look-ahead at any width and runs split by resume produce bit-identical maps. */
typedef struct {
    int64_t burn_in;        /* LogHelper burnIn, >= 0 */
    int64_t take_every_n;   /* LogHelper takeEveryN, >= 1 */
    int64_t end;            /* LogHelper total: records below it; <= 0 = no limit */
    int32_t normals;        /* 1: also accumulate unit vertex normals (needed to read with sum_normals != 0) */
    int32_t reserved;
} icp_chain_stats_params;
/* NULL = off. Takes effect at the next run from theta0, which zeroes the accumulators; resumed runs keep accumulating. */
int32_t icp_chain_set_statistics(icp_chain c, const icp_chain_stats_params *p);
/* chain in [0, C) of the resident run, or -1 = pooled over all its chains (Chan's merge in chain order, on the device).
 * Outputs (host memory) in the layout of icp_posterior_variability; any may be NULL; the direction of normal_variance is
 * chosen here (sum_normals, theta_ref as there). n_samples: S. Reading leaves the accumulators unchanged. Error if
 * statistics were off for the resident run, or if S == 0; S == 1 yields NaN variances. */
int32_t icp_chain_statistics(icp_chain c, int32_t chain, int32_t sum_normals, const double *theta_ref,
                             int64_t *n_samples, double *mean, double *cov, double *total_variance, double *normal_variance);

/* ---- (7b) chain log in the reference's JSON wire format (host functions: no CUDA context needed) ---------------------- */
/* JSONAcceptRejectLogger (api/sampling/loggers/JSONAcceptRejectLogger.scala:35,93-127) as a streaming writer and a loader.
 * The reference rewrites the whole file on every writeLog (:112-122), quadratic over a run; icp_jsonlog_append appends the
 * new records and leaves a valid JSON array after every call. component_names[i] is the generatedBy name of mixture
 * component i (the log's "name"), value_keys[3] the logvalue keys of icp_chain_io.log_values ("product", "prior" and the
 * distance evaluator's key, ProductEvaluators.scala:49-53; an empty string omits that entry). */
int32_t icp_jsonlog_open(const char *path, int32_t K, const char *const *component_names, int32_t n_components,
                         const char *const *value_keys, icp_jsonlog *out);
/* appends chain `chain` of a run's HOST log arrays ([n_steps][C] records as icp_chain_run returned them): accepted records
 * carry rigid[9] and coeff[K], rejected ones the current state's log-values with empty arrays (:101-105); NaN / infinite
 * values are written as null like spray-json does */
int32_t icp_jsonlog_append(icp_jsonlog log, int32_t n_steps, int32_t C, int32_t chain, const int32_t *log_component,
                           const uint8_t *log_accepted, const double *log_values, const double *log_theta);
int32_t icp_jsonlog_close(icp_jsonlog log);
/* loadLog (:124-127), also for files the reference wrote. capacity == 0: only *n_records is set. Otherwise arrays of
 * `capacity` records (any may be NULL): index, status, values [n][3] in the order of value_keys (3 x 64 bytes out:
 * "product", "prior", the third key found), theta [n][K+10] = sampleToModelParameters (:139-146; scale 1; NaN for rejected
 * records, whose arrays are empty), names [n][64]. */
int32_t icp_jsonlog_load(const char *path, int32_t K, int64_t capacity, int64_t *n_records, int64_t *index, uint8_t *status,
                         double *values, double *theta, char *names, char *value_keys);
/* LogHelper.samplesFromLog (apps/util/LogHelper.scala:27-37) and the loop of ReplayFittingFromLog.scala:53-66: log indices
 * burn_in, burn_in + take_every_n, ... below min(n_records, total), each replaced by the closest accepted record at or
 * before it. indices == NULL: only *n_out. Feed theta[indices] to icp_reconstruct / icp_posterior_variability. */
int32_t icp_chainlog_sample_indices(int64_t n_records, const uint8_t *status, int32_t take_every_n, int64_t total,
                                    int64_t burn_in, int64_t capacity, int64_t *n_out, int64_t *indices);

/* ---- (8) multi-GPU: one process per GPU, NCCL over NVLink (SURVEY 8e) ---------------------------------------------- */
/* Chains / random-init restarts / targets are independent (apps/femur/RunMHRandomInitComparison.scala:66-86,
 * StdIcpVsChainICPrandomInitComparisonAll.scala:107-122): rank r runs its own chains with
 * icp_chain_io.chain_id_offset = first global chain id, model and target replicated, and there is no collective on the
 * per-sample path. These entry points are the end-of-run exchange: the gather of the chain logs and the reduction of the
 * posterior statistics. The library opens libnccl.so.2 (or $ICPCUDA_NCCL_LIB) on first use; hosts that never call them
 * need no NCCL. Rank 0 obtains the 128-byte id and hands it to the other ranks through the host's own channel (the
 * Scala driver's RPC / a file / an environment variable); icp_comm_init is collective over all `world` ranks. */
#define ICP_COMM_UNIQUE_ID_BYTES 128
int32_t icp_comm_unique_id(icp_ctx ctx, uint8_t id[ICP_COMM_UNIQUE_ID_BYTES]);
int32_t icp_comm_init(icp_ctx ctx, int32_t rank, int32_t world, const uint8_t id[ICP_COMM_UNIQUE_ID_BYTES], icp_comm *out);
int32_t icp_comm_destroy(icp_comm c);
int32_t icp_comm_info(icp_comm c, int32_t *rank, int32_t *world, int32_t *nccl_version);
/* All-gather of a sharded run's chain logs (the records of JSONAcceptRejectLogger, api/sampling/loggers/
 * JSONAcceptRejectLogger.scala:93-106, as icp_chain_run_device left them in device memory). Every rank passes its own
 * [n_steps][C] arrays in local_dev and receives [world][n_steps][C] arrays (rank-major) in gathered_dev; the pointers
 * used are log_component, log_accepted, log_values, log_theta, theta_final, n_accepted, status, theta_best, value_best -
 * each either non-NULL on both sides or NULL on both. All ranks must pass the same n_steps, C, K and the same set of
 * arrays. device_ms: CUDA-event time of the exchange on this rank; bytes_received: payload that arrived here. */
int32_t icp_chainlog_gather(icp_comm c, int32_t n_steps, int32_t C, int32_t K, const icp_chain_io *local_dev,
                            const icp_chain_io *gathered_dev, double *device_ms, int64_t *bytes_received);
/* icp_posterior_variability over the samples of ALL ranks (apps/util/PosteriorVariability.scala:30-73): every rank passes
 * the S_local (>= 0) logged parameter vectors it holds (host memory); the per-vertex sums are all-reduced (global mean
 * first, then the moments centred on it), and every rank receives the same maps as one call over the union would give
 * (up to summation order). S_total: number of samples over all ranks. */
int32_t icp_variability_allreduce(icp_comm c, icp_model m, int32_t S_local, const double *theta_local, int32_t sum_normals,
                                  const double *theta_ref, double *mean, double *cov, double *total_variance,
                                  double *normal_variance, int64_t *S_total);

/* ---- (9) GPMM construction from analytic kernels (the step before the hot path) -------------------- */
/* One term of the matrix-valued kernel of apps/femur/CreateGPModel.scala:68-83:
 *   k(x, y) = sum_t scale_t * exp(-|x - y|^2 / sigma_t^2) * A_t
 * (Scalismo GaussianKernel3D(sigma) * scale; DiagonalKernel3D: A = I; the anisotropic base kernel: A = baseMatrix). */
typedef struct {
    double scale;
    double sigma;
    double A[9]; /* row-major 3 x 3 */
} icp_kernel_term;
/* out (3 nx) x (3 ny) row-major: block (i, j) = k(x_i, y_j). n_terms in [1, 8]. */
int32_t icp_gpmm_kernel_matrix(icp_ctx ctx, int32_t nx, const double *x, int32_t ny, const double *y,
                               const icp_kernel_term *terms, int32_t n_terms, double *out);
/* Leading n_top eigenpairs of a symmetric positive semi-definite n x n matrix A (row-major; the Nystrom kernel matrix)
 * by one-sided Jacobi on the device: w (n_top, descending), V (n x n_top row-major, unit columns, the largest-magnitude
 * entry of every eigenvector positive). */
int32_t icp_gpmm_eigen_psd(icp_ctx ctx, int32_t n, const double *A, int32_t n_top, double *w, double *V);
/* LowRankGaussianProcess.approximateGPNystrom (CreateGPModel.scala:86) after the eigen-decomposition of the m-point
 * kernel matrix (V: 3m x rank row-major eigenvectors, w: the rank leading eigenvalues, all > 0): basis (3N x rank row-major) =
 * k(pts, nys_pts) V diag(sqrt(m) / w), variance (rank, may be NULL) = w / m, i.e. the pcaBasis / pcaVariance of the
 * StatisticalMeshModel over `pts`. rank <= min(224, 3 m). */
int32_t icp_gpmm_nystrom_extend(icp_ctx ctx, int32_t N, const double *pts, int32_t m, const double *nys_pts,
                                const icp_kernel_term *terms, int32_t n_terms, int32_t rank, const double *V,
                                const double *w, double *basis, double *variance);


/* ---- (9b) the face kernel (apps/bfm/FaceKernel.scala) --------------------------------------------------------------- */
/* SpatiallyVaryingMultiscaleKernel (:26-55) under FaceKernel's symmetrisation about the plane x = 0 (:58-100):
 *   k(x, y)      = sum_l scale_l w_l(x) w_l(y) B3(2^level_l x, 2^level_l y) I_3,
 *   B3(a, b)     = prod_d sum_k beta3(a_d - k) beta3(b_d - k)        (Scalismo BSplineKernel[_3D](order = 3, scale = 0))
 *   k_face(x, y) = symmetric_weight (I k(x, y) + diag(-1, 1, 1) k(x, ybar)) + plain_weight k(x, y),  ybar = (-y_x, y_y, y_z)
 * FaceKernel.scala:60-70 uses levels -6..-2 with scales 128, 64, 32, 10, 4 and the weights 0.7 / 0.3. symmetric_weight = 0
 * evaluates the plain multiscale kernel. */
typedef struct {
    int32_t n_levels;          /* 1..8 */
    int32_t level[8];          /* LevelWithScale.level */
    double scale[8];           /* LevelWithScale.scale */
    double symmetric_weight;   /* 0.7 */
    double plain_weight;       /* 0.3 */
} icp_face_kernel;
/* out (3 nx) x (3 ny) row-major. Region weights of the face mask (FaceMask.computeSmoothedRegions, :33-35) per level and
 * point: wx [n_levels][nx], wy [n_levels][ny], wy_mirror [n_levels][ny] = the weights at the mirrored points ybar; any of
 * them NULL = 1 (no mask). */
int32_t icp_gpmm_face_kernel_matrix(icp_ctx ctx, int32_t nx, const double *x, const double *wx, int32_t ny, const double *y,
                                    const double *wy, const double *wy_mirror, const icp_face_kernel *kernel, double *out);
/* icp_gpmm_nystrom_extend for the face kernel (the BFM-sized model of BASELINE config 5): w_pts [n_levels][N],
 * w_nys / w_nys_mirror [n_levels][m] or NULL */
int32_t icp_gpmm_face_nystrom_extend(icp_ctx ctx, int32_t N, const double *pts, const double *w_pts, int32_t m,
                                     const double *nys_pts, const double *w_nys, const double *w_nys_mirror,
                                     const icp_face_kernel *kernel, int32_t rank, const double *V, const double *w, double *basis,
                                     double *variance);

#ifdef __cplusplus
}
#endif
#endif /* ICPCUDA_H */
