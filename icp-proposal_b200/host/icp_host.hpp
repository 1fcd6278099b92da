// icp_host.hpp - C++17 host-side mirror of the reference's operator API for the hot path, header-only, on top of
// the C ABI of libicpcuda.so (include/icpcuda.h). Same class names, constructor arguments and method meaning as the
// Scala classes (paths relative to src/main/scala of the reference):
//
//   ModelFittingParameters                                   api/sampling/ModelFittingParameters.scala:27-66
//   NonRigidIcpProposal                                      api/sampling/proposals/NonRigidIcpProposal.scala:30-153
//   RandomShapeUpdateProposal                                api/sampling/proposals/RandomShapeUpdateProposal.scala:25-46
//   GaussianAxisRotationProposal / ...TranslationProposal    api/sampling/proposals/PoseProposals.scala:31-90
//   IndependentPointDistanceEvaluator, HausdorffDistanceEvaluator,
//   CollectiveAverageHausdorffDistanceBoundaryAwareEvaluator, ModelPriorEvaluator, EvaluationCaching
//                                                            api/sampling/evaluators/*.scala
//   MixtureProposal, ProductEvaluator, MetropolisHastings    Scalismo (SURVEY.md Appendix A8/A9)
//   SamplingRegistration                                     api/sampling/SamplingRegistration.scala:36-93
//   JSONAcceptRejectLogger                                   api/sampling/loggers/JSONAcceptRejectLogger.scala:35-146
//
// The Scala/Panama binding of INTEGRATION.md has the same shape; this file is what can be compiled in this image
// (g++, no JVM). Everything that touches a mesh or a K x K matrix runs on the GPU; there is no CPU fallback.
#pragma once

#include <cmath>
#include <cstdint>
#include <cstring>
#include <ctime>
#include <fstream>
#include <map>
#include <memory>
#include <random>
#include <sstream>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "icpcuda.h"

namespace icp_host {

inline void check(int32_t rc, icp_ctx ctx = nullptr) {
    if (rc == ICP_OK) return;
    char buf[1024];
    icp_last_error(ctx, buf, sizeof buf);
    throw std::runtime_error("libicpcuda error " + std::to_string(rc) + ": " + buf);
}

enum class IcpProjectionDirection { ModelSampling, TargetSampling, ModelAndTargetSampling };
enum class EvaluationMode { ModelToTargetEvaluation = 0, TargetToModelEvaluation = 1, SymmetricEvaluation = 2 };

// theta = [s | t(3) | rot(3) | centre(3) | alpha(K)]; equality by the bytes of allParameters, generatedBy excluded
struct ModelFittingParameters {
    std::vector<double> allParameters;
    std::string generatedBy = "Anonymous";
    int rank() const { return (int)allParameters.size() - 10; }
    const double *shape() const { return allParameters.data() + 10; }
    bool operator==(const ModelFittingParameters &o) const {
        return allParameters.size() == o.allParameters.size() &&
               std::memcmp(allParameters.data(), o.allParameters.data(), allParameters.size() * sizeof(double)) == 0;
    }
    std::string key() const { return std::string((const char *)allParameters.data(), allParameters.size() * sizeof(double)); }
};

class Context {
public:
    explicit Context(int device = 0) { check(icp_ctx_create(device, &h_)); }
    ~Context() { icp_ctx_destroy(h_); }
    Context(const Context &) = delete;
    icp_ctx handle() const { return h_; }
private:
    icp_ctx h_ = nullptr;
};

class StatisticalMeshModel {
public:
    StatisticalMeshModel(Context &ctx, const std::vector<double> &ref, const std::vector<int32_t> &cells,
                         const std::vector<double> &basis, const std::vector<double> &variance)
        : ctx_(ctx), ref_(ref), N_((int)ref.size() / 3), K_((int)variance.size()) {
        check(icp_model_create(ctx.handle(), N_, (int)cells.size() / 3, K_, ref.data(), nullptr, basis.data(), variance.data(),
                               cells.data(), &h_), ctx.handle());
    }
    ~StatisticalMeshModel() { icp_model_destroy(h_); }
    int rank() const { return K_; }
    int numberOfPoints() const { return N_; }
    icp_model handle() const { return h_; }
    icp_ctx ctx() const { return ctx_.handle(); }
    // SamplingRegistration.initialParametersZero (SamplingRegistration.scala:40-43)
    ModelFittingParameters initialParameters() const {
        ModelFittingParameters p;
        p.allParameters.assign(K_ + 10, 0.0);
        p.allParameters[0] = 1.0;
        for (int i = 0; i < N_; i++)
            for (int d = 0; d < 3; d++) p.allParameters[7 + d] += ref_[3 * i + d] / N_;
        return p;
    }
    std::vector<double> transformedMesh(const ModelFittingParameters &theta) const {
        std::vector<double> xyz((size_t)3 * N_);
        check(icp_reconstruct(h_, 1, theta.allParameters.data(), xyz.data()), ctx());
        return xyz;
    }
private:
    Context &ctx_;
    std::vector<double> ref_;
    int N_, K_;
    icp_model h_ = nullptr;
};

class TriangleMesh3D {
public:
    TriangleMesh3D(Context &ctx, const std::vector<double> &verts, const std::vector<int32_t> &cells) : verts_(verts) {
        check(icp_target_create(ctx.handle(), (int)verts.size() / 3, (int)cells.size() / 3, verts.data(), cells.data(), &h_), ctx.handle());
    }
    ~TriangleMesh3D() { icp_target_destroy(h_); }
    icp_target handle() const { return h_; }
    const std::vector<double> &points() const { return verts_; }
private:
    std::vector<double> verts_;
    icp_target h_ = nullptr;
};

// ---- proposals -------------------------------------------------------------------------------------------------
struct ProposalGeneratorWithTransition {
    virtual ~ProposalGeneratorWithTransition() = default;
    virtual ModelFittingParameters propose(const ModelFittingParameters &theta) = 0;
    virtual double logTransitionProbability(const ModelFittingParameters &from, const ModelFittingParameters &to) = 0;
    virtual void flatten(double weight, std::vector<icp_component> &out, std::vector<std::string> &names) = 0;
    double logTransitionRatio(const ModelFittingParameters &from, const ModelFittingParameters &to) {
        return logTransitionProbability(from, to) - logTransitionProbability(to, from);
    }
};

inline bool same_except_shape(const ModelFittingParameters &a, const ModelFittingParameters &b) {
    for (int i = 0; i < 10; i++)
        if (!(a.allParameters[i] == b.allParameters[i])) return false;
    return true;
}

class NonRigidIcpProposal : public ProposalGeneratorWithTransition {
public:
    NonRigidIcpProposal(StatisticalMeshModel &model, TriangleMesh3D &target, double stepLength, double tangentialNoise,
                        double noiseAlongNormal, const std::vector<int32_t> &modelPointIds, const std::vector<double> &targetPoints,
                        IcpProjectionDirection projectionDirection = IcpProjectionDirection::ModelSampling, bool boundaryAware = true,
                        std::string generatedBy = "ShapeIcpProposal", uint64_t seed = 1024)
        : model_(model), generatedBy_(std::move(generatedBy)), rng_(seed) {
        icp_proposal_params p{stepLength, tangentialNoise, noiseAlongNormal,
                              projectionDirection == IcpProjectionDirection::TargetSampling ? ICP_TARGET_SAMPLING : ICP_MODEL_SAMPLING,
                              boundaryAware ? 1 : 0};
        check(icp_proposal_create(model.handle(), target.handle(), &p, modelPointIds.data(), (int)modelPointIds.size(),
                                  targetPoints.data(), (int)targetPoints.size() / 3, &h_), model.ctx());
    }
    ~NonRigidIcpProposal() override { icp_proposal_destroy(h_); }
    ModelFittingParameters propose(const ModelFittingParameters &theta) override {
        std::vector<double> z(model_.rank());
        for (auto &v : z) v = normal_(rng_);                       // posterior.sample(), :55
        ModelFittingParameters out;
        out.allParameters.resize(theta.allParameters.size());
        check(icp_propose(h_, 1, theta.allParameters.data(), z.data(), out.allParameters.data()), model_.ctx());
        out.generatedBy = generatedBy_;
        return out;
    }
    double logTransitionProbability(const ModelFittingParameters &from, const ModelFittingParameters &to) override {
        double v = 0;
        check(icp_log_transition(h_, 1, from.allParameters.data(), to.allParameters.data(), &v), model_.ctx());
        return v;                                                   // -inf is a value (:73)
    }
    void flatten(double weight, std::vector<icp_component> &out, std::vector<std::string> &names) override {
        out.push_back(icp_component{ICP_PROP_ICP, 0, weight, 0.0, h_});
        names.push_back(generatedBy_);
    }
private:
    StatisticalMeshModel &model_;
    std::string generatedBy_;
    std::mt19937_64 rng_;
    std::normal_distribution<double> normal_{0.0, 1.0};
    icp_proposal h_ = nullptr;
};

class RandomShapeUpdateProposal : public ProposalGeneratorWithTransition {
public:
    RandomShapeUpdateProposal(const StatisticalMeshModel &model, double stdev, std::string generatedBy = "RandomShapeUpdateProposal",
                              uint64_t seed = 1024)
        : rank_(model.rank()), stdev_(stdev), generatedBy_(std::move(generatedBy)), rng_(seed) {}
    ModelFittingParameters propose(const ModelFittingParameters &theta) override {
        ModelFittingParameters out = theta;
        for (int j = 0; j < rank_; j++) out.allParameters[10 + j] += stdev_ * normal_(rng_);
        out.generatedBy = generatedBy_;
        return out;
    }
    double logTransitionProbability(const ModelFittingParameters &from, const ModelFittingParameters &to) override {
        if (!same_except_shape(from, to)) return -INFINITY;      // :39
        double ss = 0;
        for (int j = 0; j < rank_; j++) { double r = to.allParameters[10 + j] - from.allParameters[10 + j]; ss += r * r; }
        return -0.5 * (rank_ * std::log(2 * M_PI) + rank_ * std::log(stdev_ * stdev_) + ss / (stdev_ * stdev_));
    }
    void flatten(double weight, std::vector<icp_component> &out, std::vector<std::string> &names) override {
        out.push_back(icp_component{ICP_PROP_RANDOM_SHAPE, 0, weight, stdev_, nullptr});
        names.push_back(generatedBy_);
    }
private:
    int rank_;
    double stdev_;
    std::string generatedBy_;
    std::mt19937_64 rng_;
    std::normal_distribution<double> normal_{0.0, 1.0};
};

// kind 0: GaussianAxisRotationProposal (axis 0 roll/phi, 1 pitch/theta, 2 yaw/psi), kind 1: GaussianAxisTranslationProposal
class GaussianAxisPoseProposal : public ProposalGeneratorWithTransition {
public:
    GaussianAxisPoseProposal(int kind, double sdev, int axis, std::string generatedBy, uint64_t seed = 1024)
        : kind_(kind), slot0_(kind == 0 ? 4 : 1), axis_(axis), sdev_(sdev), generatedBy_(std::move(generatedBy)), rng_(seed) {
        if (axis < 0 || axis > 2) throw std::invalid_argument("axis < 3 required");
    }
    ModelFittingParameters propose(const ModelFittingParameters &theta) override {
        ModelFittingParameters out = theta;
        out.allParameters[slot0_ + axis_] += sdev_ * normal_(rng_);
        out.generatedBy = generatedBy_;
        return out;
    }
    double logTransitionProbability(const ModelFittingParameters &from, const ModelFittingParameters &to) override {
        for (size_t i = 0; i < from.allParameters.size(); i++) {
            if ((int)i >= slot0_ && (int)i < slot0_ + 3) continue;   // PoseProposals.scala:48 / :82
            if (!(from.allParameters[i] == to.allParameters[i])) return -INFINITY;
        }
        double r = to.allParameters[slot0_ + axis_] - from.allParameters[slot0_ + axis_];
        return -(r * r) / (2 * sdev_ * sdev_) - std::log(sdev_ * std::sqrt(2 * M_PI));
    }
    void flatten(double weight, std::vector<icp_component> &out, std::vector<std::string> &names) override {
        out.push_back(icp_component{kind_ == 0 ? ICP_PROP_ROTATION : ICP_PROP_TRANSLATION, axis_, weight, sdev_, nullptr});
        names.push_back(generatedBy_);
    }
private:
    int kind_, slot0_, axis_;
    double sdev_;
    std::string generatedBy_;
    std::mt19937_64 rng_;
    std::normal_distribution<double> normal_{0.0, 1.0};
};

// Scalismo MixtureProposal with transition probability (Appendix A8); nests like the reference's mixtures
class MixtureProposal : public ProposalGeneratorWithTransition {
public:
    explicit MixtureProposal(std::vector<std::pair<double, std::shared_ptr<ProposalGeneratorWithTransition>>> proposals, uint64_t seed = 1024)
        : gens_(std::move(proposals)), rng_(seed) {
        double tot = 0;
        for (auto &p : gens_) tot += p.first;
        for (auto &p : gens_) p.first /= tot;
    }
    ModelFittingParameters propose(const ModelFittingParameters &theta) override {
        double r = uni_(rng_), acc = 0;
        for (auto &p : gens_) { acc += p.first; if (acc >= r) return p.second->propose(theta); }
        return gens_.back().second->propose(theta);
    }
    double logTransitionProbability(const ModelFittingParameters &from, const ModelFittingParameters &to) override {
        std::vector<double> l;
        double mx = -INFINITY;
        for (auto &p : gens_) { l.push_back(p.second->logTransitionProbability(from, to)); if (std::isnan(l.back())) throw std::runtime_error("NaN transition Probability!"); mx = std::max(mx, l.back()); }
        if (mx == -INFINITY) return -INFINITY;
        double s = 0;
        for (size_t i = 0; i < l.size(); i++) s += gens_[i].first * std::exp(l[i] - mx);
        return std::log(s) + mx;
    }
    void flatten(double weight, std::vector<icp_component> &out, std::vector<std::string> &names) override {
        for (auto &p : gens_) p.second->flatten(weight * p.first, out, names);
    }
private:
    std::vector<std::pair<double, std::shared_ptr<ProposalGeneratorWithTransition>>> gens_;
    std::mt19937_64 rng_;
    std::uniform_real_distribution<double> uni_{0.0, 1.0};
};

// ---- evaluators ---------------------------------------------------------------------------------------------------
struct DistributionEvaluator {
    virtual ~DistributionEvaluator() = default;
    virtual double logValue(const ModelFittingParameters &theta) = 0;
};

// device-backed distance evaluator + EvaluationCaching (Memoize(computeLogValue, 3), evaluators/EvaluationCaching.scala:26-38)
class DeviceDistanceEvaluator : public DistributionEvaluator {
public:
    DeviceDistanceEvaluator(StatisticalMeshModel &model, TriangleMesh3D &target, icp_evaluator_params prm,
                            const std::vector<int32_t> &ids, const std::vector<double> &targetPoints)
        : model_(model), prm_(prm) {
        check(icp_evaluator_create(model.handle(), target.handle(), &prm, ids.data(), (int)ids.size(), targetPoints.data(),
                                   (int)targetPoints.size() / 3, &h_), model.ctx());
    }
    ~DeviceDistanceEvaluator() override { icp_evaluator_destroy(h_); }
    double computeLogValue(const ModelFittingParameters &theta) {
        double v[3];
        int32_t st = 0;
        check(icp_eval_log_value(h_, 1, theta.allParameters.data(), v, &st), model_.ctx());
        if (st == ICP_ERR_EMPTY_SET) throw std::runtime_error("empty.max");   // CollectiveAverage...Evaluator.scala:51
        return v[2];
    }
    double logValue(const ModelFittingParameters &theta) override {
        std::string k = theta.key();
        for (auto &e : memo_) if (e.first == k) return e.second;
        double v = computeLogValue(theta);
        if (memo_.size() >= 3) memo_.erase(memo_.begin());
        memo_.emplace_back(k, v);
        return v;
    }
    icp_evaluator handle() const { return h_; }
    const icp_evaluator_params &params() const { return prm_; }
private:
    StatisticalMeshModel &model_;
    icp_evaluator_params prm_;
    icp_evaluator h_ = nullptr;
    std::vector<std::pair<std::string, double>> memo_;
};

inline std::shared_ptr<DeviceDistanceEvaluator> IndependentPointDistanceEvaluator(StatisticalMeshModel &m, TriangleMesh3D &t, double gaussMean,
        double gaussSd, EvaluationMode mode, const std::vector<int32_t> &ids, const std::vector<double> &tp) {
    return std::make_shared<DeviceDistanceEvaluator>(m, t, icp_evaluator_params{ICP_EVAL_INDEPENDENT, (int)mode, 0, 0, gaussMean, gaussSd, 0.0}, ids, tp);
}
inline std::shared_ptr<DeviceDistanceEvaluator> HausdorffDistanceEvaluator(StatisticalMeshModel &m, TriangleMesh3D &t, double rate) {
    return std::make_shared<DeviceDistanceEvaluator>(m, t, icp_evaluator_params{ICP_EVAL_HAUSDORFF, 0, 0, 0, rate, 1.0, 1.0}, std::vector<int32_t>{}, std::vector<double>{});
}
inline std::shared_ptr<DeviceDistanceEvaluator> CollectiveAverageHausdorffDistanceBoundaryAwareEvaluator(StatisticalMeshModel &m, TriangleMesh3D &t,
        double avgMean, double avgSd, double maxRate, EvaluationMode mode, const std::vector<int32_t> &ids, const std::vector<double> &tp) {
    return std::make_shared<DeviceDistanceEvaluator>(m, t, icp_evaluator_params{ICP_EVAL_COLLECTIVE, (int)mode, 0, 0, avgMean, avgSd, maxRate}, ids, tp);
}

class ModelPriorEvaluator : public DistributionEvaluator {   // not cached in the reference either
public:
    explicit ModelPriorEvaluator(StatisticalMeshModel &model) : model_(model) {}
    double logValue(const ModelFittingParameters &theta) override {
        double v = 0;
        check(icp_eval_prior(model_.handle(), 1, theta.allParameters.data(), &v), model_.ctx());
        return v;
    }
private:
    StatisticalMeshModel &model_;
};

class ProductEvaluator : public DistributionEvaluator {
public:
    explicit ProductEvaluator(std::vector<std::shared_ptr<DistributionEvaluator>> e) : evals_(std::move(e)) {}
    double logValue(const ModelFittingParameters &theta) override {
        double s = 0;
        for (auto &e : evals_) s += e->logValue(theta);
        return s;
    }
private:
    std::vector<std::shared_ptr<DistributionEvaluator>> evals_;
};

// ---- chain log ----------------------------------------------------------------------------------------------------
struct jsonLogFormat {
    int index;
    std::string name;
    std::map<std::string, double> logvalue;
    bool status;
    std::vector<double> rigid, coeff;
    std::string datetime;
};

class JSONAcceptRejectLogger {
public:
    explicit JSONAcceptRejectLogger(std::string filePath) : path_(std::move(filePath)) {}
    std::vector<jsonLogFormat> logStatus;
    int numOfAccepted = 0, numOfRejected = 0;
    void append(const std::string &name, const std::map<std::string, double> &lv, bool ok, const double *theta, int K) {
        jsonLogFormat e{numOfAccepted + numOfRejected, name, lv, ok, {}, {}, now()};
        if (ok) { e.rigid.assign(theta + 1, theta + 10); e.coeff.assign(theta + 10, theta + 10 + K); numOfAccepted++; }   // :93-99
        else numOfRejected++;                                                                                                 // :101-105 empty arrays
        logStatus.push_back(std::move(e));
    }
    void writeLog() const {
        std::ofstream f(path_);
        if (!f) throw std::runtime_error("Writing JSON log file failed!");
        f.precision(17);
        f << "[";
        for (size_t i = 0; i < logStatus.size(); i++) {
            const auto &e = logStatus[i];
            f << (i ? ",\n" : "\n") << "  {\"index\": " << e.index << ", \"name\": \"" << e.name << "\", \"logvalue\": {";
            bool first = true;
            for (auto &kv : e.logvalue) { f << (first ? "" : ", ") << "\"" << kv.first << "\": " << kv.second; first = false; }
            f << "}, \"status\": " << (e.status ? "true" : "false") << ", \"rigid\": [";
            for (size_t k = 0; k < e.rigid.size(); k++) f << (k ? ", " : "") << e.rigid[k];
            f << "], \"coeff\": [";
            for (size_t k = 0; k < e.coeff.size(); k++) f << (k ? ", " : "") << e.coeff[k];
            f << "], \"datetime\": \"" << e.datetime << "\"}";
        }
        f << "\n]\n";
    }
private:
    static std::string now() {
        char buf[32];
        std::time_t t = std::time(nullptr);
        std::strftime(buf, sizeof buf, "%Y-%m-%d %H:%M:%S", std::localtime(&t));
        return buf;
    }
    std::string path_;
};

// ---- posterior variability from a chain log -------------------------------------------------------------------------
// apps/util/LogHelper.scala:25-42
struct LogHelper {
    // indices burnIn, burnIn + takeEveryN, ... below min(log size, total), each walked back to the last accepted entry
    static std::vector<std::pair<const jsonLogFormat *, int>> samplesFromLog(const std::vector<jsonLogFormat> &log, int takeEveryN = 50,
                                                                             int total = 100, int burnIn = 0) {
        std::vector<std::pair<const jsonLogFormat *, int>> out;
        const int end = std::min((int)log.size(), total);
        for (int i = burnIn; i < end && (int)out.size() < total; i += takeEveryN) {
            int j = i;
            while (!log[j].status)
                if (--j < 0) throw std::out_of_range("no accepted sample at or before the requested log index");
            out.emplace_back(&log[j], j);
        }
        return out;
    }
    // JSONAcceptRejectLogger.sampleToModelParameters (:135-141): scale 1, the logged rigid block and coefficients
    static ModelFittingParameters sampleToModelParameters(const jsonLogFormat &e) {
        ModelFittingParameters p;
        p.allParameters.assign(1, 1.0);
        p.allParameters.insert(p.allParameters.end(), e.rigid.begin(), e.rigid.end());
        p.allParameters.insert(p.allParameters.end(), e.coeff.begin(), e.coeff.end());
        p.generatedBy = e.name;
        return p;
    }
};

// apps/util/PosteriorVariability.scala:26-74 on parameter vectors: reconstruction, normals and the per-vertex reduction run
// on the device in one call (icp_posterior_variability)
struct PosteriorVariability {
    struct Maps { std::vector<double> mean, cov, total, normal; };
    static Maps statistics(const StatisticalMeshModel &model, const std::vector<ModelFittingParameters> &samples, bool sumNormals = true,
                           const ModelFittingParameters *ref = nullptr) {
        const int N = model.numberOfPoints(), L = model.rank() + 10;
        std::vector<double> th;
        th.reserve(samples.size() * (size_t)L);
        for (const auto &s : samples) {
            if ((int)s.allParameters.size() != L) throw std::invalid_argument("sample of the wrong rank");
            th.insert(th.end(), s.allParameters.begin(), s.allParameters.end());
        }
        Maps m;
        m.mean.resize((size_t)3 * N); m.cov.resize((size_t)9 * N); m.total.resize(N); m.normal.resize(N);
        check(icp_posterior_variability(model.handle(), (int32_t)samples.size(), th.data(), sumNormals ? 1 : 0,
                                        (!sumNormals && ref) ? ref->allParameters.data() : nullptr, m.mean.data(), m.cov.data(),
                                        m.total.data(), m.normal.data()), model.ctx());
        return m;
    }
    static std::vector<double> computeDistanceMapFromMeshesTotal(const StatisticalMeshModel &model, const std::vector<ModelFittingParameters> &samples) {
        return statistics(model, samples).total;
    }
    static std::vector<double> computeDistanceMapFromMeshesNormal(const StatisticalMeshModel &model, const std::vector<ModelFittingParameters> &samples,
                                                                  const ModelFittingParameters *ref, bool sumNormals) {
        return statistics(model, samples, sumNormals, ref).normal;
    }
};

// ---- GPMM construction from analytic kernels (apps/femur/CreateGPModel.scala:68-93) -------------------------------
// sum of terms scale * exp(-|x - y|^2 / sigma^2) * A: what `*` and `+` build from Scalismo's GaussianKernel3D / DiagonalKernel3D
class MatrixValuedKernel {
public:
    std::vector<icp_kernel_term> terms;
    static MatrixValuedKernel gaussian(double sigma, double scale = 1.0) {          // DiagonalKernel3D(GaussianKernel3D(sigma), 3) * scale
        MatrixValuedKernel k;
        icp_kernel_term t{scale, sigma, {1, 0, 0, 0, 1, 0, 0, 0, 1}};
        k.terms.push_back(t);
        return k;
    }
    MatrixValuedKernel operator*(double f) const { MatrixValuedKernel k = *this; for (auto &t : k.terms) t.scale *= f; return k; }
    MatrixValuedKernel operator+(const MatrixValuedKernel &o) const {
        MatrixValuedKernel k = *this;
        k.terms.insert(k.terms.end(), o.terms.begin(), o.terms.end());
        return k;
    }
    MatrixValuedKernel withMatrix(const double B[9]) const {                         // baseMatrix * kernel(x, y) (:79)
        MatrixValuedKernel k = *this;
        for (auto &t : k.terms) {
            double a[9];
            for (int r = 0; r < 3; r++)
                for (int c = 0; c < 3; c++) a[3 * r + c] = B[3 * r] * t.A[c] + B[3 * r + 1] * t.A[3 + c] + B[3 * r + 2] * t.A[6 + c];
            std::memcpy(t.A, a, sizeof a);
        }
        return k;
    }
};

struct LowRankGaussianProcess {
    struct Model { std::vector<double> basis, variance; };   // pcaBasis 3N x K row-major, pcaVariance K
    // LowRankGaussianProcess.approximateGPNystrom (:86), every step on the device: kernel matrix of the Nystrom points, its
    // leading eigenpairs (one-sided Jacobi), Nystrom extension to all model points
    static Model approximateGPNystrom(Context &ctx, const MatrixValuedKernel &kernel, const std::vector<double> &points,
                                      const std::vector<double> &nystromPoints, int numBasisFunctions) {
        const int N = (int)points.size() / 3, m = (int)nystromPoints.size() / 3, n = 3 * m, K = numBasisFunctions;
        std::vector<double> kmm((size_t)n * n), w(K), V((size_t)n * K);
        check(icp_gpmm_kernel_matrix(ctx.handle(), m, nystromPoints.data(), m, nystromPoints.data(), kernel.terms.data(),
                                     (int)kernel.terms.size(), kmm.data()), ctx.handle());
        check(icp_gpmm_eigen_psd(ctx.handle(), n, kmm.data(), K, w.data(), V.data()), ctx.handle());
        Model out;
        out.basis.resize((size_t)3 * N * K);
        out.variance.resize(K);
        check(icp_gpmm_nystrom_extend(ctx.handle(), N, points.data(), m, nystromPoints.data(), kernel.terms.data(),
                                      (int)kernel.terms.size(), K, V.data(), w.data(), out.basis.data(), out.variance.data()), ctx.handle());
        return out;
    }
};

// ---- Metropolis-Hastings ---------------------------------------------------------------------------------------------
// Scalismo MetropolisHastings.next over the per-call (drop-in) classes
class MetropolisHastings {
public:
    MetropolisHastings(ProposalGeneratorWithTransition &generator, DistributionEvaluator &evaluator, uint64_t seed = 1024)
        : gen_(generator), eval_(evaluator), rng_(seed) {}
    ModelFittingParameters next(const ModelFittingParameters &current, bool *accepted = nullptr) {
        double currentP = eval_.logValue(current);
        ModelFittingParameters proposal = gen_.propose(current);
        double proposalP = eval_.logValue(proposal);
        double t = gen_.logTransitionRatio(current, proposal);
        double a = proposalP - currentP - t;
        bool ok = a > 0.0 || uni_(rng_) < std::exp(a);
        if (accepted) *accepted = ok;
        return ok ? proposal : current;
    }
private:
    ProposalGeneratorWithTransition &gen_;
    DistributionEvaluator &eval_;
    std::mt19937_64 rng_;
    std::uniform_real_distribution<double> uni_{0.0, 1.0};
};

// SamplingRegistration.runfitting (SamplingRegistration.scala:45-93) on the fused device runner
class SamplingRegistration {
public:
    SamplingRegistration(StatisticalMeshModel &model, TriangleMesh3D &sample, uint64_t seed = 1024) : model_(model), sample_(sample), seed_(seed) {}
    struct Result {
        ModelFittingParameters best;
        double bestProduct = -INFINITY;
        int64_t accepted = 0;
        int steps = 0;
        std::vector<jsonLogFormat> log;   // the chain log in the reference's record layout (also written to jsonName)
        int64_t variabilitySamples = 0;   // with a variability request: S, and the maps (PosteriorVariability layout)
        PosteriorVariability::Maps variability;
    };
    // PosteriorVariability over the samples LogHelper.samplesFromLog(log, takeEveryN, total, burnIn) selects, accumulated
    // inside the run (icp_chain_set_statistics / icp_chain_statistics) instead of from the chain log
    struct VariabilityRequest {
        int64_t takeEveryN = 50, total = 0, burnIn = 0;   // total <= 0: no limit
        bool sumNormals = true;
        const ModelFittingParameters *ref = nullptr;      // sumNormals == false: normals of this state (nullptr: reference mesh)
    };
    // evaluator: the device evaluator behind evaluators("product") - build it with makeProductEvaluator so that it
    // carries prior x distance (ProductEvaluators.scala:44-47); distanceKey: the key of the distance term in the
    // evaluator map ("distance", "distance_haussdorff", "collective_distance")
    Result runfitting(DeviceDistanceEvaluator &evaluator, const std::string &distanceKey, ProposalGeneratorWithTransition &generator,
                      int numOfSamples, const ModelFittingParameters &initial, const std::string &jsonName = "",
                      const VariabilityRequest *variability = nullptr) {
        std::vector<icp_component> comps;
        std::vector<std::string> names;
        generator.flatten(1.0, comps, names);
        icp_evaluator ev = evaluator.handle();
        const int K = model_.rank(), L = K + 10;
        icp_chain chain = nullptr;
        check(icp_chain_create(model_.handle(), sample_.handle(), comps.data(), (int)comps.size(), ev, 1, &chain), model_.ctx());
        std::vector<int32_t> comp(numOfSamples);
        std::vector<uint8_t> acc(numOfSamples);
        std::vector<double> vals((size_t)3 * numOfSamples), thl((size_t)L * numOfSamples), fin(L);
        int64_t nacc = 0;
        icp_chain_io io{};
        io.seed = seed_;
        io.log_component = comp.data(); io.log_accepted = acc.data(); io.log_values = vals.data(); io.log_theta = thl.data();
        io.theta_final = fin.data(); io.n_accepted = &nacc;
        Result r;
        int32_t rc = ICP_OK;
        if (variability) {
            icp_chain_stats_params sp{variability->burnIn, variability->takeEveryN, variability->total, variability->sumNormals ? 1 : 0, 0};
            rc = icp_chain_set_statistics(chain, &sp);
        }
        if (rc == ICP_OK) rc = icp_chain_run(chain, 1, numOfSamples, initial.allParameters.data(), &io);
        if (rc == ICP_OK && variability) {
            const int N = model_.numberOfPoints();
            PosteriorVariability::Maps &v = r.variability;
            v.mean.resize((size_t)3 * N); v.cov.resize((size_t)9 * N); v.total.resize(N); v.normal.resize(N);
            const ModelFittingParameters *ref = variability->sumNormals ? nullptr : variability->ref;
            rc = icp_chain_statistics(chain, -1, variability->sumNormals ? 1 : 0, ref ? ref->allParameters.data() : nullptr,
                                      &r.variabilitySamples, v.mean.data(), v.cov.data(), v.total.data(), v.normal.data());
        }
        icp_chain_destroy(chain);
        check(rc, model_.ctx());
        r.best = initial; r.accepted = nacc; r.steps = numOfSamples;
        JSONAcceptRejectLogger logger(jsonName);
        for (int s = 0; s < numOfSamples; s++) {
            bool ok = acc[s] != 0;
            if (ok && vals[3 * s] > r.bestProduct) {          // BestSampleLogger
                r.bestProduct = vals[3 * s];
                r.best.allParameters.assign(thl.begin() + (size_t)s * L, thl.begin() + (size_t)(s + 1) * L);
                r.best.generatedBy = names[comp[s]];
            }
            logger.append(names[comp[s]], {{"product", vals[3 * s]}, {"prior", vals[3 * s + 1]}, {distanceKey, vals[3 * s + 2]}}, ok,
                          thl.data() + (size_t)s * L, K);
        }
        if (!jsonName.empty()) logger.writeLog();
        r.log = std::move(logger.logStatus);
        return r;
    }
private:
    StatisticalMeshModel &model_;
    TriangleMesh3D &sample_;
    uint64_t seed_;
};

// ProductEvaluators.proximityAndIndependent on the device: prior x Gaussian-point distance in one evaluator handle
inline std::shared_ptr<DeviceDistanceEvaluator> makeProductEvaluator(StatisticalMeshModel &m, TriangleMesh3D &t, icp_evaluator_params prm,
                                                                     const std::vector<int32_t> &ids, const std::vector<double> &tp) {
    prm.use_prior = 1;
    return std::make_shared<DeviceDistanceEvaluator>(m, t, prm, ids, tp);
}

}  // namespace icp_host
