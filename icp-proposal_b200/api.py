"""Host-side mirror of the reference's operator API for the hot path (same names, argument meaning and
error behaviour as the Scala classes), implemented as thin calls into libicpcuda.so.

The reference is Scala on Scalismo (no JVM in this image), so this mirror is what the parity tests and
bench.py drive; INTEGRATION.md shows the equivalent Scala/Panama binding. Paths below are relative to
src/main/scala of the reference.

  ModelFittingParameters, PoseParameters, ShapeParameters, ScaleParameter   api/sampling/ModelFittingParameters.scala
  NonRigidIcpProposal                                                       api/sampling/proposals/NonRigidIcpProposal.scala
  RandomShapeUpdateProposal                                                 api/sampling/proposals/RandomShapeUpdateProposal.scala
  GaussianAxisRotationProposal, GaussianAxisTranslationProposal            api/sampling/proposals/PoseProposals.scala
  IndependentPointDistanceEvaluator, HausdorffDistanceEvaluator,
  CollectiveAverageHausdorffDistanceBoundaryAwareEvaluator,
  ModelPriorEvaluator, AcceptAllEvaluator, EvaluationCaching               api/sampling/evaluators/*.scala
  ProductEvaluators, MixedProposalDistributions                            api/sampling/{ProductEvaluators,MixedProposalDistributions}.scala
  MixtureProposal, MetropolisHastings, ProductEvaluator                    Scalismo (SURVEY.md Appendix A8/A9)
  SamplingRegistration                                                      api/sampling/SamplingRegistration.scala
  JSONAcceptRejectLogger, jsonLogFormat                                     api/sampling/loggers/JSONAcceptRejectLogger.scala
  IcpBasedSurfaceFitting, RegistrationComparison                           api/other/*.scala
  LogHelper, PosteriorVariability                                           apps/util/{LogHelper,PosteriorVariability}.scala
  GaussianKernel3D, DiagonalKernel3D, MatrixValuedKernel,
  LowRankGaussianProcess.approximateGPNystrom, femurKernel                  apps/femur/CreateGPModel.scala (Scalismo kernels, SURVEY 8f rank 4)

Only O(K) bookkeeping happens here (as it does on the JVM in the reference); everything that touches a mesh
or a K x K matrix runs on the GPU. There is no CPU fallback.
"""
from __future__ import annotations

import dataclasses
import datetime
import json
import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib, core

# ---- enums ---------------------------------------------------------------------------------------------
ModelSampling, TargetSampling, ModelAndTargetSampling = "ModelSampling", "TargetSampling", "ModelAndTargetSampling"
ModelToTargetEvaluation, TargetToModelEvaluation, SymmetricEvaluation = 0, 1, 2
RollAxis, PitchAxis, YawAxis = 0, 1, 2   # rotation._1 (phi), ._2 (theta), ._3 (psi)  (PoseProposals.scala:36-44)


# ---- parameters ----------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class ScaleParameter:
    s: float = 1.0

    @property
    def parameters(self):
        return np.array([self.s])


@dataclasses.dataclass(frozen=True)
class PoseParameters:
    translation: Tuple[float, float, float]
    rotation: Tuple[float, float, float]
    rotationCenter: Tuple[float, float, float]

    @property
    def parameters(self):
        return np.concatenate([np.asarray(self.translation, float), np.asarray(self.rotation, float),
                               np.asarray(self.rotationCenter, float)])


@dataclasses.dataclass(frozen=True)
class ShapeParameters:
    parameters: np.ndarray


class ModelFittingParameters:
    """theta container; equality is by the bytes of allParameters (the reference compares hash codes,
    ModelFittingParameters.scala:54-61); generatedBy is not part of equality."""

    def __init__(self, scalaParameter: ScaleParameter, poseParameters: PoseParameters, shapeParameters: ShapeParameters,
                 generatedBy: str = "Anonymous"):
        self.scalaParameter, self.poseParameters, self.shapeParameters = scalaParameter, poseParameters, shapeParameters
        self.generatedBy = generatedBy
        self.allParameters = np.concatenate([scalaParameter.parameters, poseParameters.parameters,
                                             np.asarray(shapeParameters.parameters, float)])

    @staticmethod
    def from_vector(theta, generatedBy="Anonymous"):
        theta = np.asarray(theta, float)
        return ModelFittingParameters(ScaleParameter(float(theta[0])),
                                      PoseParameters(tuple(theta[1:4]), tuple(theta[4:7]), tuple(theta[7:10])),
                                      ShapeParameters(theta[10:].copy()), generatedBy)

    def copy(self, **kw):
        d = dict(scalaParameter=self.scalaParameter, poseParameters=self.poseParameters, shapeParameters=self.shapeParameters,
                 generatedBy=self.generatedBy)
        d.update(kw)
        return ModelFittingParameters(**d)

    def __eq__(self, other):
        return isinstance(other, ModelFittingParameters) and self.allParameters.tobytes() == other.allParameters.tobytes()

    def __hash__(self):
        return hash(self.allParameters.tobytes())


# ---- meshes / model --------------------------------------------------------------------------------------
class StatisticalMeshModel(core.Model):
    """scalismo.statisticalmodel.StatisticalMeshModel stand-in backed by icp_model."""

    def instance(self, coefficients):
        return self.reconstruct(self.theta(alpha=coefficients, center=(0, 0, 0)))[0]

    def transformedMesh(self, theta: ModelFittingParameters):
        """ModelFittingParameters.transformedMesh (ModelFittingParameters.scala:108-110)."""
        return self.reconstruct(theta.allParameters)[0]

    def initial_parameters(self) -> ModelFittingParameters:
        """SamplingRegistration.initialParametersZero (SamplingRegistration.scala:40-43)."""
        c = self.ref.mean(0)
        return ModelFittingParameters(ScaleParameter(1.0), PoseParameters((0, 0, 0), (0, 0, 0), tuple(c)),
                                      ShapeParameters(np.zeros(self.K)))


class TriangleMesh3D(core.Target):
    pass


def _decimated_ids(model, n):
    """decimatedModel.referenceMesh.pointSet.pointIds are 0..n_dec-1 and index the FULL mesh (SURVEY Appendix B1)."""
    return np.arange(min(int(n), model.N), dtype=np.int32)


def _decimated_points(target, n):
    """Stand-in for target.operations.decimate(n).pointSet.points when the caller does not pass the list it got from
    Scalismo/VTK: an even subsample of the target vertices (n >= Nt keeps the mesh unchanged, as VTK does)."""
    nt = len(target.verts)
    if n >= nt:
        return target.verts.copy()
    return target.verts[np.linspace(0, nt - 1, int(n)).round().astype(int)].copy()


# ---- densities (Breeze, SURVEY Appendix A15) ----------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class Gaussian:
    mu: float
    sigma: float

    def logPdf(self, x):
        return -((x - self.mu) ** 2) / (2 * self.sigma ** 2) - math.log(self.sigma * math.sqrt(2 * math.pi))


@dataclasses.dataclass(frozen=True)
class Exponential:
    rate: float

    def logPdf(self, x):
        return math.log(self.rate) - self.rate * x


# ---- proposals ---------------------------------------------------------------------------------------------
class NonRigidIcpProposal:
    """ProposalGenerator + TransitionProbability (NonRigidIcpProposal.scala:30-153)."""

    def __init__(self, model: StatisticalMeshModel, target: TriangleMesh3D, stepLength, tangentialNoise, noiseAlongNormal,
                 numOfSamplePoints, projectionDirection=ModelSampling, boundaryAware=True, generatedBy="ShapeIcpProposal",
                 rand: Optional[np.random.Generator] = None, model_point_ids=None, target_points=None):
        if projectionDirection not in (ModelSampling, TargetSampling):
            raise ValueError("a single NonRigidIcpProposal samples one direction; use MixedProposalDistributions.mixedProposalICP")
        self.model, self.target = model, target
        self.stepLength, self.generatedBy, self.projectionDirection = stepLength, generatedBy, projectionDirection
        self.rand = rand if rand is not None else np.random.default_rng()
        ids = _decimated_ids(model, numOfSamplePoints) if model_point_ids is None else model_point_ids
        tp = _decimated_points(target, numOfSamplePoints) if target_points is None else target_points
        self.dev = core.IcpProposal(model, target, stepLength, tangentialNoise, noiseAlongNormal,
                                    _lib.TARGET_SAMPLING if projectionDirection == TargetSampling else _lib.MODEL_SAMPLING,
                                    boundaryAware, ids, tp)

    def propose(self, theta: ModelFittingParameters) -> ModelFittingParameters:
        z = self.rand.standard_normal(self.model.K)          # posterior.sample(), :55
        out = self.dev.propose(theta.allParameters, z)[0]
        return ModelFittingParameters.from_vector(out, self.generatedBy)

    def logTransitionProbability(self, frm: ModelFittingParameters, to: ModelFittingParameters) -> float:
        return float(self.dev.log_transition(frm.allParameters, to.allParameters)[0])

    def device_component(self, weight):
        return dict(kind=_lib.PROP_ICP, weight=weight, proposal=self.dev, name=self.generatedBy)


class RandomShapeUpdateProposal:
    """RandomShapeUpdateProposal.scala:25-46 (O(K) host arithmetic, as in the reference)."""

    def __init__(self, model, stdev, generatedBy="RandomShapeUpdateProposal", rand=None):
        self.rank, self.stdev, self.generatedBy = model.K, stdev, generatedBy
        self.rand = rand if rand is not None else np.random.default_rng()

    def propose(self, theta):
        a = theta.shapeParameters.parameters + self.stdev * self.rand.standard_normal(self.rank)
        return theta.copy(shapeParameters=ShapeParameters(a), generatedBy=self.generatedBy)

    def logTransitionProbability(self, frm, to):
        if not np.array_equal(to.allParameters[:10], frm.allParameters[:10]):
            return -math.inf
        r = to.shapeParameters.parameters - frm.shapeParameters.parameters
        k, s2 = self.rank, self.stdev ** 2
        return -0.5 * (k * math.log(2 * math.pi) + k * math.log(s2) + float(r @ r) / s2)

    def device_component(self, weight):
        return dict(kind=_lib.PROP_RANDOM_SHAPE, weight=weight, sd=self.stdev, name=self.generatedBy)


class _GaussianAxisProposal:
    kind, slot0 = None, None

    def __init__(self, sdev, axis, generatedBy, rand=None):
        self.sdev, self.axis, self.generatedBy = sdev, int(axis), generatedBy
        if not 0 <= self.axis < 3:
            raise ValueError("axis < 3 required")
        self.rand = rand if rand is not None else np.random.default_rng()

    def propose(self, theta):
        v = theta.allParameters.copy()
        v[self.slot0 + self.axis] += self.sdev * self.rand.standard_normal()
        return ModelFittingParameters.from_vector(v, self.generatedBy)

    def logTransitionProbability(self, frm, to):
        a, b = frm.allParameters, to.allParameters
        mask = np.ones(len(a), bool)
        mask[self.slot0:self.slot0 + 3] = False            # PoseProposals.scala:48 / :82
        if not np.array_equal(a[mask], b[mask]):
            return -math.inf
        return Gaussian(0.0, self.sdev).logPdf(b[self.slot0 + self.axis] - a[self.slot0 + self.axis])

    def device_component(self, weight):
        return dict(kind=self.kind, weight=weight, sd=self.sdev, axis=self.axis, name=self.generatedBy)


class GaussianAxisRotationProposal(_GaussianAxisProposal):
    kind, slot0 = _lib.PROP_ROTATION, 4

    def __init__(self, sdevRot, axis, generatedBy="RotationProposal", rand=None):
        super().__init__(sdevRot, axis, generatedBy, rand)


class GaussianAxisTranslationProposal(_GaussianAxisProposal):
    kind, slot0 = _lib.PROP_TRANSLATION, 1

    def __init__(self, sdevTrans, axis, generatedBy="TranslationProposal", rand=None):
        super().__init__(sdevTrans, axis, generatedBy, rand)


class MixtureProposal:
    """Scalismo MixtureProposal with transition probability (SURVEY Appendix A8); nests like the reference's."""

    def __init__(self, proposals: Sequence[Tuple[float, object]], rand=None):
        tot = sum(w for w, _ in proposals)
        self.weights = [w / tot for w, _ in proposals]
        self.generators = [p for _, p in proposals]
        self.rand = rand if rand is not None else np.random.default_rng()

    @staticmethod
    def fromProposalsWithTransition(*proposals, rand=None):
        return MixtureProposal(list(proposals), rand)

    def propose(self, current):
        r = self.rand.random()
        cdf = np.cumsum(self.weights)
        i = int(np.argmax(cdf >= r)) if (cdf >= r).any() else len(cdf) - 1
        return self.generators[i].propose(current)

    def logTransitionProbability(self, frm, to):
        ls = [g.logTransitionProbability(frm, to) for g in self.generators]
        if any(math.isnan(l) for l in ls):
            raise ArithmeticError("NaN transition Probability!")
        mx = max(ls)
        if mx == -math.inf:
            return -math.inf
        return math.log(sum(w * math.exp(l - mx) for w, l in zip(self.weights, ls))) + mx

    def logTransitionRatio(self, frm, to):
        return self.logTransitionProbability(frm, to) - self.logTransitionProbability(to, frm)

    def flatten(self, scale=1.0):
        """Leaf components with their effective weights, for the fused device chain."""
        out = []
        for w, g in zip(self.weights, self.generators):
            out += g.flatten(scale * w) if isinstance(g, MixtureProposal) else [g.device_component(scale * w)]
        return out


class MixedProposalDistributions:
    """api/sampling/MixedProposalDistributions.scala:29-68."""

    @staticmethod
    def mixedRandomPoseProposal(rotYaw=0.01, rotPitch=0.01, rotRoll=0.01, transX=0.1, transY=0.1, transZ=0.1, rand=None):
        return MixtureProposal([
            (0.5, GaussianAxisRotationProposal(rotYaw, YawAxis, f"RotationYaw-{rotYaw}", rand)),
            (0.5, GaussianAxisRotationProposal(rotPitch, PitchAxis, f"RotationPitch-{rotPitch}", rand)),
            (0.5, GaussianAxisRotationProposal(rotRoll, RollAxis, f"RotationRoll-{rotRoll}", rand)),
            (0.5, GaussianAxisTranslationProposal(transX, 0, f"TranslationX-{transX}", rand)),
            (0.5, GaussianAxisTranslationProposal(transY, 1, f"TranslationY-{transY}", rand)),
            (0.5, GaussianAxisTranslationProposal(transZ, 2, f"TranslationZ-{transZ}", rand))], rand)

    @staticmethod
    def mixedRandomShapeProposal(model, steps=(0.1,), rand=None):
        return MixtureProposal([(0.5, RandomShapeUpdateProposal(model, s, f"RandomShape-{s}", rand)) for s in steps], rand)

    @staticmethod
    def mixedProposalICP(model, target, numOfSamplePoints, projectionDirection=ModelAndTargetSampling, tangentialNoise=10.0,
                         noiseAlongNormal=5.0, stepLength=0.1, boundaryAware=True, rand=None, model_point_ids=None,
                         target_points=None):
        mk = lambda d: NonRigidIcpProposal(model, target, stepLength, tangentialNoise, noiseAlongNormal, numOfSamplePoints, d,
                                           boundaryAware, f"IcpProposal-{d}-{stepLength}Step", rand, model_point_ids, target_points)
        if projectionDirection == TargetSampling:
            props = [(0.5, mk(TargetSampling))]
        elif projectionDirection == ModelSampling:
            props = [(0.5, mk(ModelSampling))]
        else:
            props = [(0.5, mk(TargetSampling)), (0.5, mk(ModelSampling))]   # :58-64 target first
        return MixtureProposal(props, rand)


# ---- evaluators ----------------------------------------------------------------------------------------------
class EvaluationCaching:
    """Memoize(computeLogValue, 3) (evaluators/EvaluationCaching.scala:26-38)."""

    _cache_size = 3

    def logValue(self, sample):
        cache = self.__dict__.setdefault("_memo", {})
        key = sample.allParameters.tobytes()
        if key not in cache:
            if len(cache) >= self._cache_size:
                cache.pop(next(iter(cache)))
            cache[key] = self.computeLogValue(sample)
        return cache[key]


class _DeviceEvaluator(EvaluationCaching):
    dev: core.Evaluator

    def computeLogValue(self, sample):
        v, st = self.dev.log_value(sample.allParameters, with_status=True)
        if st[0] == _lib.ERR_EMPTY_SET:
            raise ValueError("empty.max")   # the reference throws UnsupportedOperationException("empty.max")
        return float(v[0, 2])


class IndependentPointDistanceEvaluator(_DeviceEvaluator):
    def __init__(self, model, targetMesh, likelihoodModel: Gaussian, evaluationMode, numberOfPointsForComparison,
                 model_point_ids=None, target_points=None):
        ids = _decimated_ids(model, numberOfPointsForComparison) if model_point_ids is None else model_point_ids
        tp = _decimated_points(targetMesh, numberOfPointsForComparison) if target_points is None else target_points
        self.dev = core.Evaluator(model, targetMesh, _lib.EVAL_INDEPENDENT, evaluationMode, False, likelihoodModel.mu,
                                  likelihoodModel.sigma, 0.0, ids, tp)


class HausdorffDistanceEvaluator(_DeviceEvaluator):
    def __init__(self, model, targetMesh, likelihoodModel: Exponential):
        self.dev = core.Evaluator(model, targetMesh, _lib.EVAL_HAUSDORFF, 0, False, likelihoodModel.rate)


class CollectiveAverageHausdorffDistanceBoundaryAwareEvaluator(_DeviceEvaluator):
    def __init__(self, model, targetMesh, likelihoodModelAvg: Gaussian, likelihoodModelMax: Exponential, evaluationMode,
                 numberOfPointsForComparison, model_point_ids=None, target_points=None):
        ids = _decimated_ids(model, numberOfPointsForComparison) if model_point_ids is None else model_point_ids
        tp = _decimated_points(targetMesh, numberOfPointsForComparison) if target_points is None else target_points
        self.dev = core.Evaluator(model, targetMesh, _lib.EVAL_COLLECTIVE, evaluationMode, False, likelihoodModelAvg.mu,
                                  likelihoodModelAvg.sigma, likelihoodModelMax.rate, ids, tp)


class ModelPriorEvaluator:
    """Not cached in the reference either (evaluators/ModelPriorEvaluator.scala:24-31)."""

    def __init__(self, model):
        self.model = model

    def logValue(self, theta):
        return float(self.model.prior(theta.allParameters)[0])


class AcceptAllEvaluator(EvaluationCaching):
    def computeLogValue(self, sample):
        return 0.0


class ProductEvaluator:
    def __init__(self, *evaluators):
        self.evaluators = evaluators

    def logValue(self, sample):
        return sum(e.logValue(sample) for e in self.evaluators)


class ProductEvaluators:
    """api/sampling/ProductEvaluators.scala:28-94: name -> evaluator maps (keys become the JSON logvalue keys)."""

    @staticmethod
    def acceptAll():
        return {"product": ProductEvaluator(AcceptAllEvaluator())}

    @staticmethod
    def proximityAndIndependent(model, target, evaluationMode, uncertainty=1.0, numberOfEvaluationPoints=100, **kw):
        dist = IndependentPointDistanceEvaluator(model, target, Gaussian(0, uncertainty), evaluationMode, numberOfEvaluationPoints, **kw)
        prior = ModelPriorEvaluator(model)
        return {"product": ProductEvaluator(prior, dist), "prior": prior, "distance": dist}

    @staticmethod
    def proximityAndHausdorff(model, target, uncertainty=1.0):
        dist = HausdorffDistanceEvaluator(model, target, Exponential(uncertainty))
        prior = ModelPriorEvaluator(model)
        return {"product": ProductEvaluator(prior, dist), "prior": prior, "distance_haussdorff": dist}

    @staticmethod
    def proximityAndCollectiveHausdorffBoundaryAware(model, target, evaluationMode, uncertaintyAvg=1.0, uncertaintyMax=5.0,
                                                     mean=0.0, numberOfEvaluationPoints=100, **kw):
        dist = CollectiveAverageHausdorffDistanceBoundaryAwareEvaluator(model, target, Gaussian(mean, uncertaintyAvg),
                                                                        Exponential(uncertaintyMax), evaluationMode,
                                                                        numberOfEvaluationPoints, **kw)
        prior = ModelPriorEvaluator(model)
        return {"product": ProductEvaluator(prior, dist), "prior": prior, "collective_distance": dist}


# ---- chain log -----------------------------------------------------------------------------------------------
@dataclasses.dataclass
class jsonLogFormat:
    index: int
    name: str
    logvalue: Dict[str, float]
    status: bool
    rigid: List[float]
    coeff: List[float]
    datetime: str


class JSONAcceptRejectLogger:
    """loggers/JSONAcceptRejectLogger.scala:42-182: same record layout and file format."""

    def __init__(self, filePath: Optional[str], evaluators: Optional[Dict[str, object]] = None):
        self.filePath, self.evaluators = filePath, evaluators
        if filePath and os.path.dirname(filePath) and not os.path.isdir(os.path.dirname(filePath)):
            raise IOError(f"JSON log path does not exist: {os.path.dirname(filePath)}!")
        self.logStatus: List[jsonLogFormat] = []
        self.logSamples: List[ModelFittingParameters] = []
        self.numOfAccepted = self.numOfRejected = 0

    @property
    def totalSamples(self):
        return self.numOfAccepted + self.numOfRejected

    @staticmethod
    def _now():
        return datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S")

    def _map(self, sample, default):
        if self.evaluators is not None:
            return {k: float(e.logValue(sample)) for k, e in self.evaluators.items()}
        return {"product": float(default)}

    def accept(self, current, sample, generator, evaluator):
        self.logStatus.append(jsonLogFormat(self.totalSamples, sample.generatedBy, self._map(sample, evaluator.logValue(sample)), True,
                                            sample.poseParameters.parameters.tolist(), sample.shapeParameters.parameters.tolist(),
                                            self._now()))
        self.logSamples.append(sample)
        self.numOfAccepted += 1

    def reject(self, current, sample, generator, evaluator):
        # the CURRENT state's values with empty parameter arrays (:101-105)
        self.logStatus.append(jsonLogFormat(self.totalSamples, sample.generatedBy, self._map(current, evaluator.logValue(current)),
                                            False, [], [], self._now()))
        self.numOfRejected += 1

    def append_device_log(self, names, keys, component, accepted, values, theta):
        """Appends the log of one device chain (icp_chain_run) in the reference's record layout."""
        for s in range(len(component)):
            ok = bool(accepted[s])
            lv = dict(zip(keys, (float(v) for v in values[s])))
            th = theta[s]
            self.logStatus.append(jsonLogFormat(self.totalSamples, names[int(component[s])], lv, ok,
                                                th[1:10].tolist() if ok else [], th[10:].tolist() if ok else [], self._now()))
            if ok:
                self.logSamples.append(ModelFittingParameters.from_vector(th, names[int(component[s])]))
                self.numOfAccepted += 1
            else:
                self.numOfRejected += 1

    def percentRejected(self):
        return round(self.numOfRejected / max(self.totalSamples, 1) + 1e-12, 2)

    def percentAccepted(self):
        return 1.0 - self.percentRejected()

    def percentAcceptedOfType(self, name):
        f = [l for l in self.logStatus if l.name == name]
        return sum(l.status for l in f) / len(f) if f else float("nan")

    def prettyPrint(self):
        # spray-json cannot represent NaN / infinities (it writes null): keep the file loadable by the reference's loader
        def clean(x):
            if isinstance(x, float) and not math.isfinite(x):
                return None
            if isinstance(x, dict):
                return {k: clean(v) for k, v in x.items()}
            if isinstance(x, list):
                return [clean(v) for v in x]
            return x
        return json.dumps([clean(dataclasses.asdict(l)) for l in self.logStatus], indent=2, allow_nan=False)

    def writeLog(self):
        try:
            with open(self.filePath, "w") as f:
                f.write(self.prettyPrint())
        except Exception as e:
            raise IOError("Writing JSON log file failed!") from e

    def loadLog(self):
        with open(self.filePath) as f:
            return [jsonLogFormat(**d) for d in json.load(f)]

    @staticmethod
    def sampleToModelParameters(sample: jsonLogFormat) -> ModelFittingParameters:
        r = sample.rigid
        return ModelFittingParameters(ScaleParameter(1.0), PoseParameters(tuple(r[0:3]), tuple(r[3:6]), tuple(r[6:9])),
                                      ShapeParameters(np.asarray(sample.coeff, float)))

    def getBestFittingParsFromJSON(self):
        best = max((l for l in self.loadLog() if l.status), key=lambda l: l.logvalue["product"])
        return self.sampleToModelParameters(best)


# ---- posterior variability from a chain log ------------------------------------------------------------------------
class LogHelper:
    """apps/util/LogHelper.scala:25-42."""

    @staticmethod
    def samplesFromLog(log: Sequence[jsonLogFormat], takeEveryN: int = 50, total: int = 100, burnIn: int = 0):
        def getLogIndex(i):
            while not log[i].status:
                i -= 1
                if i < 0:
                    raise IndexError("no accepted sample at or before the requested log index")
            return i
        filtered = [(log[j], j) for j in (getLogIndex(i) for i in range(burnIn, min(len(log), total), takeEveryN))]
        return filtered[:min(total, len(filtered))]

    @staticmethod
    def logSamples2thetas(log: Sequence[jsonLogFormat]) -> np.ndarray:
        return np.stack([JSONAcceptRejectLogger.sampleToModelParameters(l).allParameters for l in log])

    @staticmethod
    def logSamples2shapes(model: "StatisticalMeshModel", log: Sequence[jsonLogFormat]) -> np.ndarray:
        """One batched device reconstruction instead of a transformedMesh call per entry: S x N x 3."""
        return model.reconstruct(LogHelper.logSamples2thetas(log))


class PosteriorVariability:
    """apps/util/PosteriorVariability.scala:26-74. The reference takes the reconstructed meshes; here the samples stay
    parameter vectors (a log, or an S x (K+10) array) and reconstruction, normals and the per-vertex reduction run on
    the device in one call (icp_posterior_variability). `ref` is the parameter vector whose mesh carries the colour map
    (the reference passes the best sample's mesh); None = the model's reference mesh."""

    @staticmethod
    def _thetas(samples):
        if len(samples) and isinstance(samples[0], jsonLogFormat):
            return LogHelper.logSamples2thetas(samples)
        if len(samples) and isinstance(samples[0], ModelFittingParameters):
            return np.stack([t.allParameters for t in samples])
        return np.asarray(samples, float)

    @staticmethod
    def _ref(ref):
        return ref.allParameters if isinstance(ref, ModelFittingParameters) else ref

    @staticmethod
    def computeDistanceMapFromMeshesTotal(model, samples, ref=None) -> np.ndarray:
        return core.posterior_variability(model, PosteriorVariability._thetas(samples), True, None)["total_variance"]

    @staticmethod
    def computeDistanceMapFromMeshesNormal(model, samples, ref=None, sumNormals: bool = True) -> np.ndarray:
        return core.posterior_variability(model, PosteriorVariability._thetas(samples), sumNormals,
                                          None if sumNormals else PosteriorVariability._ref(ref))["normal_variance"]

    @staticmethod
    def statistics(model, samples, ref=None, sumNormals: bool = True):
        """mean, covariance, total and normal variance in one device pass."""
        return core.posterior_variability(model, PosteriorVariability._thetas(samples), sumNormals,
                                          None if sumNormals else PosteriorVariability._ref(ref))


# ---- GPMM construction from analytic kernels (apps/femur/CreateGPModel.scala) -----------------------------------------
class MatrixValuedKernel:
    """Sum of terms scale * exp(-|x - y|^2 / sigma^2) * A: what `*` and `+` build from Scalismo's GaussianKernel3D /
    DiagonalKernel3D in CreateGPModel.scala:74-80."""

    def __init__(self, terms):
        self.terms = list(terms)     # (scale, sigma, A or None)

    def __mul__(self, factor):
        if isinstance(factor, (int, float)):
            return MatrixValuedKernel([(s * float(factor), sg, a) for s, sg, a in self.terms])
        return NotImplemented

    __rmul__ = __mul__

    def __add__(self, other):
        return MatrixValuedKernel(self.terms + other.terms)

    def with_matrix(self, A):
        """baseMatrix * kernel(x, y) (CreateGPModel.scala:79)."""
        A = np.asarray(A, float)
        return MatrixValuedKernel([(s, sg, A if a is None else A @ np.asarray(a, float)) for s, sg, a in self.terms])


def GaussianKernel3D(sigma, scaleFactor=1.0):
    """Scalismo GaussianKernel3D(sigma): exp(-|x - y|^2 / sigma^2); scalar, lifted to 3 x 3 by DiagonalKernel3D or a matrix."""
    return MatrixValuedKernel([(float(scaleFactor), float(sigma), None)])


def DiagonalKernel3D(kernel: MatrixValuedKernel, outputDim=3):
    if outputDim != 3:
        raise ValueError("3-D deformation fields only")
    return kernel


def getAxisOfMainVariance(points):
    """CreateGPModel.scala:49-55: left singular vectors of the point covariance."""
    c = np.asarray(points, float) - np.asarray(points, float).mean(0)
    u, _, _ = np.linalg.svd(c.T @ c / len(c))
    return u


def femurKernel(referencePoints):
    """The kernel of CreateGPModel.scala:70-83: 10x more variance along the bone's main axis on the 90 mm scale, isotropic
    40 mm and 10 mm kernels."""
    d = getAxisOfMainVariance(referencePoints)
    baseMatrix = d @ np.diag([10.0, 1.0, 1.0]) @ d.T
    return (GaussianKernel3D(90) * 10.0).with_matrix(baseMatrix) + DiagonalKernel3D(GaussianKernel3D(40), 3) * 5.0 + \
        DiagonalKernel3D(GaussianKernel3D(10), 3) * 3.0


class FaceKernel:
    """apps/bfm/FaceKernel.scala:58-104: SpatiallyVaryingMultiscaleKernel (order-3 B-spline kernels on the levels -6..-2 with
    the scales 128, 64, 32, 10, 4, weighted by the face mask's smoothed regions) under the symmetrisation about x = 0,
    0.7 symmetric + 0.3 plain. `regionWeights(level, points) -> weights` plays FaceMask.computeSmoothedRegions (the mask is
    BFM data that is not part of the reference checkout); None = no mask."""

    levelsAndScales = ((-6, 128.0), (-5, 64.0), (-4, 32.0), (-3, 10.0), (-2, 4.0))

    def __init__(self, regionWeights=None, levelsAndScales=None, symmetricWeight=0.7, plainWeight=0.3):
        self.regionWeights = regionWeights
        if levelsAndScales is not None:
            self.levelsAndScales = tuple(levelsAndScales)
        self.symmetricWeight, self.plainWeight = symmetricWeight, plainWeight

    @property
    def levels(self):
        return [l for l, _ in self.levelsAndScales]

    @property
    def scales(self):
        return [s for _, s in self.levelsAndScales]

    def weights(self, points, mirrored=False):
        if self.regionWeights is None:
            return None
        p = np.asarray(points, float).reshape(-1, 3)
        if mirrored:
            p = p * np.array([-1.0, 1.0, 1.0])
        return np.stack([np.asarray(self.regionWeights(l, p), float) for l in self.levels])

    def matrix(self, ctx, x, y):
        return core.gpmm_face_kernel_matrix(ctx, x, y, self.levels, self.scales, self.symmetricWeight, self.plainWeight,
                                            self.weights(x), self.weights(y), self.weights(y, True))


class LowRankGaussianProcess:
    @staticmethod
    def approximateGPNystrom(ctx: core.Context, kernel, points, nystromPoints, numBasisFunctions: int):
        """Scalismo LowRankGaussianProcess.approximateGPNystrom as CreateGPModel.scala:86 calls it, every step on the device:
        kernel matrix of the Nystrom points, its leading eigenpairs (one-sided Jacobi), Nystrom extension to every model
        point. Returns (basis 3N x K, variance K) = pcaBasis / pcaVariance of the StatisticalMeshModel; eigenvector signs:
        largest-magnitude entry positive."""
        nys = np.asarray(nystromPoints, float).reshape(-1, 3)
        if isinstance(kernel, FaceKernel):
            w, v = core.gpmm_eigen_psd(ctx, kernel.matrix(ctx, nys, nys), numBasisFunctions)
            return core.gpmm_face_nystrom_extend(ctx, points, nys, kernel.levels, kernel.scales, v, w, kernel.symmetricWeight,
                                                 kernel.plainWeight, kernel.weights(points), kernel.weights(nys), kernel.weights(nys, True))
        kmm = core.gpmm_kernel_matrix(ctx, nys, nys, kernel.terms)
        w, v = core.gpmm_eigen_psd(ctx, kmm, numBasisFunctions)
        return core.gpmm_nystrom_extend(ctx, points, nys, kernel.terms, v, w)


# ---- Metropolis-Hastings -----------------------------------------------------------------------------------------
class MetropolisHastings:
    """Scalismo MetropolisHastings.next driven through the per-call API (what a Scalismo chain would do with the
    drop-in L2 classes). SamplingRegistration uses the fused device runner instead."""

    def __init__(self, generator, evaluator, rand=None):
        self.generator, self.evaluator = generator, evaluator
        self.rand = rand if rand is not None else np.random.default_rng()

    def next(self, current, logger=None):
        currentP = self.evaluator.logValue(current)
        proposal = self.generator.propose(current)
        proposalP = self.evaluator.logValue(proposal)
        t = self.generator.logTransitionRatio(current, proposal)
        a = proposalP - currentP - t
        if a > 0.0 or self.rand.random() < math.exp(a):
            if logger:
                logger.accept(current, proposal, self.generator, self.evaluator)
            return proposal
        if logger:
            logger.reject(current, proposal, self.generator, self.evaluator)
        return current

    def iterator(self, start, logger=None):
        cur = start
        while True:
            cur = self.next(cur, logger)
            yield cur


class SamplingRegistration:
    """api/sampling/SamplingRegistration.scala:36-93, on the fused device chain runner."""

    def __init__(self, model: StatisticalMeshModel, sample: TriangleMesh3D, seed=1024):
        self.model, self.sample, self.seed = model, sample, seed
        self.initialParametersZero = model.initial_parameters()
        self.variability = None   # runfitting(variability=...)

    @staticmethod
    def _device_evaluator(model, target, evaluators):
        dist_key = next((k for k in evaluators if k not in ("product", "prior")), None)
        use_prior = "prior" in evaluators
        if dist_key is None:
            return core.Evaluator(model, target, _lib.EVAL_ACCEPT_ALL, 0, use_prior), ["product", "prior", "distance"]
        p = evaluators[dist_key].dev.params
        ev = core.Evaluator(model, target, p.kind, p.mode, use_prior, p.p0, p.p1, p.p2, evaluators[dist_key].dev.ids,
                            evaluators[dist_key].dev.tp)
        return ev, ["product", "prior", dist_key]

    def runfitting(self, evaluators, generator: MixtureProposal, numOfSamples, initialModelParameters=None, jsonName=None,
                   n_chains=1, initial_batch=None, variability=None):
        """Returns the best sample (BestSampleLogger); writes the JSON chain log when jsonName is given.
        n_chains > 1 runs independent chains batched on the GPU and returns the list of per-chain best samples.
        variability: dict(takeEveryN, total=0, burnIn=0, sumNormals=True, perChain=False) - the posterior variability maps
        (PosteriorVariability.scala:30-73) of the samples LogHelper.samplesFromLog would take from the chain log, accumulated
        inside the run (icp_chain_statistics; total <= 0: no limit). They are left in self.variability: one dict pooled over
        the chains, or a list with one dict per chain (perChain), each as core.posterior_variability returns it plus n."""
        comps = generator.flatten()
        names = [c["name"] for c in comps]
        ev, keys = self._device_evaluator(self.model, self.sample, evaluators)
        chain = core.Chain(self.model, self.sample, comps, ev, max_chains=n_chains)
        if variability is not None:
            sum_normals = bool(variability.get("sumNormals", True))
            chain.set_statistics(int(variability.get("burnIn", 0)), int(variability["takeEveryN"]), int(variability.get("total", 0)),
                                 normals=sum_normals)
        if initial_batch is not None:
            th0 = np.asarray(initial_batch, float)
        else:
            th0 = np.tile((initialModelParameters or self.initialParametersZero).allParameters, (n_chains, 1))
        out = chain.run(th0, numOfSamples, seed=self.seed)
        # BestSampleLogger (SamplingRegistration.scala:58,87) tracked on the device: theta0 and the state that is current
        # after every step compete, so a retained initial state can win (icp_chain_io.theta_best / value_best)
        best = []
        for c in range(n_chains):
            same = np.nonzero((out["theta"][:, c] == out["theta_best"][c]).all(axis=1) & out["accepted"][:, c])[0]
            name = names[int(out["component"][same[0], c])] if len(same) else "Anonymous"
            best.append(ModelFittingParameters.from_vector(out["theta_best"][c], name))
        self.last_run = out
        if variability is not None:
            if variability.get("perChain", False):
                self.variability = [chain.statistics(c, sum_normals) for c in range(n_chains)]
            else:
                self.variability = chain.statistics(-1, sum_normals)
        if jsonName is not None:
            # the device log goes to the reference's file format through the library's streaming writer (icp_jsonlog_*)
            native = core.JsonLog(jsonName, self.model.K, names, keys)
            native.append(out, chain=0)
            native.close()
            self.logger = JSONAcceptRejectLogger(jsonName)
        chain.close(); ev.close()
        return best[0] if n_chains == 1 else best


# ---- deterministic ICP and metrics ------------------------------------------------------------------------------------
class IcpBasedSurfaceFitting:
    """api/other/IcpBasedSurfaceFitting.scala:29-127 (identity pose, as IcpRegistration.scala:40-43 uses it)."""

    def __init__(self, model, target, numOfSamplePoints, stepLength=1.0, projectionDirection=ModelSampling, rand=None,
                 model_point_ids=None, target_points=None):
        self.model, self.target, self.stepLength, self.projectionDirection = model, target, stepLength, projectionDirection
        self.rand = rand if rand is not None else np.random.default_rng(1024)
        # UniformMeshSampler3D(...).sample -> nearest reference vertex ids / target surface points (:51-53)
        self.ids = (self.rand.integers(0, model.N, numOfSamplePoints) if model_point_ids is None else np.asarray(model_point_ids)).astype(np.int32)
        self.tp = _decimated_points(target, numOfSamplePoints) if target_points is None else np.asarray(target_points, float)

    def _plan(self, numIterations, iterationSeq, initialCoefficients, directions):
        """(batched, theta0 (C, K + 10), directions (iters, C)) of runfitting's arguments; draws the coins from self.rand."""
        K = self.model.K
        batched = initialCoefficients is not None and np.ndim(initialCoefficients) == 2
        alpha = np.zeros((1, K)) if initialCoefficients is None else np.asarray(initialCoefficients, float).reshape(-1, K)
        n_fits = len(alpha)
        iters = len(iterationSeq) * (numIterations + 1)        # recursion runs numIterations + 1 times per sigma (:55-109)
        if self.projectionDirection == ModelAndTargetSampling:
            if directions is None:
                target = self.rand.random((iters, n_fits)) >= 0.5
            else:
                target = np.asarray(directions, dtype=object) == TargetSampling
                target = np.broadcast_to(target.reshape(iters, -1), (iters, n_fits))
        else:
            target = np.full((iters, n_fits), self.projectionDirection == TargetSampling)
        theta0 = np.stack([self.model.theta(alpha=a, center=(0, 0, 0)) for a in alpha])
        return batched, theta0, np.where(target, _lib.TARGET_SAMPLING, _lib.MODEL_SAMPLING).astype(np.int32)

    def _finish(self, batched, alpha_final):
        if batched:
            self.coefficients = alpha_final
            return [self.model.instance(a) for a in alpha_final]
        self.coefficients = alpha_final[0]
        return self.model.instance(alpha_final[0])

    def runfitting(self, numIterations, iterationSeq=(1.0, 0.1, 0.01), initialCoefficients=None, directions=None):
        """The whole loop on the device (core.StdIcp). initialCoefficients of shape (C, K) runs C independent fits and returns
        C instances (self.coefficients becomes C x K); directions is then (iterations, C) or (iterations,) for all fits. With
        ModelAndTargetSampling and no directions the coin is self.rand, drawn iteration by iteration (fit by fit) as before."""
        batched, theta0, dirs = self._plan(numIterations, iterationSeq, initialCoefficients, directions)
        runner = core.StdIcp(self.model, self.target, self.ids, self.tp, self.stepLength, _lib.MODEL_SAMPLING, len(theta0))
        try:
            out = runner.run(theta0, np.asarray(iterationSeq, float), numIterations, directions=dirs, log=False)
        finally:
            runner.close()
        return self._finish(batched, out["alpha_final"])

    @staticmethod
    def runfittings(fittings, numIterations, iterationSeq=(1.0, 0.1, 0.01), initialCoefficients=None, directions=None):
        """runfitting of several fittings of one model, typically one per target, as one device run (a core.StdIcp target
        set). initialCoefficients and directions hold one entry per fitting, each as runfitting takes it (None: runfitting's
        default for every fitting). Each fitting draws its coins from its own self.rand and gets its own coefficients, so its
        result equals its own runfitting. Returns the list of what each fitting's runfitting returns."""
        fittings = list(fittings)
        if not fittings:
            raise ValueError("runfittings needs at least one fitting")
        f0 = fittings[0]
        for g, f in enumerate(fittings[1:], 1):
            for field, same in (("model", f.model is f0.model), ("model_point_ids", np.array_equal(f.ids, f0.ids)),
                                ("stepLength", f.stepLength == f0.stepLength),
                                ("projectionDirection", f.projectionDirection == f0.projectionDirection)):
                if not same:
                    raise ValueError(f"fittings[{g}].{field} differs from fittings[0]: only the target may differ")
        inits = [None] * len(fittings) if initialCoefficients is None else list(initialCoefficients)
        dirs_in = [None] * len(fittings) if directions is None else list(directions)
        if len(inits) != len(fittings) or len(dirs_in) != len(fittings):
            raise ValueError("initialCoefficients and directions need one entry per fitting")
        plans = [f._plan(numIterations, iterationSeq, a, d) for f, a, d in zip(fittings, inits, dirs_in)]
        counts = [len(p[1]) for p in plans]
        theta0 = np.concatenate([p[1] for p in plans])
        dirs = np.concatenate([p[2] for p in plans], axis=1)
        tidx = np.repeat(np.arange(len(fittings)), counts)
        runner = core.StdIcp(f0.model, model_point_ids=f0.ids, step_length=f0.stepLength, direction=_lib.MODEL_SAMPLING,
                             max_fits=len(theta0), targets=[(f.target, f.tp) for f in fittings])
        try:
            out = runner.run(theta0, np.asarray(iterationSeq, float), numIterations, directions=dirs, log=False,
                             target_index=tidx if len(fittings) > 1 else None)
        finally:
            runner.close()
        ends = np.cumsum(counts)
        return [f._finish(p[0], out["alpha_final"][e - n:e]) for f, p, n, e in zip(fittings, plans, counts, ends)]


class RegistrationComparison:
    """api/other/RegistrationComparison.scala:22-49 for a model instance theta against the target."""

    @staticmethod
    def evaluateReconstruction2GroundTruth(id_, model, theta: ModelFittingParameters, target):
        avg, hd, _, _ = core.registration_metrics(model, target, theta.allParameters)[0]
        print(f"ID: {id_} average2surface: {avg} hausdorff: {hd}")
        return avg, hd

    @staticmethod
    def evaluateReconstruction2GroundTruthBoundaryAware(id_, model, theta: ModelFittingParameters, target):
        _, _, avg, mx = core.registration_metrics(model, target, theta.allParameters)[0]
        print(f"ID: {id_} average2surface: {avg} max: {mx}")
        return avg, mx

    @staticmethod
    def evaluateReconstructions2GroundTruth(model, thetas, targets, target_index=None, dice=False, n_samples=10000, seed=0,
                                            unit_samples=None):
        """The scoring stage of StdIcpVsChainICPrandomInitComparisonAll.scala:43-47 for many results at once: row c of thetas
        (ModelFittingParameters, or a (C, K + 10) array) against targets[target_index[c]], as one device call per measure
        (core.registration_metrics / core.dice_coefficient over the target set). Returns the (C, 4) metrics {average2surface,
        hausdorff, boundary-aware average, boundary-aware max}, and with dice=True also the (C,) Dice coefficients
        (n_samples / seed / unit_samples as core.dice_coefficient). Prints nothing."""
        th = thetas if isinstance(thetas, np.ndarray) else np.stack(
            [t.allParameters if isinstance(t, ModelFittingParameters) else np.asarray(t, float) for t in thetas])
        metrics = core.registration_metrics(model, targets, th, target_index=target_index)
        if not dice:
            return metrics
        return metrics, core.dice_coefficient(model, targets, th, unit_samples=unit_samples, n_samples=n_samples, seed=seed,
                                              target_index=target_index)
