"""Extract the structural protocols of the reference's model / acquisition boundary into a JSON fixture.

    python tests/golden/make_protocols.py TRIESTE_CHECKOUT/trieste      (writes tests/golden/reference_protocols.json)

The reference's boundary for this path is a set of Python structural protocols (SURVEY.md §8b):
trieste/models/interfaces.py:38-327 (ProbabilisticModel and its Supports*/Has* refinements) and
trieste/acquisition/interface.py:27-157 (AcquisitionFunctionBuilder & co).  TensorFlow is not installable here, so the
files are parsed with ``ast`` (never imported): for every class the fixture records its bases and, per method, the argument
names in order (without ``self``), which of them are keyword-only and which have defaults.  tests/test_protocol_conformance.py
checks the native classes against the fixture.
"""
import ast
import json
import os
import sys

FILES = {
    "models/interfaces.py": ["ProbabilisticModel", "TrainableProbabilisticModel", "SupportsPredictJoint", "SupportsPredictY",
                             "SupportsGetKernel", "SupportsGetObservationNoise", "SupportsGetInternalData",
                             "SupportsGetMeanFunction", "FastUpdateModel", "HasTrajectorySampler", "HasReparamSampler",
                             "ReparametrizationSampler", "TrajectorySampler", "TrajectoryFunctionClass"],
    "models/gpflow/interface.py": ["SupportsCovarianceBetweenPoints", "GPflowPredictor"],
    "acquisition/interface.py": ["AcquisitionFunctionClass", "AcquisitionFunctionBuilder", "SingleModelAcquisitionBuilder",
                                 "GreedyAcquisitionFunctionBuilder", "SingleModelGreedyAcquisitionBuilder",
                                 "VectorizedAcquisitionFunctionBuilder", "SingleModelVectorizedAcquisitionBuilder"],
    "acquisition/sampler.py": ["ThompsonSampler"],
}


def _base_name(b):
    if isinstance(b, ast.Subscript):
        b = b.value
    if isinstance(b, ast.Attribute):
        return b.attr
    return getattr(b, "id", None)


def extract(path, wanted):
    tree = ast.parse(open(path).read())
    out = {}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name in wanted:
            methods = {}
            for item in node.body:
                if isinstance(item, ast.FunctionDef) and (not item.name.startswith("_") or item.name in ("__call__", "__init__")):
                    if any(isinstance(d, ast.Name) and d.id == "overload" for d in item.decorator_list):
                        continue
                    a = item.args
                    pos = [x.arg for x in a.posonlyargs + a.args if x.arg != "self"]
                    n_def = len(a.defaults)
                    methods[item.name] = {
                        "args": pos,
                        "kwonly": [x.arg for x in a.kwonlyargs],
                        "with_default": pos[len(pos) - n_def:] if n_def else [],
                        "property": any(isinstance(d, ast.Name) and d.id == "property" for d in item.decorator_list),
                        "line": item.lineno,
                    }
            out[node.name] = {"bases": [b for b in map(_base_name, node.bases) if b], "methods": methods, "line": node.lineno}
    return out


def build(ref):
    fixture = {}
    for rel, wanted in FILES.items():
        fixture[rel] = extract(os.path.join(ref, rel), wanted)
    return fixture


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    fx = build(sys.argv[1])
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_protocols.json")
    json.dump(fx, open(dst, "w"), indent=1, sort_keys=True)
    print("wrote", dst, {k: sorted(v) for k, v in fx.items()}, file=sys.stderr)
