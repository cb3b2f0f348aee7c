"""The drop-in boundary (SURVEY.md 8b): every hot-path name keeps the reference's signature.

`tests/golden/reference_signatures.json` holds the reference's side: the parameters of each boundary function and the
fields of each boundary dataclass of jstmn/cppflow (regenerated from a checkout of it by
tests/golden/make_golden_signatures.py).  `inspect.signature` of the repo's functions is compared with it: the
reference's parameters must come first, in the same order, with the same names and defaults; anything the repo adds
(e.g. `mesh_validator=`, `native=`) must be optional.  Dataclasses of the boundary must have the reference's fields in
the reference's order."""
import dataclasses
import importlib
import inspect
import json
import numbers
import os

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden", "reference_signatures.json")

FUNCTIONS = [  # (module, qualified name)
    ("search", "dp_search"), ("search", "joint_limit_almost_violations_3d"),
    ("collision_detection", "qpaths_batched_env_collisions"), ("collision_detection", "qpaths_batched_self_collisions"),
    ("collision_detection", "get_only_non_colliding_qpaths"),
    ("optimization", "run_lm_optimization"), ("optimization", "run_lm_alternating_loss"),
    ("optimization", "levenberg_marquardt_only_pose"), ("optimization", "levenberg_marquardt_full"),
    ("optimization_utils", "LmResidualFns.get_r_and_J"), ("optimization_utils", "get_6d_pose_errors"),
    ("optimization_utils", "clamp_to_joint_limits"), ("optimization_utils", "x_is_valid"),
    ("evaluation_utils", "angular_changes"), ("evaluation_utils", "errors_are_below_threshold"),
    ("data_type_utils", "problem_from_filename"),
]
DATACLASSES = [
    ("optimization", "OptimizationProblem"), ("optimization", "OptimizationState"), ("optimization", "OptimizationResult"),
    ("lm_hyper_parameters", "OptimizationParameters"), ("data_types", "Constraints"), ("data_types", "Problem"),
    ("data_types", "PlannerSettings"), ("data_types", "TimingData"),
]


def resolve(mod, qual):
    obj = importlib.import_module(mod)
    for part in qual.split("."):
        obj = getattr(obj, part)
    return obj


def describe_params(fn):
    """[name, kind, has default, repr of the default, the default as a number (numeric defaults only)] per parameter;
    numeric defaults compare by value, so that a numpy scalar and a float of the same value agree whatever their repr."""
    out = []
    for p in inspect.signature(fn).parameters.values():
        has = p.default is not inspect.Parameter.empty
        num = float(p.default) if has and isinstance(p.default, numbers.Real) and not isinstance(p.default, bool) else None
        out.append([p.name, str(p.kind), has, repr(p.default) if has else None, num])
    return out


def _same_default(r, o):
    if r[4] is not None and o[4] is not None:
        return r[4] == o[4]
    return r[3] == o[3]


@pytest.fixture(scope="module")
def signatures():
    with open(GOLDEN) as f:
        ref = json.load(f)
    assert sorted(ref["functions"]) == sorted(f"{m}.{q}" for m, q in FUNCTIONS)
    assert sorted(ref["dataclasses"]) == sorted(f"{m}.{q}" for m, q in DATACLASSES)
    res = {"functions": {}, "dataclasses": {}}
    for mod, qual in FUNCTIONS:
        name = f"{mod}.{qual}"
        res["functions"][name] = [ref["functions"][name]["params"], describe_params(resolve("cppflow_b200." + mod, qual))]
    for mod, qual in DATACLASSES:
        name = f"{mod}.{qual}"
        ours = [f.name for f in dataclasses.fields(resolve("cppflow_b200." + mod, qual))]
        res["dataclasses"][name] = [ref["dataclasses"][name]["fields"], ours]
    return res


def test_function_signatures_keep_the_reference_prefix(signatures):
    problems = []
    for name, (ref, ours) in signatures["functions"].items():
        if len(ours) < len(ref):
            problems.append(f"{name}: {len(ours)} parameters, the reference has {len(ref)}")
            continue
        for i, (r, o) in enumerate(zip(ref, ours)):
            if r[0] != o[0]:
                problems.append(f"{name}: parameter {i} is '{o[0]}', the reference calls it '{r[0]}'")
            elif r[2] != o[2] and r[2]:
                problems.append(f"{name}: '{r[0]}' has a default in the reference, none here")
            elif r[2] and o[2] and not _same_default(r, o):
                problems.append(f"{name}: default of '{r[0]}' is {o[3]}, the reference has {r[3]}")
        for o in ours[len(ref):]:
            if not o[2] and "VAR_" not in o[1]:
                problems.append(f"{name}: extra parameter '{o[0]}' has no default")
    assert not problems, "\n".join(problems)


def test_dataclass_fields_keep_the_reference_order(signatures):
    problems = []
    for name, (ref, ours) in signatures["dataclasses"].items():
        if ours[: len(ref)] != ref:
            problems.append(f"{name}: fields {ours}, the reference has {ref}")
    assert not problems, "\n".join(problems)
