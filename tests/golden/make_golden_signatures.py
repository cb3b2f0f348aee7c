"""Regenerate tests/golden/reference_signatures.json from a checkout of the reference (jstmn/cppflow).

    CPPFLOW_REFERENCE_DIR=<checkout> python tests/golden/make_golden_signatures.py

The reference package is imported with the stubs of make_golden.py (jrl / klampt / ikflow / matplotlib are not
installable offline) and the parameters of each boundary function and the fields of each boundary dataclass that
tests/test_boundary_signatures.py checks are written.  Nothing outside the repository is read at test time.
"""
import dataclasses
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)

from tests.test_boundary_signatures import DATACLASSES, FUNCTIONS, GOLDEN, describe_params, resolve  # noqa: E402


def main():
    reference = os.environ.get("CPPFLOW_REFERENCE_DIR", "")
    if not os.path.isdir(os.path.join(reference, "cppflow")):
        sys.exit("set CPPFLOW_REFERENCE_DIR to a checkout of the reference cppflow (the directory holding cppflow/)")
    import make_golden as MG

    MG.install_stubs()
    sys.path.insert(0, os.path.abspath(reference))
    import cppflow  # noqa: F401  (the real reference package)

    out = {"source": "imported from a checkout of the reference by make_golden_signatures.py",
           "functions": {}, "dataclasses": {}}
    for mod, qual in FUNCTIONS:
        out["functions"][f"{mod}.{qual}"] = {"params": describe_params(resolve("cppflow." + mod, qual)),
                                            "evidence": "imported"}
    for mod, qual in DATACLASSES:
        fields = [f.name for f in dataclasses.fields(resolve("cppflow." + mod, qual))]
        out["dataclasses"][f"{mod}.{qual}"] = {"fields": fields, "evidence": "imported"}
    with open(GOLDEN, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", GOLDEN)


if __name__ == "__main__":
    main()
