"""Expected arrays for the YAML ingestion tests, produced by the UNMODIFIED reference loader.

TEST INFRASTRUCTURE ONLY.  Runs in the build container (needs /root/reference):

    python oracle/make_golden_ingest.py

For every YAML case under tests/golden/yaml/ it calls the reference's own
`load_dcop_from_file` (pydcop/dcop/yamldcop.py:62-122), then evaluates every constraint on every
assignment through the reference's relation objects (`constraint(**assignment)`,
pydcop/dcop/relations.py:598-617,803-828) and every variable cost through `cost_for_val`
(pydcop/dcop/objects.py:498-503).  Tables are written with their axes in SORTED variable-name
order, because the reference's own axis order for intentional constraints is a Python set order
(pydcop/utils/expressionfunction.py:74,220).  Output: tests/golden/ingest_expected.json.
"""
import itertools
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)

CASES = {
    "mixed_grammar": ["mixed_grammar.yaml"],
    "split_problem": ["split_problem.yaml", "split_agents.yaml"],
}


def describe(dcop):
    out = {"name": dcop.name, "objective": dcop.objective, "variables": {}, "constraints": {}}
    for name, v in dcop.variables.items():
        dom = list(v.domain)
        cost = getattr(v, "cost_for_val", None)
        out["variables"][name] = {
            "domain": dom,
            "initial_value": (dom.index(v.initial_value) if v.initial_value is not None else -1),
            "unary": [float(cost(x)) if cost else 0.0 for x in dom],
        }
    for name, c in dcop.constraints.items():
        dims = sorted(c.dimensions, key=lambda v: v.name)
        doms = [list(v.domain) for v in dims]
        table = [float(c(**{v.name: x for v, x in zip(dims, combo)}))
                 for combo in itertools.product(*doms)]
        out["constraints"][name] = {"scope": [v.name for v in dims], "table": table}
    return out


def main():
    import ref_shim
    ref_shim.install()
    from pydcop.dcop.yamldcop import load_dcop_from_file
    ydir = os.path.join(ROOT, "tests", "golden", "yaml")
    expected = {}
    for case, files in CASES.items():
        dcop = load_dcop_from_file([os.path.join(ydir, f) for f in files])
        expected[case] = dict(describe(dcop), files=files)
    path = os.path.join(ROOT, "tests", "golden", "ingest_expected.json")
    with open(path, "w") as f:
        json.dump(expected, f, indent=1, sort_keys=True)
    print("wrote", path, {k: (len(v["variables"]), len(v["constraints"])) for k, v in expected.items()})
    # the reference's own test instances (its tests/instances/, copied to tests/golden/instances/): per file
    # "<file>/meta" (JSON: external variables or not, declaration order of variables and constraints, sorted
    # scopes) and "<file>/<constraint>" (the table, axes in sorted variable-name order)
    import numpy as np
    idir = os.path.join(ROOT, "tests", "golden", "instances")
    out = {}
    for fn in sorted(f for f in os.listdir(idir) if f.endswith((".yaml", ".yml"))):
        dcop = load_dcop_from_file([os.path.join(idir, fn)])
        meta = {"external_variables": bool(dcop.external_variables)}
        if not dcop.external_variables:
            d = describe(dcop)
            meta.update(var_order=list(dcop.variables), con_order=list(dcop.constraints),
                        scopes={n: c["scope"] for n, c in d["constraints"].items()})
            out.update({f"{fn}/{n}": np.array(c["table"]) for n, c in d["constraints"].items()})
        out[f"{fn}/meta"] = np.array(json.dumps(meta))
    path = os.path.join(ROOT, "tests", "golden", "instances_expected.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main()
