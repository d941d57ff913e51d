"""Names, defaults and allowed values of the UNMODIFIED reference's algorithm parameters
(`algo_params` of pydcop/algorithms/{maxsum,dsa,mgm}.py).  TEST INFRASTRUCTURE ONLY; needs the reference:

    python oracle/make_golden_algo_params.py

Output: tests/golden/algo_params.json, {algorithm: {parameter: {"default": ..., "values": [...] or null}}}.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)


def main():
    import ref_shim
    ref_shim.install()
    from pydcop.algorithms import load_algorithm_module
    out = {name: {p.name: {"default": p.default_value, "values": list(p.values) if p.values else None}
                  for p in load_algorithm_module(name).algo_params}
           for name in ("maxsum", "dsa", "mgm")}
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "algo_params.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote", path)


if __name__ == "__main__":
    main()
