#!/usr/bin/env python
"""Random instances and parameters: the UNMODIFIED reference (lock-step, oracle/make_golden.py) against
the C oracle, cycle by cycle — extends the pinning beyond the committed fixtures.

TEST INFRASTRUCTURE.   python oracle/fuzz_vs_reference.py [n_cases] [seed] [--save FILE.npz]
Prints one JSON line: {"cases": n, "failures": [...]}.  With --save, the cases (instance arrays, parameters and
the reference's trajectories) are stored so that `check` can replay them against the oracle without the
reference (tests/golden/fuzz_vs_reference_seed*.npz).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import oracle as orc  # noqa: E402

# what `check` reads of a run: the instance as the oracle takes it and the reference's trajectories
KEYS = ("dom_size", "factor_ptr", "edge_var", "table_off", "tables", "var_ptr", "var_edge", "var_con", "unary",
        "init_value", "var_rank", "q_state", "r_state", "q_sent", "r_sent", "value", "cost")


def maxsum_case(rng):
    import make_golden as G
    n_vars = int(rng.integers(4, 14))
    doms = [int(x) for x in rng.choice([2, 3, 4, 5], size=int(rng.integers(1, 3)))]
    arities = [int(a) for a in rng.choice([1, 2, 2, 3], size=3) if a <= n_vars]
    scale = float(rng.choice([1.0, 1e-6, 1e6, 1e18]))
    vs, cs = G.random_instance(rng, n_vars, doms, int(rng.integers(3, 16)), arities,
                               int_tables=bool(rng.integers(0, 2)), with_var_costs=bool(rng.integers(0, 2)),
                               n_unary=int(rng.integers(0, 3)))
    for c in cs:
        c._m[...] = c._m * scale
    params = {"damping": float(rng.choice([0.0, 0.3, 0.5, 0.9])),
              "damping_nodes": str(rng.choice(["vars", "factors", "both", "none"])),
              "stability": float(rng.choice([0.001, 0.1, 0.5])),
              "start_messages": str(rng.choice(["leafs", "leafs_vars", "all"])), "noise": 0.0}
    mode = str(rng.choice(["min", "max"]))
    arr, meta = G.run_maxsum(vs, cs, params, mode, 10, seed=int(rng.integers(1, 1000)))
    p = {k: v for k, v in params.items() if k != "noise"}
    return {"kind": "maxsum", "params": p, "mode": mode, "scale": scale}, arr


def check_maxsum(case, arr):
    p, mode, scale = case["params"], case["mode"], case["scale"]
    o = orc.MaxSumOracle(arr, np.float64, mode=mode, **p).init()
    for k in range(11):
        if k:
            o.step()
        if not (np.array_equal(o.q, arr["q_state"][k], equal_nan=True) and np.array_equal(o.r, arr["r_state"][k], equal_nan=True)
                and np.array_equal(o.q_sent, arr["q_sent"][k]) and np.array_equal(o.r_sent, arr["r_sent"][k])):
            return f"maxsum messages differ at cycle {k}: {p} {mode} scale={scale}"
        if not np.array_equal(o.value, arr["value"][k]):
            # reported selection: ties at the ulp level are arrival-order dependent in the reference
            return None if scale != 1.0 else f"maxsum values differ at cycle {k}: {p} {mode}"
    return None


def dsa_case(rng):
    import make_golden as G
    n_vars = int(rng.integers(5, 18))
    vs, cs = G.random_instance(rng, n_vars, [int(x) for x in rng.choice([2, 3, 4], size=2)], int(rng.integers(4, 20)),
                               [int(a) for a in rng.choice([2, 2, 3], size=2) if a <= n_vars])
    for c in cs:
        c._m[...] = rng.integers(0, 3, size=c._m.shape)
    params = {"variant": str(rng.choice(["A", "B", "C"])), "probability": float(rng.choice([0.3, 0.7, 1.0])),
              "stop_cycle": int(rng.choice([0, 0, 6]))}
    mode = str(rng.choice(["min", "max"]))
    seed = int(rng.integers(1, 1000))
    arr, meta = G.run_dsa(vs, cs, params, mode, 10, seed=seed)
    return {"kind": "dsa", "params": params, "mode": mode, "seed": seed}, arr


def check_dsa(case, arr):
    params, mode = case["params"], case["mode"]
    o = orc.DsaOracle(arr, np.float64, mode=mode, seed=case["seed"], **params).init()
    for k in range(11):
        if k:
            o.step()
        if not np.array_equal(o.val, arr["value"][k]):
            return f"dsa values differ at cycle {k}: {params} {mode}"
    return None


def mgm_case(rng):
    import make_golden as G
    import make_golden_mgm as GM
    n_vars = int(rng.integers(5, 18))
    vs, cs = G.random_instance(rng, n_vars, [int(x) for x in rng.choice([2, 3, 4], size=2)], int(rng.integers(4, 20)),
                               [int(a) for a in rng.choice([1, 2, 2, 3], size=3) if a <= n_vars])
    for c in cs:
        c._m[...] = rng.integers(0, 4, size=c._m.shape)
    if rng.integers(0, 2):
        vs2 = GM.dyadic_costs(rng, vs)
        cs, vs = GM.rebuild(cs, vs2), vs2
    params = {"stop_cycle": int(rng.choice([0, 0, 7]))}
    mode = str(rng.choice(["min", "max"]))
    seed = int(rng.integers(1, 1000))
    arr, meta = GM.run_mgm(vs, cs, params, mode, 9, seed=seed)
    return {"kind": "mgm", "params": params, "mode": mode, "seed": seed}, arr


def check_mgm(case, arr):
    params, mode = case["params"], case["mode"]
    o = orc.MgmOracle(arr, np.float64, mode=mode, seed=case["seed"], **params).init()
    for k in range(10):
        if k:
            o.step()
        if not np.array_equal(o.val, arr["value"][k]):
            return f"mgm values differ at cycle {k}: {params} {mode}"
        known = ~np.isnan(arr["cost"][k])
        if not np.array_equal(o.cost[known], arr["cost"][k][known]):
            return f"mgm costs differ at cycle {k}: {params} {mode}"
    return None


CHECKS = {"maxsum": check_maxsum, "dsa": check_dsa, "mgm": check_mgm}


def check(case, arr):
    """Failure text of one case replayed through the oracle, or None."""
    return CHECKS[case["kind"]](case, arr)


def save(path, cases):
    out = {}
    for i, (case, arr) in enumerate(cases):
        out[f"{i}/case"] = np.array(json.dumps(case))
        out.update({f"{i}/{k}": np.asarray(arr[k]) for k in KEYS if k in arr})
    np.savez_compressed(path, **out)


def load(path):
    """[(case, arrays)] as `save` stored them."""
    with np.load(path) as z:
        n = sum(1 for k in z.files if k.endswith("/case"))
        return [(json.loads(str(z[f"{i}/case"])),
                 {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(f"{i}/") and not k.endswith("/case")})
                for i in range(n)]


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_path = sys.argv[sys.argv.index("--save") + 1] if "--save" in sys.argv else None
    if out_path:
        args.remove(out_path)
    n = int(args[0]) if args else 30
    rng = np.random.default_rng(int(args[1]) if len(args) > 1 else 0)
    cases, failures = [], []
    for i in range(n):
        case, arr = (maxsum_case, dsa_case, mgm_case)[i % 3](rng)
        cases.append((case, arr))
        f = check(case, arr)
        if f:
            failures.append(f"case {i}: {f}")
    if out_path:
        save(out_path, cases)
    print(json.dumps({"cases": n, "failures": failures}))


if __name__ == "__main__":
    main()
