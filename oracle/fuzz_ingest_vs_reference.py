#!/usr/bin/env python
"""Random pyDcop YAML problems with random intentional constraints (arithmetic, abs, round, max, //, %,
**, comparisons, conditional expressions over int / float / range domains): the tables pydcop_b200.ingest
produces against the UNMODIFIED reference loader evaluated assignment by assignment.

TEST INFRASTRUCTURE.   python oracle/fuzz_ingest_vs_reference.py [n_files] [--save FILE.npz]
Last line: "constraints compared N bad B {tabulation statistics}".  With --save, what the reference made of every
problem is stored so that `compare` can replay it without the reference (tests/golden/fuzz_ingest_vs_reference.npz).
"""
import itertools
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), HERE]
import numpy as np  # noqa: E402
from pydcop_b200 import ingest  # noqa: E402


def rand_expr(rnd, names, depth=0):
    if depth > 2 or rnd.random() < 0.3:
        return rnd.choice(names + [str(rnd.choice([0, 1, 2, 3, 0.5, -1.5, 7]))])
    k = rnd.random()
    a, b = rand_expr(rnd, names, depth+1), rand_expr(rnd, names, depth+1)
    if k < 0.45: return f"({a} {rnd.choice(['+','-','*'])} {b})"
    if k < 0.55: return f"abs({a})"
    if k < 0.65: return f"({a} if {b} {rnd.choice(['==','<','>=','!='])} {rand_expr(rnd,names,depth+1)} else {rand_expr(rnd,names,depth+1)})"
    if k < 0.72: return f"round({a})"
    if k < 0.79: return f"max({a}, {b})"
    if k < 0.86: return f"({a} // 2)"
    if k < 0.93: return f"({a} % 3)"
    return f"({a} ** 2)"


def problem_text(seed):
    rnd = random.Random(seed)
    doms = {"di": [-2, -1, 0, 1, 2, 3], "df": [0.5, 1.25, -2.0, 3.0], "dr": ["0..4"]}
    lines = ["name: fuzz", "objective: min", "domains:"]
    for d, v in doms.items():
        lines.append(f"  {d}: {{values: {v}}}")
    lines.append("variables:")
    names = [f"v{i}" for i in range(5)]
    for n in names:
        lines.append(f"  {n}: {{domain: {rnd.choice(list(doms))}}}")
    lines.append("constraints:")
    for c in range(8):
        sub = rnd.sample(names, rnd.randint(1, 3))
        expr = rand_expr(rnd, sub)
        lines.append(f"  c{c}: {{type: intention, function: \"{expr}\"}}")
    var_dom = {n: None for n in names}
    for ln in lines:
        for n in names:
            if ln.startswith(f"  {n}: {{domain: "):
                var_dom[n] = ln.split("domain: ")[1].rstrip("}")
    real = {"di": doms["di"], "df": doms["df"], "dr": [0, 1, 2, 3, 4]}
    for c in range(3):      # extensional constraints: cost -> "a b | c d", some cells left to `default`
        sub = rnd.sample(names, rnd.randint(1, 2))
        cells = list(itertools.product(*[real[var_dom[n]] for n in sub]))
        by_cost = {}
        for cell in cells:
            if rnd.random() < 0.8:
                by_cost.setdefault(rnd.choice([0, 1, 2.5, -3, 10]), []).append(" ".join(str(x) for x in cell))
        lines.append(f"  e{c}:")
        lines.append("    type: extensional")
        lines.append(f"    variables: {sub[0] if len(sub) == 1 and rnd.random() < 0.5 else '[' + ', '.join(sub) + ']'}")
        lines.append(f"    default: {rnd.choice([0, 7, -1.5])}")
        lines.append("    values:")
        for cost, asg in by_cost.items():
            lines.append(f"      {cost}: \"{' | '.join(asg)}\"")
        if not by_cost:
            lines[-1] = "    values: {}"
    return "\n".join(lines) + "\n"


def reference_tables(text):
    """What the reference makes of `text`: None when its loader rejects it, else {"evaluates": bool, "tables":
    {constraint: (scope in sorted name order, table over that scope)}}; "evaluates" is False when evaluating some
    constraint on some assignment raises."""
    from pydcop.dcop.yamldcop import load_dcop
    try:
        ref = load_dcop(text)
    except Exception:
        return None
    tables = {}
    try:
        for cn, c in ref.constraints.items():
            dims = sorted(c.dimensions, key=lambda v: v.name)
            tables[cn] = ([v.name for v in dims],
                          [float(c(**{v.name: x for v, x in zip(dims, combo)}))
                           for combo in itertools.product(*[list(v.domain) for v in dims])])
    except Exception:
        return {"evaluates": False, "tables": {}}
    return {"evaluates": True, "tables": tables}


def compare(seed, text, expected, stats):
    """(constraints compared, failure texts) of ingest.loads_yaml(text) against `expected` (reference_tables)."""
    if expected is None:
        return 0, []
    try:
        mine = ingest.loads_yaml(text)
    except Exception as e:
        # acceptable only if the reference also fails when evaluating
        return 0, ([] if not expected["evaluates"] else [f"MINE FAILED but reference evaluates: {seed} {e!r}"])
    if not expected["evaluates"]:
        return 0, [f"reference fails to evaluate, mine loads: {seed}"]
    for k in stats:
        stats[k] += mine.meta["tabulation"][k]
    a, total, bad = mine.arrays, 0, []
    for ci, cn in enumerate(mine.con_names):
        want_scope, want = expected["tables"][cn]
        scope = [mine.var_names[i] for i in a["edge_var"][a["factor_ptr"][ci]:a["factor_ptr"][ci + 1]]]
        if sorted(scope) != want_scope:
            bad.append(f"SCOPE {seed} {cn} {scope} {want_scope}")
            continue
        shape = tuple(len(mine.values_of(n)) for n in scope)
        order = sorted(range(len(scope)), key=lambda k: scope[k])
        t = np.transpose(np.asarray(a["tables"][a["table_off"][ci]:a["table_off"][ci + 1]]).reshape(shape), order)
        total += 1
        if not np.array_equal(t.reshape(-1), np.array(want), equal_nan=True):
            bad.append(f"TABLE {seed} {cn} {t.reshape(-1)[:5]} {want[:5]}")
    return total, bad


def save(path, expected):
    out = {}
    for seed, exp in expected.items():
        out[f"{seed}/meta"] = np.array(json.dumps(None if exp is None else
                                                  {"evaluates": exp["evaluates"],
                                                   "scopes": {cn: s for cn, (s, _) in exp["tables"].items()}}))
        out.update({f"{seed}/{cn}": np.array(t, np.float64) for cn, (_, t) in (exp or {"tables": {}})["tables"].items()})
    np.savez_compressed(path, **out)


def load(path):
    """{seed: reference_tables(problem_text(seed))} as `save` stored it."""
    out = {}
    with np.load(path) as z:
        for k in z.files:
            if k.endswith("/meta"):
                seed = int(k.split("/")[0])
                meta = json.loads(str(z[k]))
                out[seed] = None if meta is None else {
                    "evaluates": meta["evaluates"],
                    "tables": {cn: (s, z[f"{seed}/{cn}"].tolist()) for cn, s in meta["scopes"].items()}}
    return out


def main():
    import logging
    import ref_shim
    ref_shim.install()
    logging.disable(logging.CRITICAL)
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_path = sys.argv[sys.argv.index("--save") + 1] if "--save" in sys.argv else None
    if out_path:
        args.remove(out_path)
    total, bad, stats, expected = 0, [], {"vectorised": 0, "scalar": 0, "shared": 0}, {}
    for seed in range(int(args[0]) if args else 40):
        text = problem_text(seed)
        expected[seed] = reference_tables(text)
        n, b = compare(seed, text, expected[seed], stats)
        total, bad = total + n, bad + b
    for line in bad:
        print(line)
    if out_path:
        save(out_path, expected)
    print("constraints compared", total, "bad", len(bad), stats)


if __name__ == "__main__":
    main()
