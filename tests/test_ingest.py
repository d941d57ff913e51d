"""YAML / object / binary ingestion (pydcop_b200/ingest.py, SURVEY.md §8(f).2) against what the
UNMODIFIED reference loader produces (tests/golden/ingest_expected.json, written by
oracle/make_golden_ingest.py), on the reference's own test instances (tests/golden/instances/) and on
random problems (oracle/fuzz_ingest_vs_reference.py), from what that loader made of them."""
import glob
import itertools
import json
import os

import numpy as np
import pytest

from pydcop_b200 import ingest
from pydcop_b200.generators import random_factor_graph
from pydcop_b200.layout import layout_from_instance

HERE = os.path.dirname(os.path.abspath(__file__))
YDIR = os.path.join(HERE, "golden", "yaml")
with open(os.path.join(HERE, "golden", "ingest_expected.json")) as f:
    EXPECTED = json.load(f)


def sorted_axis_table(d, ci):
    """Table of constraint `ci` with axes permuted to sorted variable-name order."""
    a = d.arrays
    scope = a["edge_var"][a["factor_ptr"][ci]:a["factor_ptr"][ci + 1]]
    names = [d.var_names[i] for i in scope]
    shape = tuple(int(a["dom_size"][i]) for i in scope)
    t = np.asarray(a["tables"][a["table_off"][ci]:a["table_off"][ci + 1]]).reshape(shape)
    order = sorted(range(len(names)), key=lambda k: names[k])
    return [names[k] for k in order], np.transpose(t, order).reshape(-1)


def check_against(d, exp):
    assert d.name == exp["name"] and d.objective == exp["objective"]
    assert d.var_names == list(exp["variables"]) or sorted(d.var_names) == sorted(exp["variables"])
    uoff = np.concatenate([[0], np.cumsum(d.arrays["dom_size"])])
    for i, n in enumerate(d.var_names):
        ev = exp["variables"][n]
        assert d.values_of(i) == ev["domain"], n
        assert int(d.arrays["init_value"][i]) == ev["initial_value"], n
        assert d.arrays["unary"][uoff[i]:uoff[i + 1]].tolist() == ev["unary"], n  # bit-exact
    assert sorted(d.con_names) == sorted(exp["constraints"])
    for ci, n in enumerate(d.con_names):
        scope, table = sorted_axis_table(d, ci)
        assert scope == exp["constraints"][n]["scope"], n
        assert table.tolist() == exp["constraints"][n]["table"], n  # bit-exact


@pytest.mark.parametrize("case", sorted(EXPECTED))
def test_yaml_matches_reference_loader(case):
    exp = EXPECTED[case]
    d = ingest.load_yaml([os.path.join(YDIR, f) for f in exp["files"]])
    check_against(d, exp)
    # graph arrays are consistent and pack
    a = d.arrays
    assert a["var_ptr"][-1] == len(a["edge_var"])
    assert (a["edge_var"][a["var_edge"]] == np.repeat(np.arange(d.n_vars), np.diff(a["var_ptr"]))).all()
    for v in range(d.n_vars):  # incident edges in constraint order (factor_graph.py:277-280)
        s = a["var_edge"][a["var_ptr"][v]:a["var_ptr"][v + 1]]
        assert (np.diff(s) > 0).all()
    L = layout_from_instance(d.instance())
    assert L.n_vars == d.n_vars and L.n_factors == d.n_constraints


def test_vectorised_and_scalar_paths_both_used():
    d = ingest.load_yaml(os.path.join(YDIR, "mixed_grammar.yaml"))
    st = d.meta["tabulation"]
    assert st["vectorised"] >= 3 and st["scalar"] >= 3
    d2 = ingest.load_yaml([os.path.join(YDIR, "split_problem.yaml")])
    assert d2.meta["tabulation"]["shared"] == 2  # e01 / e12 / e20 are one function up to renaming


def test_tabulate_expression_falls_back_when_numpy_semantics_differ():
    doms = [list(range(6)), list(range(6))]
    cases = {
        "max(a, b)": lambda a, b: max(a, b),                    # raises on arrays
        "a if a > b else b": lambda a, b: a if a > b else b,    # raises on arrays
        "int(a / 2) + b": lambda a, b: int(a / 2) + b,          # raises on arrays
        "a * b - 3": lambda a, b: a * b - 3,                    # vectorises
        "const": lambda a, b: 7,                                # scalar result, broadcast
        "str": lambda a, b: float(len(str(a) + str(b))),        # str() of an array: wrong, caught
    }
    for name, fn in cases.items():
        stats = {}
        t = ingest.tabulate_expression(lambda a, b, fn=fn: fn(a, b), ["a", "b"], doms, stats=stats)
        want = np.array([[float(fn(x, y)) for y in doms[1]] for x in doms[0]])
        assert (t == want).all(), name
    # a silent element-wise mismatch is caught by the sampled check
    stats = {}
    fn = lambda a, b: (a + b) if isinstance(a, int) else (a + b + 1)  # noqa: E731
    t = ingest.tabulate_expression(fn, ["a", "b"], doms, stats=stats)
    assert stats == {"scalar": 1}
    assert (t == np.add.outer(np.arange(6), np.arange(6))).all()


def test_expression_scope_and_errors():
    e = ingest.Expression("abs(zeta - alpha) + source_x if False else zeta * 2")
    assert e.variable_names == ["zeta", "alpha"]  # first appearance; builtins and source* excluded
    assert e(zeta=3, alpha=1) == 6
    with pytest.raises(TypeError):
        e(zeta=1)
    with pytest.raises(TypeError):
        e(zeta=1, alpha=2, beta=3)
    with pytest.raises(SyntaxError):
        ingest.Expression("a +* b")
    body = ingest.Expression("t = a * 2\nreturn t + b")
    assert body.has_return and body.variable_names == ["a", "b"] and body(a=2, b=1) == 5
    assert ingest.Expression("a + b").canonical_key == ingest.Expression("x + y").canonical_key
    assert ingest.Expression("a - b").canonical_key != ingest.Expression("a + b").canonical_key


@pytest.mark.parametrize("text,err", [
    ("objective: min\n", "Missing name"),
    ("name: x\nobjective: best\n", "Objective"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\nvariables: {v: {domain: e}}\n",
     "unknown domain"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\n"
     "variables: {v: {domain: d, initial_value: 5}}\n", "initial value"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\nvariables: {v: {domain: d}}\n"
     "constraints: {c: {type: intention, function: v + w}}\n", "Missing variable w"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\nvariables: {v: {domain: d}}\n"
     "constraints: {c: {function: v}}\n", "type is mandatory"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\nvariables: {v: {domain: d}}\n"
     "constraints: {c: {type: extensional, variables: v, values: {3: '7'}}}\n", "not in the domain"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\nvariables: {v: {domain: d}}\n"
     "constraints: {c: {type: extensional, variables: v, values: {3: '1'}}}\n", "no default"),
    ("name: x\nobjective: min\ndomains: {d: {values: [1, 2]}}\n"
     "variables: {v: {domain: d, cost_function: v + w}}\n", "must depend on"),
])
def test_yaml_errors(text, err):
    with pytest.raises(ValueError, match=err):
        ingest.loads_yaml(text)


def test_noise_level_is_seeded_and_bounded():
    text = ("name: n\nobjective: min\ndomains: {d: {values: [0, 1, 2]}}\n"
            "variables:\n  v: {domain: d, cost_function: v * 1.0, noise_level: 0.05}\n")
    a = ingest.loads_yaml(text, seed=3).arrays["unary"]
    b = ingest.loads_yaml(text, seed=3).arrays["unary"]
    c = ingest.loads_yaml(text, seed=4).arrays["unary"]
    assert (a == b).all() and not (a == c).all()
    assert ((a - [0, 1, 2]) >= 0).all() and ((a - [0, 1, 2]) <= 0.05).all()
    u = ingest.add_noise(np.zeros(50), 0.01, seed=1)
    assert (u >= 0).all() and (u <= 0.01).all() and len(set(u.tolist())) == 50
    assert (ingest.add_noise(np.ones(4), 0.0) == 1).all()


def test_binary_container_round_trip(tmp_path):
    d = ingest.load_yaml(os.path.join(YDIR, "mixed_grammar.yaml"))
    p = tmp_path / "m.fgb"
    size = ingest.save_instance(p, d, table_dtype=np.float64)
    assert size == os.path.getsize(p)
    for mm in (True, False):
        e = ingest.load_instance(p, mmap=mm)
        assert (e.name, e.objective, e.var_names, e.con_names) == (d.name, d.objective, d.var_names, d.con_names)
        assert e.var_domain == d.var_domain and e.domain_values == d.domain_values
        for k in ingest.ARRAY_KEYS:
            assert np.array_equal(np.asarray(e.arrays[k]), d.arrays[k]), k
            assert e.arrays[k].dtype == d.arrays[k].dtype
    check_against(ingest.load_instance(p), EXPECTED["mixed_grammar"])
    # float32 tables by default, arrays on 4 KiB boundaries, names optional
    inst = random_factor_graph(500, 4, 900, 2, seed=2)
    g = ingest.from_arrays(inst, name="rnd")
    q = tmp_path / "r.fgb"
    ingest.save_instance(q, g, names=False)
    h = ingest.load_instance(q)
    assert h.arrays["tables"].dtype == np.float32 and isinstance(h.arrays["tables"], np.memmap)
    assert h.arrays["tables"].offset % 4096 == 0
    assert np.array_equal(h.arrays["tables"], inst["tables"])
    assert h.var_names[:2] == ["v0", "v1"] and h.n_constraints == 900
    La, Lb = layout_from_instance(g.instance()), layout_from_instance(h.instance())
    assert np.array_equal(La.tables, Lb.tables) and np.array_equal(La.slot_roff, Lb.slot_roff)


def test_binary_container_rejects_garbage(tmp_path):
    p = tmp_path / "bad.fgb"
    p.write_bytes(b"not a dcop file at all")
    with pytest.raises(ValueError, match="not a pydcop_b200 instance"):
        ingest.load_instance(p)
    d = ingest.from_arrays(random_factor_graph(50, 3, 60, 2, seed=1))
    q = tmp_path / "t.fgb"
    ingest.save_instance(q, d)
    data = q.read_bytes()
    q.write_bytes(data[: len(data) - 100])
    with pytest.raises(ValueError, match="truncated"):
        ingest.load_instance(q)


def test_cost_of_assignment_matches_direct_evaluation():
    d = ingest.load_yaml([os.path.join(YDIR, "split_problem.yaml")])
    rng = np.random.default_rng(0)
    exp = EXPECTED["split_problem"]
    for _ in range(20):
        idx = [int(rng.integers(0, s)) for s in d.arrays["dom_size"]]
        asg = d.assignment(idx)
        want = sum(exp["variables"][n]["unary"][idx[i]] for i, n in enumerate(d.var_names))
        for n, c in exp["constraints"].items():
            shape = [len(exp["variables"][v]["domain"]) for v in c["scope"]]
            pos = [exp["variables"][v]["domain"].index(asg[v]) for v in c["scope"]]
            want += c["table"][int(np.ravel_multi_index(pos, shape))]
        assert d.cost(idx) == pytest.approx(want, rel=1e-12)


# ---- duck-typed pyDcop objects (no reference needed) -------------------------------------------
class _Dom(list):
    def __init__(self, name, values):
        super().__init__(values)
        self.name = name


class _Var:
    def __init__(self, name, dom, initial_value=None, cost=None):
        self.name, self.domain, self.initial_value = name, dom, initial_value
        if cost is not None:
            self.cost_for_val = cost


class _FnCon:
    """Shape of NAryFunctionRelation built from a string (relations.py:1293-1307)."""

    class _F:
        def __init__(self, text):
            self.expression, self._fixed_vars, self._source_file = text, {}, None
            self._e = ingest.Expression(text)
            self.variable_names = self._e.variable_names
            self.calls = 0

        def __call__(self, **kw):
            self.calls += 1
            return self._e(**kw)

    def __init__(self, name, text, dims):
        self.name, self.dimensions, self.function = name, dims, self._F(text)

    def __call__(self, **kw):
        return self.function(**kw)


class _MatCon:
    def __init__(self, name, dims, m):
        self.name, self.dimensions, self._m = name, dims, np.asarray(m)


class _Dcop:
    def __init__(self, variables, constraints):
        self.name, self.objective = "duck", "max"
        self.variables = {v.name: v for v in variables}
        self.constraints = {c.name: c for c in constraints}


def test_from_dcop_objects():
    d4, d3 = _Dom("d4", [0, 1, 2, 3]), _Dom("d3", ["a", "b", "c"])
    x, y, z = _Var("x", d4, 2, lambda v: v * 0.5), _Var("y", d4), _Var("z", d3, "b")
    c1 = _FnCon("c1", "abs(y - x) * 3", [x, y])          # dimension order != first-appearance order
    c2 = _FnCon("c2", "abs(x - y) * 3", [y, x])
    c3 = _FnCon("c3", "1 if z == 'a' else x", [x, z])    # scalar fallback
    c4 = _MatCon("c4", [z, y], np.arange(12).reshape(3, 4))
    d = ingest.from_dcop(_Dcop([x, y, z], [c1, c2, c3, c4]))
    assert d.objective == "max" and d.var_names == ["x", "y", "z"]
    assert d.arrays["init_value"].tolist() == [2, -1, 1]
    assert d.arrays["unary"][:4].tolist() == [0.0, 0.5, 1.0, 1.5]
    a = d.arrays
    for ci, c in enumerate([c1, c2, c3]):
        doms = [list(v.domain) for v in c.dimensions]
        want = [float(c.function._e(**{v.name: val for v, val in zip(c.dimensions, combo)}))
                for combo in itertools.product(*doms)]
        assert a["tables"][a["table_off"][ci]:a["table_off"][ci + 1]].tolist() == want
    assert a["tables"][a["table_off"][3]:].tolist() == list(range(12))
    assert a["edge_var"].tolist() == [0, 1, 1, 0, 0, 2, 2, 1]
    # the expression text is used directly: the relation objects are never called
    assert c1.function.calls == 0 and c3.function.calls == 0
    with pytest.raises(ValueError):
        ingest.from_dcop(None, variables=[x])


# ---- the reference's own instances and loader --------------------------------------------------
def test_reference_test_instances_load_identically():
    """The reference's own tests/instances (copied to tests/golden/instances/) against what its loader made of
    them (tests/golden/instances_expected.npz, oracle/make_golden_ingest.py); where the reference is importable,
    also the object route against the text route."""
    import ref_shim
    files = sorted(glob.glob(os.path.join(HERE, "golden", "instances", "*.y*ml")))
    assert len(files) >= 10
    expected = np.load(os.path.join(HERE, "golden", "instances_expected.npz"))
    n = 0
    for fn in files:
        meta = json.loads(str(expected[os.path.basename(fn) + "/meta"]))
        if meta["external_variables"]:
            with pytest.raises(NotImplementedError):
                ingest.load_yaml(fn)
            continue
        d = ingest.load_yaml(fn)
        assert d.var_names == meta["var_order"] and d.con_names == meta["con_order"]
        for ci, cn in enumerate(d.con_names):
            want = expected[f"{os.path.basename(fn)}/{cn}"].tolist()
            scope, table = sorted_axis_table(d, ci)
            assert scope == meta["scopes"][cn] and table.tolist() == want, (fn, cn)
        if ref_shim.reference_available():
            # the object route gives the same arrays as the text route (up to scope order)
            ref_shim.install()
            from pydcop.dcop.yamldcop import load_dcop_from_file
            ref = load_dcop_from_file([fn])  # a bare str is iterated char by char (yamldcop.py:85)
            o = ingest.from_dcop(ref)
            for ci in range(d.n_constraints):
                assert sorted_axis_table(o, ci)[1].tolist() == sorted_axis_table(d, ci)[1].tolist()
            assert np.array_equal(o.arrays["unary"], d.arrays["unary"]) or any(
                hasattr(v, "noise_level") for v in ref.variables.values())
        n += 1
    assert n >= 10


def test_text_level_sharing_is_safe():
    """Constraints of one form share one compiled expression; string literals, placeholder-like
    names, builtins used as names and locally assigned names do not get confused."""
    text = ("name: s\nobjective: min\ndomains:\n  d: {values: [0, 1, 2]}\n  s: {values: [v1, v2, x]}\n"
            "variables:\n  v1: {domain: d}\n  v2: {domain: d}\n  v3: {domain: d}\n  _a0: {domain: d}\n"
            "  p: {domain: s}\n  q: {domain: s}\n"
            "constraints:\n"
            "  c12: {type: intention, function: 3 * v1 - v2}\n"
            "  c23: {type: intention, function: 3 * v2 - v3}\n"
            "  c31: {type: intention, function: 3 * v3 - v1}\n"
            '  lit1: {type: intention, function: "1 if p == \'v1\' else 0"}\n'
            '  lit2: {type: intention, function: "1 if q == \'v2\' else 0"}\n'
            "  ph: {type: intention, function: _a0 * 2 + v1}\n"
            "  loc:\n    type: intention\n    function: |\n      v3 = v1 * 2\n      return v3 + v2\n")
    d = ingest.loads_yaml(text)
    a = d.arrays

    def table(name):
        ci = d.con_names.index(name)
        scope = [d.var_names[i] for i in a["edge_var"][a["factor_ptr"][ci]:a["factor_ptr"][ci + 1]]]
        return scope, a["tables"][a["table_off"][ci]:a["table_off"][ci + 1]].tolist()

    want = [3.0 * x - y for x in range(3) for y in range(3)]
    assert table("c12") == (["v1", "v2"], want)
    assert table("c23") == (["v2", "v3"], want)
    assert table("c31") == (["v3", "v1"], want)
    assert table("lit1") == (["p"], [1.0, 0.0, 0.0])
    assert table("lit2") == (["q"], [0.0, 1.0, 0.0])
    assert table("ph") == (["_a0", "v1"], [2.0 * x + y for x in range(3) for y in range(3)])
    assert table("loc") == (["v1", "v2"], [2.0 * x + y for x in range(3) for y in range(3)])
    assert d.meta["tabulation"]["shared"] == 2


def test_random_expressions_tabulate_like_the_reference():
    """oracle/fuzz_ingest_vs_reference.py: 60 random YAML problems (480 intentional constraints) through
    the reference loader, assignment by assignment (stored by its `--save` as
    tests/golden/fuzz_ingest_vs_reference.npz), and through the ingestion — identical tables whichever
    of the vectorised / scalar / shared routes a constraint took."""
    import fuzz_ingest_vs_reference as F
    expected = F.load(os.path.join(HERE, "golden", "fuzz_ingest_vs_reference.npz"))
    assert sorted(expected) == list(range(60))
    total, bad, stats = 0, [], {"vectorised": 0, "scalar": 0, "shared": 0}
    for seed in range(60):
        n, b = F.compare(seed, F.problem_text(seed), expected[seed], stats)
        total, bad = total + n, bad + b
    assert total >= 400 and bad == [], bad
    assert stats["vectorised"] > 0 and stats["scalar"] > 0


@pytest.mark.parametrize("seed", [0, 1, 11, 2 ** 31 + 5, 2 ** 40 + 3, -7, 123456789012345678901234567890])
def test_vectorised_noise_stream_equals_the_stdlib_generator(seed):
    """ingest.add_noise draws the MaxSum noise (objects.py:566-567) in one vectorised call; the values are the
    ones `random.Random(seed).uniform(0, noise)` produces one at a time."""
    import random
    from pydcop_b200 import ingest
    r = random.Random(seed)
    want = np.array([r.uniform(0, 0.01) for _ in range(257)])
    got = ingest.add_noise(np.zeros(257), 0.01, seed)
    assert np.array_equal(got, want)
    base = np.linspace(0, 3, 257)
    r = random.Random(seed)
    assert np.array_equal(ingest.add_noise(base, 0.5, seed), base + np.array([r.uniform(0, 0.5) for _ in range(257)]))
