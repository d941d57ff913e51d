"""Host logic of the direct solve entry (pydcop_b200/solve.py) with the oracle standing in for the
GPU engine: parameter handling, termination, result dict, cost evaluation."""
import inspect
import itertools
import json
import os

import numpy as np
import pytest

from _oracle_engine import OracleEngine
import oracle as orc
from pydcop_b200 import ingest, solve as S
from pydcop_b200.generators import random_factor_graph

HERE = os.path.dirname(os.path.abspath(__file__))
YDIR = os.path.join(HERE, "golden", "yaml")
SPLIT = [os.path.join(YDIR, "split_problem.yaml"), os.path.join(YDIR, "split_agents.yaml")]


def brute_force(dcop):
    best = None
    sizes = [int(s) for s in dcop.arrays["dom_size"]]
    for idx in itertools.product(*(range(s) for s in sizes)):
        c = dcop.cost(idx)
        if best is None or (c > best[0] if dcop.objective == "max" else c < best[0]):
            best = (c, idx)
    return best


def test_maxsum_result_dict_and_cost():
    res = S.solve(SPLIT, "maxsum", {"stop_cycle": 30, "noise": 0}, engine_factory=OracleEngine)
    assert set(res) >= {"status", "assignment", "cost", "violation", "time", "cycle", "msg_count",
                        "msg_size"}
    assert res["status"] == "FINISHED" and res["cycle"] == 30 and res["violation"] == 0
    d = ingest.load_yaml(SPLIT)
    assert set(res["assignment"]) == set(d.var_names)
    idx = [d.values_of(i).index(res["assignment"][n]) for i, n in enumerate(d.var_names)]
    assert res["cost"] == pytest.approx(d.cost(idx), rel=1e-12)
    # same assignment as driving the oracle directly on the same arrays
    o = orc.MaxSumOracle(d.instance(), np.float64, mode="max").init().step(30)
    assert o.value.tolist() == idx
    # objective max: nothing beats the brute-force optimum; on this instance MaxSum finds it
    opt, opt_idx = brute_force(d)
    assert res["cost"] <= opt + 1e-9
    assert res["assignment"]["lonely"] == 0  # isolated variable: argmax of 2 - lonely
    json.dumps(res)  # serialisable as is


def test_dsa_is_reproducible_from_the_seed_and_respects_stop_cycle():
    kw = dict(algo="dsa_gpu", engine_factory=OracleEngine)
    a = S.solve(SPLIT, algo_params={"stop_cycle": 25, "variant": "A"}, seed=5, **kw)
    b = S.solve(SPLIT, algo_params={"stop_cycle": 25, "variant": "A"}, seed=5, **kw)
    assert a["assignment"] == b["assignment"] and a["cycle"] == 25 and a["status"] == "FINISHED"
    seen = {json.dumps(S.solve(SPLIT, algo_params={"stop_cycle": 1}, seed=s, **kw)["assignment"],
                       sort_keys=True) for s in range(6)}
    assert len(seen) > 1  # different seeds, different random starts
    assert a["assignment"]["lonely"] == 0


def test_mgm_reaches_a_one_opt_assignment():
    d = ingest.load_yaml(SPLIT)
    res = S.solve(d, "mgm", {"stop_cycle": 15}, seed=2, engine_factory=OracleEngine)
    assert res["status"] == "FINISHED" and res["cycle"] == 15 and res["algo"] == "mgm"
    idx = [d.values_of(i).index(res["assignment"][n]) for i, n in enumerate(d.var_names)]
    o = orc.MgmOracle(dict(d.instance(), var_rank=S.name_rank(d)), np.float64, mode="max",
                      stop_cycle=15, seed=2).init().step(15)
    assert o.val.tolist() == idx and o.cycle == 14
    assert S.name_rank(ingest.from_arrays(random_factor_graph(12, 2, 5, 2, seed=1))).tolist() == \
        [0, 1, 4, 5, 6, 7, 8, 9, 10, 11, 2, 3]   # v0 v1 v10 v11 v2 ... : names sort as strings


def test_timeout_ends_an_unbounded_run():
    calls = []
    res = S.solve(SPLIT, "maxsum", timeout=0.3, chunk=5, engine_factory=OracleEngine,
                  on_cycle=lambda c, v: calls.append((c, v.copy())))
    assert res["status"] == "TIMEOUT" and res["cycle"] >= 5 and res["cycle"] % 5 == 0
    assert [c for c, _ in calls] == list(range(5, res["cycle"] + 1, 5))
    with pytest.raises(ValueError, match="does not stop by itself"):
        S.solve(SPLIT, "maxsum", engine_factory=OracleEngine)


@pytest.mark.parametrize("params,err", [
    ({"dampin": 0.3}, "Unknown parameter"),
    ({"damping": "high"}, "Invalid value for parameter damping"),
    ({"damping_nodes": "some"}, "Invalid value for parameter damping_nodes"),
    ({"start_messages": "none"}, "Invalid value"),
])
def test_parameter_validation(params, err):
    with pytest.raises(ValueError, match=err):
        S.solve(SPLIT, "maxsum", dict(params, stop_cycle=1), engine_factory=OracleEngine)
    with pytest.raises(ValueError, match="unknown algorithm"):
        S.solve(SPLIT, "dpop", {"stop_cycle": 1}, engine_factory=OracleEngine)
    p = S.check_params("dsa", {"stop_cycle": "12", "probability": "0.5"})
    assert p["stop_cycle"] == 12 and p["probability"] == 0.5 and p["variant"] == "B"


def test_reference_defaults_are_mirrored():
    """Same names and defaults as the reference modules' algo_params (tests/golden/algo_params.json, written
    from the reference by oracle/make_golden_algo_params.py)."""
    with open(os.path.join(HERE, "golden", "algo_params.json")) as f:
        golden = json.load(f)
    for name, mine in (("maxsum", S.MAXSUM_DEFAULTS), ("dsa", S.DSA_DEFAULTS), ("mgm", S.MGM_DEFAULTS)):
        ref = golden[name]
        # stop_cycle on MaxSum is this package's extension (also on the maxsum_gpu plugin module)
        assert set(ref) == set(mine) - ({"stop_cycle"} if name == "maxsum" else set())
        for k, p in ref.items():
            assert mine[k] == p["default"], (name, k)
            if p["values"]:
                assert tuple(p["values"]) == S._CHOICES[k]


def test_every_input_form_loads(tmp_path):
    d = ingest.load_yaml(SPLIT)
    p = tmp_path / "s.fgb"
    ingest.save_instance(p, d, table_dtype=np.float64)
    kw = dict(algo="maxsum", algo_params={"stop_cycle": 10, "noise": 0}, engine_factory=OracleEngine)
    want = S.solve(d, **kw)["assignment"]
    assert S.solve(str(p), **kw)["assignment"] == want          # binary container, by magic
    assert S.solve(SPLIT[0], **kw)["assignment"] == want        # single YAML path
    inst = random_factor_graph(40, 3, 60, 2, seed=3)
    r = S.solve(inst, **kw)                                     # raw arrays
    assert sorted(r["assignment"]) == sorted(f"v{i}" for i in range(40))
    with pytest.raises(TypeError):
        S.load(42)


def test_infinity_counts_as_violation():
    text = ("name: hard\nobjective: min\ndomains: {d: {values: [0, 1]}}\n"
            "variables: {a: {domain: d}, b: {domain: d}}\n"
            "constraints:\n  ne: {type: intention, function: 10000 if a == b else 0}\n"
            "  pa: {type: intention, function: 10000 if a == 0 else 1}\n")
    d = ingest.loads_yaml(text)
    assert S.solution_cost(d, [0, 0], infinity=10000) == (2, 0.0)
    assert S.solution_cost(d, [1, 0], infinity=10000) == (0, 1.0)
    assert S.solution_cost(d, [0, 0]) == (0, 20000.0)         # `pydcop solve` default: -i inf
    assert S.solution_cost(d, [1, 1], infinity=10000) == (1, 1.0)
    assert S.solution_cost(d, [0, 0], infinity=float("inf")) == (0, 20000.0)


def test_engine_construction_arguments_exist():
    """_default_engine cannot run here (no GPU); at least bind its keyword arguments against the
    engines' signatures so a renamed parameter fails on CPU."""
    import ast
    from pydcop_b200 import engine as E
    tree = ast.parse(inspect.getsource(S._default_engine))
    calls = {n.func.id: n for n in ast.walk(tree)
             if isinstance(n, ast.Call) and isinstance(n.func, ast.Name)}
    for cls in (E.MaxSumEngine, E.DsaEngine, E.MgmEngine):
        names = {k.arg for k in calls[cls.__name__].keywords}
        sig = set(inspect.signature(cls.__init__).parameters)
        assert names and names <= sig, (cls.__name__, names - sig)
        assert len(calls[cls.__name__].args) == 1  # the layout


def test_cli_prints_json(tmp_path, capsys, monkeypatch):
    monkeypatch.setattr(S, "_default_engine",
                        lambda kind, layout, dcop, params, mode, precision, device, seed:
                        OracleEngine(kind, layout, dcop.instance(), dict(params, mode=mode, seed=seed or 0)))
    out = tmp_path / "i.fgb"
    rc = S.main(["-a", "dsa", "-p", "stop_cycle:5", "-p", "variant:C", "--seed", "1",
                 "--save", str(out), *SPLIT])
    assert rc == 0
    res = json.loads(capsys.readouterr().out)
    assert res["cycle"] == 5 and res["algo"] == "dsa" and len(res["assignment"]) == 6
    assert ingest.load_instance(out).n_vars == 6
    # per-cycle metrics in the reference's CSV columns
    csvf = tmp_path / "run.csv"
    rc = S.main(["-a", "maxsum", "-p", "stop_cycle:12", "-p", "noise:0", "--run_metrics", str(csvf),
                 "--metrics_every", "4", *SPLIT])
    assert rc == 0
    final = json.loads(capsys.readouterr().out)
    lines = csvf.read_text().strip().splitlines()
    assert lines[0] == "cycle,time,cost,violation,msg_count,msg_size,status"
    assert [int(ln.split(",")[0]) for ln in lines[1:]] == [4, 8, 12, 12]
    assert lines[-1].endswith("FINISHED") and float(lines[-1].split(",")[2]) == final["cost"]


def test_reference_cli_known_answers():
    """The end-to-end known answers of the reference's CLI tests (tests/dcop_cli/test_solve.py:41-48,
    102-108): graph_coloring1.yaml -> {v1: R, v2: G, v3: R}, secp_simple1.yaml -> {l1: 0, l2: 3, l3: 4,
    m1: 3}, through the direct entry (ingestion of the reference's own YAML files, copied to tests/golden/instances/,
    + MaxSum)."""
    inst_dir = os.path.join(HERE, "golden", "instances")
    r = S.solve(os.path.join(inst_dir, "graph_coloring1.yaml"), "maxsum", {"stop_cycle": 30}, seed=1,
                engine_factory=OracleEngine)
    assert r["assignment"] == {"v1": "R", "v2": "G", "v3": "R"} and r["violation"] == 0
    r = S.solve(os.path.join(inst_dir, "secp_simple1.yaml"), "maxsum", {"stop_cycle": 30}, seed=1,
                engine_factory=OracleEngine)
    assert r["assignment"] == {"l1": 0, "l2": 3, "l3": 4, "m1": 3}
    # the committed trajectory of the same instance ends in the same assignment
    inst, meta = orc.load_golden(os.path.join(HERE, "golden", "ms_secp_simple1.npz"))
    names = [str(n) for n in inst["var_names"]]
    assert dict(zip(names, inst["value"][-1].tolist())) == {"l1": 0, "l2": 3, "l3": 4, "m1": 3}


def test_host_solution_cost_equals_the_references_known_answers():
    """tests/golden/solution_cost.json holds (violations, cost) computed by the UNMODIFIED reference
    (oracle/make_golden_cost.py; constraint tables and variable costs with entries equal to `infinity`):
    the host evaluation used through the engine seam reproduces them; the device reduction is checked
    against the same file in tests/test_gpu_solve.py."""
    import json
    from pydcop_b200 import ingest
    for prob in json.load(open(os.path.join(os.path.dirname(__file__), "golden", "solution_cost.json"))):
        d = ingest.from_arrays({k: np.asarray(prob[k]) for k in ("dom_size", "factor_ptr", "edge_var", "tables", "unary")})
        for case in prob["cases"]:
            viol, cost = S.solution_cost(d, case["value_index"], prob["infinity"])
            assert viol == case["violation"], prob["name"]
            assert cost == pytest.approx(case["cost"], rel=1e-12, abs=1e-12), prob["name"]
