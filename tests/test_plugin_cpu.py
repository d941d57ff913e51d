"""The pyDcop drop-in boundary, exercised with the UNMODIFIED reference in thread mode (the copy in
oracle/_ref/, see oracle/install_reference.py).  There is no GPU here, so the end-to-end runs put the CPU
oracle behind the session's engine seam — that checks the plugin plumbing (registration, closure
detection, value reporting, cycle counting, FINISHED status), not the kernels; without the seam
the product path must fail loudly instead of falling back."""
import os
import time

import numpy as np
import pytest

import oracle as orc
import ref_shim

pytestmark = pytest.mark.skipif(not ref_shim.reference_available(),
                                reason="no reference: oracle/_ref/ not installed")

INSTANCES = os.path.join(ref_shim.REFERENCE_ROOT, "tests", "instances")


def retry_once(fn):
    """The end-to-end tests below run the reference's real agent threads, orchestrator timers and
    0.02 s polling; on a loaded build machine one of them occasionally misses a wall-clock window.
    They assert deterministic RESULTS, so a single re-run on failure is safe and keeps `-x` usable."""
    import functools

    @functools.wraps(fn)
    def wrapper(*a, **k):
        try:
            return fn(*a, **k)
        except AssertionError:
            from pydcop_b200.algorithms._session import GpuSession
            GpuSession.reset()
            time.sleep(1.0)
            return fn(*a, **k)
    return wrapper


@pytest.fixture(scope="module")
def pydcop_ready():
    ref_shim.install()
    import logging
    logging.disable(logging.CRITICAL)
    from pydcop_b200 import launcher
    launcher.install()
    yield
    logging.disable(logging.NOTSET)


from _oracle_engine import OracleEngine as _OracleEngine  # noqa: E402


@pytest.fixture
def oracle_seam(pydcop_ready):
    from pydcop_b200.algorithms._session import GpuSession
    GpuSession.reset()
    GpuSession.engine_factory = _OracleEngine
    yield GpuSession
    GpuSession.engine_factory = None
    GpuSession.reset()


def test_modules_are_discovered_and_loaded(pydcop_ready):
    from pydcop.algorithms import list_available_algorithms, load_algorithm_module
    names = list_available_algorithms()
    assert "maxsum_gpu" in names and "dsa_gpu" in names and "maxsum" in names
    ref, gpu = load_algorithm_module("maxsum"), load_algorithm_module("maxsum_gpu")
    assert gpu.GRAPH_TYPE == ref.GRAPH_TYPE == "factor_graph"
    ref_params = {p.name: p for p in ref.algo_params}
    gpu_params = {p.name: p for p in gpu.algo_params}
    for n, p in ref_params.items():   # every reference parameter, same type / values / default
        assert gpu_params[n] == p
    assert {"stop_cycle", "precision", "seed", "session"} <= set(gpu_params)
    refd, gpud = load_algorithm_module("dsa"), load_algorithm_module("dsa_gpu")
    assert gpud.GRAPH_TYPE == refd.GRAPH_TYPE == "constraints_hypergraph"
    for p in refd.algo_params:
        assert {q.name: q for q in gpud.algo_params}[p.name] == p
    refm, gpum = load_algorithm_module("mgm"), load_algorithm_module("mgm_gpu")
    assert "mgm_gpu" in names and gpum.GRAPH_TYPE == refm.GRAPH_TYPE == "constraints_hypergraph"
    for p in refm.algo_params:
        assert {q.name: q for q in gpum.algo_params}[p.name] == p


def test_memory_and_load_models_match_reference(pydcop_ready):
    from pydcop.algorithms import load_algorithm_module
    from pydcop.computations_graph import constraints_hypergraph, factor_graph
    from pydcop.dcop.yamldcop import load_dcop_from_file
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "secp_simple1.yaml")])
    fg = factor_graph.build_computation_graph(dcop)
    ref, gpu = load_algorithm_module("maxsum"), load_algorithm_module("maxsum_gpu")
    for node in fg.nodes:
        assert gpu.computation_memory(node) == ref.computation_memory(node)
        for nb in node.neighbors:
            assert gpu.communication_load(node, nb) == ref.communication_load(node, nb)
    hg = constraints_hypergraph.build_computation_graph(dcop)
    refd, gpud = load_algorithm_module("dsa"), load_algorithm_module("dsa_gpu")
    refm, gpum = load_algorithm_module("mgm"), load_algorithm_module("mgm_gpu")
    for node in hg.nodes:
        assert gpud.computation_memory(node) == refd.computation_memory(node)
        assert gpum.computation_memory(node) == refm.computation_memory(node)
        for nb in node.neighbors:
            assert gpud.communication_load(node, nb) == refd.communication_load(node, nb)
            assert gpum.communication_load(node, nb) == refm.communication_load(node, nb)


@retry_once
def test_solve_api_maxsum_gpu_known_answer(oracle_seam):
    """tests/api/test_api_solve.py:35-60 of the reference, with --algo maxsum_gpu."""
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    from pydcop.algorithms import AlgorithmDef
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    # stop_cycle fixes the number of cycles, so the answer does not depend on how many cycles fit
    # in the wall-clock budget (the reference's solve() always waits for its timeout, run.py:130-133)
    algo = AlgorithmDef.build_with_default_param("maxsum_gpu", {"stop_cycle": 40}, mode=dcop.objective)
    assignment = solve(dcop, algo, "adhoc", timeout=8)
    assert assignment == {"v1": "R", "v2": "G", "v3": "R"}


def _run_gc10_with_stop_cycle():
    from pydcop.algorithms import AlgorithmDef, load_algorithm_module
    from pydcop.computations_graph import factor_graph
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.distribution import adhoc
    from pydcop.infrastructure.run import run_local_thread_dcop
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring_10_4_15_0.1.yml")])
    algo_module = load_algorithm_module("maxsum_gpu")
    algo = AlgorithmDef.build_with_default_param("maxsum_gpu", {"stop_cycle": 30, "seed": 1},
                                                 mode=dcop.objective)
    cg = factor_graph.build_computation_graph(dcop)
    dist = adhoc.distribute(cg, dcop.agents.values(), computation_memory=algo_module.computation_memory,
                            communication_load=algo_module.communication_load)
    orchestrator = run_local_thread_dcop(algo, cg, dist, dcop, 1e9)
    try:
        orchestrator.deploy_computations()
        t0 = time.time()
        orchestrator.run(timeout=60)
        elapsed = time.time() - t0
        metrics = orchestrator.end_metrics()
        status = orchestrator.status
    finally:
        orchestrator.stop_agents(5)
        orchestrator.stop()
    return status, elapsed, metrics


@retry_once
def test_run_finishes_with_stop_cycle_and_counts_cycles(oracle_seam):
    status, elapsed, metrics = _run_gc10_with_stop_cycle()
    # `pydcop solve` prints FINISHED exactly when the run ended before the timeout because every
    # computation called finished() (commands/solve.py:547-553, orchestrator.py:898-913)
    assert status not in ("TIMEOUT", "STOPPED") and elapsed < 55, (status, elapsed)
    assert metrics["cycle"] == 30
    assert set(metrics["assignment"]) == {f"v{i}" for i in range(10)}
    assert metrics["violation"] == 0 and metrics["cost"] is not None
    # with a seed the run is reproducible although the agents register in thread order
    oracle_seam.reset()
    _, _, again = _run_gc10_with_stop_cycle()
    assert again["assignment"] == metrics["assignment"] and again["cost"] == metrics["cost"]


@retry_once
def test_solve_api_dsa_gpu(oracle_seam):
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    from pydcop.algorithms import AlgorithmDef
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    algo = AlgorithmDef.build_with_default_param("dsa_gpu", {"stop_cycle": 40, "seed": 3}, mode=dcop.objective)
    assignment = solve(dcop, algo, "oneagent", timeout=8)
    assert assignment in ({"v1": "R", "v2": "G", "v3": "R"}, {"v1": "G", "v2": "R", "v3": "G"})


@retry_once
def test_solve_api_mgm_gpu_matches_reference_mgm_fixed_point(oracle_seam):
    """MGM through the unmodified orchestrator with --algo mgm_gpu: a proper colouring of the
    3-variable chain (tests/api/test_api_solve.py style), a 1-opt assignment on the 10-variable
    instance: no single variable can improve alone — MGM's fixed point."""
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    from pydcop.algorithms import AlgorithmDef
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    algo = AlgorithmDef.build_with_default_param("mgm_gpu", {"stop_cycle": 20, "seed": 3}, mode=dcop.objective)
    assignment = solve(dcop, algo, "oneagent", timeout=8)
    assert assignment in ({"v1": "R", "v2": "G", "v3": "R"}, {"v1": "G", "v2": "R", "v3": "G"})
    oracle_seam.reset()
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring_10_4_15_0.1.yml")])
    algo = AlgorithmDef.build_with_default_param("mgm_gpu", {"stop_cycle": 30, "seed": 5}, mode=dcop.objective)
    assignment = solve(dcop, algo, "oneagent", timeout=8)
    _, cost = dcop.solution_cost(assignment, 1e9)
    for v in dcop.variables.values():
        for x in v.domain:
            _, c = dcop.solution_cost(dict(assignment, **{v.name: x}), 1e9)
            assert c >= cost - 1e-9, (v.name, x)


def test_no_gpu_means_loud_failure_not_fallback(pydcop_ready):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pydcop_b200.algorithms._session import GpuSession
    from pydcop_b200.engine import EngineError
    from pydcop.algorithms import AlgorithmDef, ComputationDef, load_algorithm_module
    from pydcop.computations_graph import factor_graph
    from pydcop.dcop.yamldcop import load_dcop_from_file
    GpuSession.reset()
    GpuSession.engine_factory = None
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    algo = AlgorithmDef.build_with_default_param("maxsum_gpu", {"session": "nogpu"}, mode="min")
    module = load_algorithm_module("maxsum_gpu")
    comps = []
    for node in factor_graph.build_computation_graph(dcop).nodes:
        c = module.build_computation(ComputationDef(node, algo))
        c.message_sender = lambda *a, **k: None
        c.periodic_action_handler = type("H", (), {"set_periodic_action": lambda s, p, cb: cb,
                                                   "remove_periodic_action": lambda s, h: None})()
        comps.append(c)
    for c in comps:
        c.start()
    s = comps[0]._session        # the proxies keep their session; the registry forgets it once the worker ends
    s.thread.join(timeout=30)
    assert isinstance(s.error, EngineError)
    assert GpuSession.get("maxsum:nogpu", "maxsum") is not s   # a later run under the same name starts afresh
    with pytest.raises(EngineError):
        comps[0]._poll()
    GpuSession.reset()


@retry_once
def test_cli_drop_in_without_gpu_reports_the_engine_error(pydcop_ready, tmp_path):
    """`pydcop solve --algo maxsum_gpu` through the unmodified CLI: the algorithm is accepted by the
    reference's argparse (choices come from list_available_algorithms) and, with no GPU in this
    container, the failure is printed — not silently replaced by a CPU computation."""
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    code = (
        "import sys; sys.path[:0] = [%r, %r]\n"
        "import ref_shim; ref_shim.install()\n"
        "from pydcop_b200 import launcher\n"
        "launcher.main(['-t', '5', 'solve', '--algo', 'maxsum_gpu', '--algo_params', 'stop_cycle:5',"
        " '-d', 'adhoc', %r])\n"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
         os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"),
         os.path.join(INSTANCES, "graph_coloring1.yaml"))
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True,
                       timeout=120, cwd=str(tmp_path))
    assert "EngineError" in r.stderr and "no CPU fallback" in r.stderr, r.stderr[-2000:]
    assert '"assignment": {}' in r.stdout            # nothing was computed on the CPU instead


@retry_once
@pytest.mark.parametrize("algo,extra", [("maxsum_gpu", []), ("dsa_gpu", ["--algo_params", "seed:3"]),
                                        ("mgm_gpu", ["--algo_params", "seed:3"])])
def test_cli_solve_end_to_end_with_cycle_metrics(pydcop_ready, tmp_path, algo, extra):
    """The unmodified `pydcop solve` CLI (argument parsing, distribution, orchestrator, agents, metrics
    collection on every cycle, JSON result) with --algo <x>_gpu; the engine seam holds the oracle since
    this container has no GPU.  tests/dcop_cli/test_solve.py:39-108 of the reference, for the GPU modules."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    metrics = tmp_path / "run.csv"
    code = (
        "import sys; sys.path[:0] = [%r, %r, %r]\n"
        "import ref_shim; ref_shim.install()\n"
        "from pydcop_b200 import launcher\n"
        "from pydcop_b200.algorithms._session import GpuSession\n"
        "from _oracle_engine import OracleEngine\n"
        "GpuSession.engine_factory = OracleEngine\n"
        "launcher.main(['-t', '20', 'solve', '--algo', %r, '--algo_params', 'stop_cycle:20', *%r,"
        " '--collect_on', 'cycle_change', '--run_metrics', %r, '-d', 'oneagent', %r])\n"
    ) % (root, os.path.join(root, "oracle"), os.path.join(root, "tests"), algo, extra, str(metrics),
         os.path.join(INSTANCES, "graph_coloring1.yaml"))
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True,
                       timeout=180, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout[r.stdout.index("{"):])
    assert out["status"] == "FINISHED" and out["cycle"] == 20 and out["violation"] == 0
    assert out["assignment"] in ({"v1": "R", "v2": "G", "v3": "R"}, {"v1": "G", "v2": "R", "v3": "G"})
    if algo == "maxsum_gpu":
        assert out["assignment"] == {"v1": "R", "v2": "G", "v3": "R"}
    rows = [ln for ln in metrics.read_text().splitlines() if ln.strip()]
    assert len(rows) >= 5 and "cycle" in rows[0]          # header + one line per collected cycle


@retry_once
@pytest.mark.parametrize("collect,dist", [(["--collect_on", "value_change"], "adhoc"),
                                          (["--collect_on", "period", "--period", "0.1"], "oneagent")])
def test_cli_solve_other_collection_modes_and_distributions(pydcop_ready, tmp_path, collect, dist):
    """Same CLI path with the other metric collection modes of commands/solve.py:278-293 and the adhoc
    distribution (which calls the module's computation_memory / communication_load)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    metrics = tmp_path / "run.csv"
    code = (
        "import sys; sys.path[:0] = [%r, %r, %r]\n"
        "import ref_shim; ref_shim.install()\n"
        "from pydcop_b200 import launcher\n"
        "from pydcop_b200.algorithms._session import GpuSession\n"
        "from _oracle_engine import OracleEngine\n"
        "GpuSession.engine_factory = OracleEngine\n"
        "launcher.main(['-t', '20', 'solve', '--algo', 'maxsum_gpu', '--algo_params', 'stop_cycle:30', *%r,"
        " '--run_metrics', %r, '-d', %r, %r])\n"
    ) % (root, os.path.join(root, "oracle"), os.path.join(root, "tests"), collect, str(metrics), dist,
         os.path.join(INSTANCES, "graph_coloring1.yaml"))
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True,
                       timeout=180, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout[r.stdout.index("{"):])
    assert out["status"] == "FINISHED" and out["cycle"] == 30
    assert out["assignment"] == {"v1": "R", "v2": "G", "v3": "R"} and out["violation"] == 0
    assert out["cost"] == pytest.approx(-0.1, abs=1e-9)
    assert metrics.exists() and len(metrics.read_text().splitlines()) >= 2


def test_incomplete_session_reports_itself_instead_of_waiting_forever(pydcop_ready):
    """Process mode puts every agent in its own OS process: a session then only ever sees a part of the
    graph.  After a grace period the proxies get a clear error instead of polling until the timeout."""
    from pydcop_b200.algorithms._session import GpuSession
    from pydcop.algorithms import AlgorithmDef, ComputationDef, load_algorithm_module
    from pydcop.computations_graph import factor_graph
    from pydcop.dcop.yamldcop import load_dcop_from_file
    GpuSession.reset()
    old = GpuSession.incomplete_grace
    GpuSession.incomplete_grace = 0.2
    try:
        dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
        algo = AlgorithmDef.build_with_default_param("maxsum_gpu", {"session": "partial"}, mode="min")
        module = load_algorithm_module("maxsum_gpu")
        nodes = factor_graph.build_computation_graph(dcop).nodes
        comps = []
        for node in nodes[:2]:                      # only a part of the graph lives "in this process"
            c = module.build_computation(ComputationDef(node, algo))
            c.message_sender = lambda *a, **k: None
            c.periodic_action_handler = type("H", (), {"set_periodic_action": lambda s, p, cb: cb,
                                                       "remove_periodic_action": lambda s, h: None})()
            comps.append(c)
        for c in comps:
            c.start()
        assert comps[0]._session.poll() is None     # inside the grace period: just not ready
        time.sleep(0.3)
        with pytest.raises(RuntimeError, match="thread mode"):
            comps[0]._poll()
    finally:
        GpuSession.incomplete_grace = old
        GpuSession.reset()


def test_every_reference_instance_runs_through_the_drop_in(oracle_seam):
    """All YAML instances of the reference's test suite (string domains, cost functions, extensional and
    intentional constraints, external python sources, external variables in SimpleHouse) through the
    unmodified orchestrator with --algo maxsum_gpu: a complete assignment every time, and on the
    instances with a unique optimum the reference's own answer."""
    import contextlib
    import glob
    import io
    from pydcop.algorithms import AlgorithmDef
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    files = sorted(glob.glob(os.path.join(INSTANCES, "*.y*ml")))
    assert len(files) >= 15
    known = {"graph_coloring1.yaml": -0.1, "graph_coloring_tuto.yaml": 12, "graph_coloring_tuto_max.yaml": 53,
             "secp_simple1.yaml": 2.3, "graph_coloring_csp.yaml": 0}
    for fn in files:
        oracle_seam.reset()
        dcop = load_dcop_from_file([fn])
        algo = AlgorithmDef.build_with_default_param("maxsum_gpu", {"stop_cycle": 25, "seed": 1}, mode=dcop.objective)
        with contextlib.redirect_stdout(io.StringIO()):
            res = solve(dcop, algo, "adhoc", timeout=2)
        assert set(res) == set(dcop.variables), os.path.basename(fn)
        violation, cost = dcop.solution_cost(res, 10000)
        name = os.path.basename(fn)
        if name in known:
            assert violation == 0 and cost == pytest.approx(known[name], abs=1e-9), (name, cost)


@retry_once
def test_without_stop_cycle_the_run_ends_at_the_timeout_and_the_worker_stops(oracle_seam):
    """Like the reference's MaxSum (no termination test, maxsum.py:62): without stop_cycle the engine keeps
    cycling until the orchestrator's timeout stops the computations; the assignment so far is returned and the
    session's worker thread ends."""
    import contextlib
    import io
    from pydcop.algorithms import AlgorithmDef
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    algo = AlgorithmDef.build_with_default_param("maxsum_gpu", {"session": "no_stop", "seed": 2}, mode=dcop.objective)
    with contextlib.redirect_stdout(io.StringIO()):
        res = solve(dcop, algo, "adhoc", timeout=2)
    assert res == {"v1": "R", "v2": "G", "v3": "R"}
    session = oracle_seam.last("maxsum:no_stop")
    assert session.snapshot is not None and session.snapshot.cycle > 30 and not session.snapshot.finished
    deadline = time.time() + 10
    while session.thread.is_alive() and time.time() < deadline:
        time.sleep(0.05)
    assert not session.thread.is_alive()


@retry_once
def test_second_run_in_one_process_gets_a_fresh_session(oracle_seam):
    """pydcop.infrastructure.run.solve twice in one process with the DEFAULT session name and NO reset in
    between (ADVICE r1): the second run must not be handed the finished session of the first."""
    from pydcop.algorithms import AlgorithmDef
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    d1 = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    algo = AlgorithmDef.build_with_default_param("dsa_gpu", {"stop_cycle": 40, "seed": 3}, mode=d1.objective)
    a1 = solve(d1, algo, "oneagent", timeout=8)
    d2 = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring_10_4_15_0.1.yml")])
    algo = AlgorithmDef.build_with_default_param("dsa_gpu", {"stop_cycle": 40, "seed": 3}, mode=d2.objective)
    a2 = solve(d2, algo, "oneagent", timeout=8)
    assert set(a1) == set(d1.variables) and set(a2) == set(d2.variables)
    assert a1 in ({"v1": "R", "v2": "G", "v3": "R"}, {"v1": "G", "v2": "R", "v3": "G"})
    assert not oracle_seam._sessions      # both workers retired their session


@retry_once
def test_solve_api_adsa_gpu(oracle_seam):
    """`adsa_gpu` through the unmodified orchestrator (engine seam: the A-DSA oracle): a proper colouring of the
    3-variable chain; the module lists the reference's parameters (adsa.py:121-125)."""
    from pydcop.algorithms import AlgorithmDef, load_algorithm_module
    from pydcop.dcop.yamldcop import load_dcop_from_file
    from pydcop.infrastructure.run import solve
    import pydcop.algorithms.adsa as ref
    mod = load_algorithm_module("adsa_gpu")
    ours = {p.name: (p.type, p.default_value) for p in mod.algo_params}
    for p in ref.algo_params:
        assert ours[p.name] == (p.type, p.default_value), p.name
    assert mod.GRAPH_TYPE == ref.GRAPH_TYPE
    dcop = load_dcop_from_file([os.path.join(INSTANCES, "graph_coloring1.yaml")])
    algo = AlgorithmDef.build_with_default_param("adsa_gpu", {"stop_cycle": 40, "seed": 3}, mode=dcop.objective)
    assignment = solve(dcop, algo, "oneagent", timeout=8)
    assert assignment in ({"v1": "R", "v2": "G", "v3": "R"}, {"v1": "G", "v2": "R", "v3": "G"})
