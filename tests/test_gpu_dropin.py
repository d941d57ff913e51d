"""GPU: ONE true drop-in run — the UNMODIFIED reference CLI (`pydcop solve`: argument parsing, distribution,
orchestrator, agents in thread mode, JSON result) with `--algo maxsum_gpu` / `dsa_gpu` / `mgm_gpu` and the REAL
engine behind the proxies (no oracle in the seam).  The reference is the unmodified copy that
oracle/install_reference.py installed into oracle/_ref/ (__graft_entry__.build()); the three import shims of oracle/ref_shim.py are installed before `pydcop` is imported, nothing in
the reference is edited.  Checked: status FINISHED (every graph node finished, orchestrator.py:898-913), the cycle
count, and the assignment against the CPU oracle on the same problem (algorithms/__init__.py:527-566 loads the
module by name)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as orc
import ref_shim

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not ref_shim.reference_available(),
                                 reason="no reference: oracle/_ref/ not installed")]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INSTANCES = os.path.join(ref_shim.REFERENCE_ROOT, "tests", "instances")


def _cli(args, tmp_path, timeout=240):
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import ref_shim; ref_shim.install()\n"
            "from pydcop_b200 import launcher\n"
            "launcher.main(%r)\n") % (ROOT, os.path.join(ROOT, "oracle"), list(args))
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True,
                       timeout=timeout, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    out = r.stdout
    return json.loads(out[out.index("{"):out.rindex("}") + 1]), r.stderr


@pytest.mark.parametrize("instance", ["graph_coloring_10_4_15_0.1.yml", "graph_coloring1.yaml"])
def test_pydcop_solve_maxsum_gpu_real_engine_under_the_reference_orchestrator(tmp_path, instance):
    from pydcop_b200 import ingest
    path = os.path.join(INSTANCES, instance)
    res, err = _cli(["-t", "60", "solve", "--algo", "maxsum_gpu", "--algo_params", "stop_cycle:30",
                     "--algo_params", "noise:0", "--algo_params", "precision:f64", "-d", "adhoc", path], tmp_path)
    assert res["status"] == "FINISHED", (res, err[-1500:])
    assert res["cycle"] == 30
    d = ingest.load_yaml(path)
    o = orc.MaxSumOracle(d.instance(), np.float64, mode=d.objective).init().step(30)
    want = {n: d.values_of(i)[int(o.value[i])] for i, n in enumerate(d.var_names)}
    assert res["assignment"] == want
    from pydcop_b200 import solve as S
    viol, cost = S.solution_cost(d, o.value)     # the CLI's default `-i` is float("inf") (commands/solve.py:315-324)
    assert res["violation"] == viol and res["cost"] == pytest.approx(cost)


@pytest.mark.parametrize("algo", ["dsa_gpu", "mgm_gpu"])
def test_pydcop_solve_local_search_gpu_modules_real_engine(tmp_path, algo):
    """DSA / MGM proxies with the real engines: the run FINISHES at stop_cycle and returns a full assignment
    whose cost the reference itself evaluates (the trajectories are tied to the oracle in the engine tests)."""
    path = os.path.join(INSTANCES, "graph_coloring_10_4_15_0.1.yml")
    res, err = _cli(["-t", "60", "solve", "--algo", algo, "--algo_params", "stop_cycle:25",
                     "--algo_params", "seed:3", "-d", "adhoc", path], tmp_path)
    assert res["status"] == "FINISHED", (res, err[-1500:])
    assert len(res["assignment"]) == 10 and res["cycle"] >= 24
    assert res["violation"] <= 3      # 10 variables, 3 colours: a local search leaves at most a few conflicts
