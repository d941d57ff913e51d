"""solve() under torch.distributed (gloo, world 2): every rank calls it with the same arguments,
gets the same result, and that result equals the single-process one.  The GPU engines are
replaced through `sharded_kwargs` (MaxSum: the kernel source through the host shim; DSA: the
oracle), everything else — ingestion, noise, partition broadcast, sharding, exchange, the
collective timeout decision, the result dict — is the product code."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from _oracle_engine import OracleEngine
from pydcop_b200 import solve as S
from pydcop_b200.generators import random_factor_graph
from test_maxsum_generic_hostshim import CUDA_INC

pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")),
                                reason="CUDA toolkit headers not present")
HERE = os.path.dirname(os.path.abspath(__file__))
SPLIT = [os.path.join(HERE, "golden", "yaml", f) for f in ("split_problem.yaml", "split_agents.yaml")]


def _problem(kind):
    if kind == "yaml":
        return SPLIT
    inst = random_factor_graph(60, 4, 110, 2, seed=3, noise=0.0)
    inst["tables"] = np.floor(inst["tables"] / 3.0).astype(np.float32)
    return inst


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, kind, algo, params, kw, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        if algo == "maxsum":
            from test_multigpu_maxsum_gloo import HostEngine, _pack, _unpack
            sk = dict(engine_factory=HostEngine, pack=_pack, unpack=_unpack)
        else:
            from test_multigpu_dsa_cpu import FakeDsaEngine, _pack, _unpack
            sk = dict(engine_factory=FakeDsaEngine, pack=_pack, unpack=_unpack)
        res = S.solve(_problem(kind), algo, params, precision="f64", sharded_kwargs=sk, **kw)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", res))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, "FAIL " + repr(e) + traceback.format_exc(), None))


@pytest.mark.parametrize("kind,algo,params,kw", [
    ("yaml", "maxsum", {"stop_cycle": 20}, dict(seed=4, partition="blocks")),
    ("random", "maxsum", {"stop_cycle": 12, "noise": 0.0, "damping_nodes": "vars"}, dict(partition="multilevel")),
    ("random", "dsa", {"stop_cycle": 15, "variant": "C", "probability": 0.5}, dict(seed=9, partition="multilevel")),
    # the timeout counts from the start of solve(), set-up included: leave room for a first chunk on a busy host
    ("yaml", "dsa", {"variant": "A"}, dict(seed=2, timeout=5.0, chunk=3)),
])
def test_distributed_solve_equals_single_process(kind, algo, params, kw):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, kind, algo, params, kw, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=30)
    for rank, status, r in res:
        assert status == "ok", (rank, status)
    a, b = res[0][2], res[1][2]
    assert a["assignment"] == b["assignment"] and a["cycle"] == b["cycle"] and a["status"] == b["status"]
    assert a["n_gpus"] == 2
    if "timeout" in kw:
        assert a["status"] == "TIMEOUT" and a["cycle"] % 3 == 0 and a["cycle"] > 0
        return
    single_kw = {k: v for k, v in kw.items() if k not in ("partition",)}
    single_kw.setdefault("seed", 0)       # the distributed run defaults the seed to 0
    single = S.solve(_problem(kind), algo, params, precision="f64", engine_factory=OracleEngine, **single_kw)
    assert a["assignment"] == single["assignment"] and a["cost"] == pytest.approx(single["cost"], rel=1e-12)
    assert a["status"] == single["status"] == "FINISHED" and a["cycle"] == single["cycle"]


def test_mgm_is_refused_in_distributed_mode():
    with pytest.raises(ValueError, match="not sharded"):
        import torch.distributed as d
        port = _free_port()
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        d.init_process_group("gloo", rank=0, world_size=1)
        try:
            S.solve(SPLIT, "mgm", {"stop_cycle": 3}, distributed=True, sharded_kwargs={"engine_factory": object})
        finally:
            d.destroy_process_group()
