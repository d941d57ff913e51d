#!/usr/bin/env python
"""bench.py — MaxSum edge-message updates/s on BASELINE.json's configs (driver contract).

    python bench.py --gpus N --steps K --warmup W          (N>1: launched under torchrun)
    python bench.py --impl reference ...                   CPU arm: the oracle port, all host threads

A "step" is ONE synchronous MaxSum cycle over the whole factor graph: every factor->variable
min-marginal and every variable->factor message recomputed (2*E edge-message updates), damping,
send gate and value selection included.  N=1 workload: BASELINE.json configs[1]
(random binary DCOP, 100k vars, d=10, mean degree 4).  N>1: weak scaling, one C2-sized shard of a
single N*100k-variable graph per GPU, variable-cut partition, one NCCL halo exchange per cycle.

Timing: every timed step is bracketed by CUDA events on the launching stream; L2 is flushed
(256 MiB memset) between steps, outside the event pairs; per-rank time = sum over the K steps;
the job time is the max over ranks.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "maxsum_edge_message_updates_per_s"
UNIT = "updates/s"
E2E_CYCLES = 200  # cycles per end-to-end solve() (ingestion -> layout -> upload -> cycles -> assignment + cost)
PARITY_CYCLES = 12  # N > 1: sharded run vs one engine with the whole problem, outside the timed regions


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled in-process (NVML) every 10 ms during the timed region."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap"}

    def __init__(self, index=0):
        self.index, self.sm, self.mask, self.mx = index, [], 0, None
        self._stop = threading.Event()
        self._t = None
        self._err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            # NVML indexes physical devices; honour CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except (ValueError, IndexError):
                    pass
            self._h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self._err = repr(e)
            return
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
            except Exception as e:  # noqa: BLE001
                self._err = repr(e)
                return
            time.sleep(0.01)

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["unavailable: %s" % self._err]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.mx,
                "reasons": sorted(n for b, n in self.REASONS.items() if self.mask & b),
                "samples": len(self.sm)}


def oracle_instance(inst, L):
    tsz = np.concatenate([np.full(c.n_factors, c.table_size, np.int64) for c in L.classes]) \
        if L.classes else np.zeros(0, np.int64)
    # canonical table sizes (factor order of `inst`): invert the class permutation
    t = np.zeros(L.n_factors, np.int64)
    t[:] = tsz[L.factor_perm]
    return dict(inst, var_ptr=L.canon_var_ptr, var_edge=L.canon_var_edge,
                table_off=np.concatenate([[0], np.cumsum(t)]))


def oracle_threads():
    """OpenMP threads for the CPU arms, set EXPLICITLY (torchrun exports OMP_NUM_THREADS=1) and read back from
    the OpenMP runtime: PYDCOP_B200_CPU_THREADS, else every logical CPU of the box."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    want = int(os.environ.get("PYDCOP_B200_CPU_THREADS", "0") or 0) or (os.cpu_count() or 1)
    return orc.threads(want)


def time_oracle_blocks(o, block, min_seconds=3.0, min_repeats=5, max_seconds=40.0):
    """Median wall time of `block` cycles of the CPU oracle over >= min_repeats repeats and >= min_seconds of
    measurement (one C call per block: scratch allocated once, no per-cycle malloc / memcpy)."""
    times, t_start = [], time.perf_counter()
    while ((len(times) < min_repeats or sum(times) < min_seconds)
           and time.perf_counter() - t_start < max_seconds) or not times:
        t0 = time.perf_counter()
        o.step(block)
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), len(times), times


def cpu_baseline(inst, L, dtype=np.float32):
    """The CPU oracle (C port of the reference algorithm, OpenMP) on the same instance: median of >= 5 blocks of
    5 cycles, >= 8 s of measurement."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    nthreads = oracle_threads()
    o = orc.MaxSumOracle(oracle_instance(inst, L), dtype).init()
    o.step(2)
    block = 5
    med, reps, times = time_oracle_blocks(o, block, min_seconds=8.0, max_seconds=30.0)
    return {"value": 2.0 * L.n_edges * block / med, "unit": UNIT, "cores": nthreads, "kind": "port",
            "sample": f"median of {reps} blocks of {block} cycles of the same instance ({sum(times):.1f}s), "
                      f"oracle/dcop_oracle.c {'f32' if dtype == np.float32 else 'f64'}, OpenMP {nthreads} threads "
                      f"(omp_get_max_threads), spread min/max {min(times) / block * 1e3:.1f}/{max(times) / block * 1e3:.1f} ms per cycle"}


def reference_threadmode(seconds=10):
    """The UNMODIFIED reference's own thread-mode solve (`pydcop -t T solve -a maxsum -d adhoc`, one Python thread
    per agent: GIL-bound, effectively one core) timed on THIS box's host: BASELINE.md 3.1 (C1, the reference's
    graph_coloring_10_4_15_0.1.yml) and 3.2 (a C2-family instance with V = 100).  Reference = oracle/_ref, the
    pip-installed copy of the source tree (oracle/ref_shim.py adds three import shims, edits nothing).  Returns a
    list of cpu_baseline entries (kind `reference-threadmode`); [] with a reason when the install is absent."""
    import subprocess
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_shim
    if not ref_shim.reference_available():
        return [{"kind": "reference-threadmode", "unavailable": f"no reference at {ref_shim.REFERENCE_ROOT}"}]
    out = []
    with tempfile.TemporaryDirectory() as td:
        # C2-family instance, V = 100, d = 10, 200 binary constraints, tables as literal nested lists
        rng = np.random.default_rng(0)
        lines = ["name: c2_family_v100", "objective: min", "domains:", "  d: {values: [0,1,2,3,4,5,6,7,8,9]}",
                 "variables:"]
        lines += [f"  v{i:03d}: {{domain: d}}" for i in range(100)]
        lines.append("constraints:")
        for j in range(200):
            a, b = rng.choice(100, size=2, replace=False)
            t = rng.integers(0, 10, size=(10, 10)).tolist()
            lines += [f"  c{j:03d}:", "    type: intention", f"    function: '{t}[v{a:03d}][v{b:03d}]'"]
        lines += ["agents:"] + [f"  a{i:03d}: {{capacity: 1000}}" for i in range(300)]
        c2f = os.path.join(td, "c2_family_v100.yaml")
        open(c2f, "w").write("\n".join(lines) + "\n")
        c1 = os.path.join(ref_shim.REFERENCE_ROOT, "tests", "instances", "graph_coloring_10_4_15_0.1.yml")
        for name, path, n_edges, dist in (("C1 graph_coloring_10_4_15_0.1.yml", c1, 24, "adhoc"),
                                          ("C2-family V=100 d=10 F=200", c2f, 400, "oneagent")):
            code = ("import sys; sys.path[:0] = [%r]\nimport ref_shim; ref_shim.install()\n"
                    "from pydcop.dcop_cli import main\n"
                    "sys.argv = ['pydcop', '-t', %r, 'solve', '-a', 'maxsum', '-d', %r, %r]\nmain()\n"
                    ) % (os.path.join(ROOT, "oracle"), str(seconds), dist, path)
            try:
                r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True,
                                   timeout=seconds * 6 + 60, cwd=td)
                txt = r.stdout
                res = json.loads(txt[txt.index("{"):txt.rindex("}") + 1])
                cyc, tm = int(res.get("cycle") or 0), float(res.get("time") or seconds)
                out.append({"kind": "reference-threadmode", "value": 2.0 * n_edges * cyc / tm if cyc else 0.0,
                            "unit": UNIT, "cores": 1,
                            "sample": f"{name}: unmodified `pydcop -t {seconds} solve -a maxsum -d {dist}` in thread mode "
                                      f"(GIL-bound), {cyc} cycles in {tm:.1f}s, status {res.get('status')}, "
                                      f"msg_count {res.get('msg_count')}; host has {os.cpu_count()} logical CPUs"})
            except Exception as ex:  # noqa: BLE001 — a baseline must not cost the measured line
                out.append({"kind": "reference-threadmode", "unavailable": f"{name}: {ex!r}"[:300]})
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write `arrays` (name -> numpy array) as out_dir/<name>.npy, floats in float32 / float64 and the rest as
    float64.  When they add up to more than DUMP_LIMIT_BYTES, every array above an equal share of the limit is
    replaced by the same seeded sample of its elements (sorted flat indices from default_rng(0)), so two runs
    with the same arguments write comparable files."""
    arrays = {k: np.ravel(v if v.dtype in (np.float32, np.float64) else v.astype(np.float64))
              for k, v in arrays.items()}
    if sum(a.nbytes for a in arrays.values()) > DUMP_LIMIT_BYTES:
        share = DUMP_LIMIT_BYTES // len(arrays)
        for k, a in arrays.items():
            if a.nbytes > share:
                keep = share // a.itemsize
                arrays[k] = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def _partition_cache_path(inst, world, part):
    import hashlib
    h = hashlib.sha1(np.ascontiguousarray(inst["edge_var"]).view(np.uint8)).hexdigest()[:16]
    return os.path.join(ROOT, "gpurun_cache", f"owner_{part}_{world}_{len(inst['dom_size'])}_{h}.npy")


def shared_partition(inst, world, rank, dev, part):
    """(method name, owner array or 'blocks', error text or None): the partition is computed once on
    rank 0 and broadcast (pydcop_b200.multigpu.broadcast_owner); contiguous blocks if it fails.
    The partitioner is deterministic host code outside every timed region; an owner array precomputed
    for exactly this instance (gpurun_cache/, keyed by a hash of the scopes; tools/precompute_partitions.py)
    is used when present so that N GPUs do not sit idle behind it."""
    import torch
    import torch.distributed as dist
    from pydcop_b200.multigpu import broadcast_owner
    if part != "blocks" and world > 1:
        path = _partition_cache_path(inst, world, part)
        have = torch.tensor([int(os.path.exists(path))], dtype=torch.int32, device=dev)
        dist.all_reduce(have, op=dist.ReduceOp.MIN)
        if int(have.item()) == 1:
            owner = np.load(path).astype(np.int32)
            if owner.shape == (len(inst["dom_size"]),) and owner.max() < world:
                return part, owner, None
    owner, err = broadcast_owner(inst, world, rank, dev, part)
    if isinstance(owner, str):
        return "blocks", "blocks", err
    return part, owner, None


def side_workload(args, dev):
    """Other BASELINE configs on one GPU (not the driver's line): same timing rules."""
    import torch
    from pydcop_b200 import build_layout
    from pydcop_b200 import generators as G
    from pydcop_b200.engine import DsaEngine, MaxSumEngine, MgmEngine
    w = args.workload
    inst = {"c3": G.config_c3, "c5": G.config_c5, "target": G.config_target, "c4": G.config_c4,
            "mgm": G.config_c4, "mixed": G.config_mixed}[w]()
    L = build_layout(**inst)
    vb = 4 if args.precision == "f32" else 8
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1 and w == "mgm":
        raise SystemExit("--workload mgm is a single-GPU side line (MGM is not sharded)")
    part, part_owner, _perr = shared_partition(inst, world, rank, dev, os.environ.get("PYDCOP_B200_PARTITION", "auto"))
    if w == "c4":
        if world > 1:   # strong scaling: the same 1M-variable problem over `world` GPUs
            from pydcop_b200.multigpu_dsa import ShardedDsa
            eng = ShardedDsa(inst, rank, world, dev, precision=args.precision, seed=1, partition=part_owner,
                             halo=os.environ.get("PYDCOP_B200_HALO", "auto"))
        else:
            eng = DsaEngine(L, device=dev, precision=args.precision, seed=1)
        units, metric = L.n_vars, "dsa_variable_updates_per_s"
        d, k = 20, 6
        alg = L.n_vars * (k * (vb * d + 4 + 8 + vb) + 8)   # SURVEY 8d: ~584 B per variable update
    elif w == "mgm":    # MGM on the C4 instance (DESIGN.md §10 for the byte count)
        eng = MgmEngine(L, device=dev, precision=args.precision, seed=1)
        units, metric = L.n_vars, "mgm_variable_updates_per_s"
        d, k = 20, 6
        alg = L.n_vars * ((k * d + 2 * k + 2) * vb + 8 * k + 8)
    else:
        if world > 1:   # strong scaling of the named instance (BASELINE configs[2]: the grid over 1 -> 8 GPUs)
            from pydcop_b200.multigpu import ShardedMaxSum
            eng = ShardedMaxSum(inst, rank, world, dev, precision=args.precision,
                                halo=os.environ.get("PYDCOP_B200_HALO", "auto"), partition=part_owner)
        else:
            eng = MaxSumEngine(L, device=dev, precision=args.precision)
        units, metric = 2 * L.n_edges, METRIC
        alg = G.algorithmic_bytes_per_cycle_inst(inst, vb)
    eng.init()
    if args.profile:
        eng.step(max(3, args.warmup) + args.steps)
        torch.cuda.synchronize(dev)
        return
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    eng.step(max(3, args.warmup))
    torch.cuda.synchronize(dev)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    evs = []
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.step(1)
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize(dev)
    clocks = sampler.stop() if rank == 0 else None
    ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    parity = None
    breakdown = None
    if world > 1 and getattr(eng, "peer", None) is not None and hasattr(eng, "timed_breakdown"):
        breakdown = {k: round(1e3 * v, 2) for k, v in eng.timed_breakdown(30).items()}   # every rank takes part
        breakdown["unit"] = "us per cycle, rank 0"
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        # sharded run (exchange path as timed) against ONE engine with the whole problem, fresh start
        eng.init()
        eng.step(PARITY_CYCLES)
        got = eng.values()
        if rank == 0:
            if w == "c4":
                want = DsaEngine(L, device=dev, precision=args.precision, seed=1).init().step(PARITY_CYCLES).values()
            else:
                want = MaxSumEngine(L, device=dev, precision=args.precision,
                                    record_sent=False).init().step(PARITY_CYCLES).values()[0]
            parity = {"cycles": PARITY_CYCLES, "assignment_equals_single_gpu": bool(np.array_equal(got, want)),
                      "n_differ": int((np.asarray(got) != np.asarray(want)).sum())}
        dist.barrier()
        if rank != 0:
            return
    peaks, kind = load_peaks()
    ach = alg / (ms * 1e-3) / 1e9
    line = {"metric": metric, "value": units / (ms * 1e-3), "unit": "updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "dtype": args.precision,
            "higher_is_better": True, "data": "synthetic", "clocks": clocks,
            "scaling": "strong" if world > 1 else None,
            "config": {"workload": w, "n_vars": L.n_vars, "n_factors": L.n_factors, "n_edges": L.n_edges,
                       "l2": "flushed between timed steps (256 MiB memset, outside the event pairs)"},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"] * world, "unit": "GB/s",
                         "frac": ach / (peaks["hbm_gbs"] * world), "algorithmic_bytes_per_step": int(alg)}}
    if world > 1:
        line["parity"] = parity
        line["config"]["partition"] = part
        if breakdown is not None:
            line["breakdown"] = breakdown
        if w == "c4":
            line["config"]["boundary_values"] = int(eng.shard.n_boundary)
            line["config"]["halo"] = "peer push" if eng.peer is not None else "nccl all_to_all"
        else:
            line["config"]["cut_edges"] = int(eng.plan.n_cut_edges)
            line["config"]["halo"] = "peer push" if eng.peer is not None else "nccl all_to_all"
    print(json.dumps(line))


def workload_config(n_vars, world):
    """`config` of the main line: the workload and how it is measured — STATIC, so that the GPU arm and the
    reference arm print the same dict at every N (what a run finds out goes under `run`)."""
    return {"workload": f"random binary DCOP {n_vars} vars d=10 deg=4 (BASELINE configs[1] "
                        f"{'x%d weak' % world if world > 1 else ''})".strip(),
            "n_vars": n_vars, "n_factors": 2 * n_vars, "n_edges": 4 * n_vars, "d": 10,
            "params": "damping 0.5 both, stability 0.1, noise 0.01, start_messages leafs",
            "partition": (f"variable cut over {world} GPUs, method "
                          f"{os.environ.get('PYDCOP_B200_PARTITION', 'auto')}" if world > 1 else "single GPU"),
            "l2": "flushed between timed steps (256 MiB memset, outside the event pairs)",
            "step": "one synchronous MaxSum cycle over all edges"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--vars-per-gpu", type=int, default=100_000)
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="tuning sweeps: skip the end-to-end leg (line has no e2e key)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c5", "target", "c4", "mgm", "mixed"],
                    help="c2 (default, the driver's line) | c3 Ising 1024^2 | c5 arity-3 | target 1M vars "
                         "| c4 DSA 1M vars d=20 (variable updates/s) | mgm: MGM on the c4 instance")
    ap.add_argument("--profile", action="store_true",
                    help="lean run for ncu: init + warmup + steps back to back, no flush/e2e/JSON")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the assignment, its reported costs and the q / r messages "
                         "the last timed step left as DIR/<name>.npy (c2 workload; N > 1: the assignment)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "c2" or args.impl != "b200" or args.profile):
        ap.error("--dump-outputs writes the outputs of the timed c2 path (--impl b200, no --profile)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from pydcop_b200 import build_layout
    from pydcop_b200.generators import config_c2

    n_vars = args.vars_per_gpu * max(1, world)
    config = workload_config(n_vars, world)
    run_info = {}   # what this run found out (cut size, halo path ...): NOT part of `config`, which both arms share

    if args.impl == "reference":
        # the reference's own algorithm for this path on the host cores (C port of the pure-Python reference,
        # OpenMP): rank 0 only, same instance and `config` as the GPU arm at this N.  A "step" is one cycle; the
        # line reports the MEDIAN over >= 5 blocks of `--steps` cycles and >= 3 s of measurement.
        if rank != 0:
            return
        inst = config_c2(seed=0, n_vars=n_vars)
        L = build_layout(**inst)
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as orc
        nthreads = oracle_threads()
        o = orc.MaxSumOracle(oracle_instance(inst, L), np.float32).init()
        o.step(max(1, args.warmup))
        med, reps, times = time_oracle_blocks(o, max(1, args.steps), min_seconds=3.0, min_repeats=5, max_seconds=90.0)
        val = 2.0 * L.n_edges * args.steps / med
        sample = (f"median of {reps} blocks of {args.steps} cycles ({sum(times):.1f}s measured, min/max block "
                  f"{min(times):.3f}/{max(times):.3f}s), oracle/dcop_oracle.c f32 (C port of the pure-Python "
                  f"reference), OpenMP {nthreads} threads (omp_get_max_threads; OMP_NUM_THREADS in the environment: "
                  f"{os.environ.get('OMP_NUM_THREADS', 'unset')}), host has {os.cpu_count()} logical CPUs")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * med / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": nthreads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference "
                         "for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from pydcop_b200.engine import MaxSumEngine

    if args.workload != "c2":
        return side_workload(args, dev)
    inst = config_c2(seed=0, n_vars=n_vars)
    from pydcop_b200.generators import algorithmic_bytes_per_cycle_inst
    vb = 4 if args.precision == "f32" else 8
    n_edges_global = int(len(inst["edge_var"]))
    if world > 1:
        from pydcop_b200.multigpu import ShardedMaxSum
        part, part_owner, perr = shared_partition(inst, world, rank, dev,
                                                  os.environ.get("PYDCOP_B200_PARTITION", "auto"))
        if perr:
            run_info["partition_error"] = perr
        runner = ShardedMaxSum(inst, rank, world, dev, precision=args.precision,
                               halo=os.environ.get("PYDCOP_B200_HALO", "auto"), partition=part_owner)
        L = None
        run_info["cut_edges"] = runner.plan.n_cut_edges
        run_info["partition"] = (f"{part}: the fewer-cut of contiguous blocks and a multilevel k-way split "
                                 f"(pydcop_b200/partition.py), {runner.plan.n_cut_edges} of {n_edges_global} edges cut"
                                 if part == "auto" else f"{part}, {runner.plan.n_cut_edges} of {n_edges_global} edges cut")
    else:
        L = build_layout(**inst)
        runner = MaxSumEngine(L, device=dev, precision=args.precision, record_sent=True)
    alg_bytes = algorithmic_bytes_per_cycle_inst(inst, vb)
    updates_per_step = 2 * n_edges_global

    if args.profile:
        runner.init()
        runner.step(max(3, args.warmup) + args.steps)
        torch.cuda.synchronize(dev)
        return
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    runner.init()
    if world > 1:
        if runner.peer is None:
            run_info["halo"] = "pack kernel + ONE NCCL all_to_all (q and r rows together) + unpack kernel per cycle"
        elif getattr(runner.peer, "fused", False):
            run_info["halo"] = ("FUSED: the factor-side and variable-side kernels store every boundary row into its "
                                "consumer's buffer over NVLink (CUDA IPC) from the lane that produced it; one release "
                                "kernel publishes the cycle's epoch flag to the peers, device-side acquire wait; whole "
                                "cycle enqueued by one C call (fg_maxsum_shard_step)")
        else:
            run_info["halo"] = ("push kernel storing boundary rows straight into the peers' buffers over NVLink (CUDA "
                                "IPC), its last block releasing the cycle's epoch flag to the peers; device-side "
                                "acquire wait; whole cycle enqueued by one C call (fg_maxsum_shard_step)"
                                + ("; rows pushed right behind each side (split), 16-byte destination runs"
                                   if os.environ.get("PYDCOP_B200_PUSH_SPLIT", "1") != "0" else "; one push after both sides"))
    for _ in range(max(3, args.warmup)):
        runner.step(1)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = runner.launch_count
    evs = []
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        runner.step(1)
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    launches = runner.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:   # the state the last timed step left, read back outside the timed region
        if world > 1:
            out = {"value": runner.values()}    # collective: every rank takes part
        else:
            ft = np.float32 if args.precision == "f32" else np.float64
            value, value_cost = runner.values()
            q, r = runner.messages()
            out = {"value": value, "value_cost": value_cost.astype(ft), "q": q.astype(ft), "r": r.astype(ft)}
        if rank == 0:
            dump_outputs(args.dump_outputs, out)
    ms = sum(a.elapsed_time(b) for a, b in evs)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = updates_per_step / (ms_per_step * 1e-3)
    breakdown = None
    if world > 1:   # device time of the phases of a cycle on rank 0 (separate short loop, phases serialised)
        breakdown = {k: round(1e3 * v, 2) for k, v in runner.timed_breakdown(50).items()}
        breakdown["unit"] = "us per cycle, rank 0"
        runner.check()

    parity = None
    if world > 1:
        # outside every timed region: the sharded run (halo path as timed) against ONE engine holding the
        # whole problem on rank 0's GPU, a few cycles from a fresh start — far from convergence, so a wrong
        # or late boundary row changes the assignment
        runner.init()
        runner.step(PARITY_CYCLES)
        got = runner.values()
        if rank == 0:
            try:
                ref = MaxSumEngine(build_layout(**inst), device=dev, precision=args.precision,
                                   record_sent=False).init().step(PARITY_CYCLES)
                want = ref.values()[0]
                parity = {"cycles": PARITY_CYCLES,
                          "assignment_equals_single_gpu": bool(np.array_equal(got, want)),
                          "n_differ": int((np.asarray(got) != np.asarray(want)).sum())}
                del ref
            except Exception as ex:  # noqa: BLE001 — the check must not cost the measured line
                parity = {"cycles": PARITY_CYCLES, "error": repr(ex)}
        dist.barrier()
    # end to end through the PUBLIC API, pydcop_b200.solve.solve(): host arrays in, result dict out.  Inside the timed
    # region, every repeat: ingestion of the arrays, noise draws, layout packing (host), engine construction
    # (device allocations, host -> device copies of tables / unary / CSR from pageable host memory), init,
    # E2E_CYCLES cycles, device -> host copy of the assignment, cost / violation reduction on the device, the
    # name -> value dict.  N > 1: every rank calls solve() (the partition is given: computing it is the
    # partitioner's cost, reported separately), time = max over ranks.  Wall clock between device synchronisations.
    from pydcop_b200 import solve as S
    times, h2d, d2h = [], 0, 0
    if not args.no_e2e:
        del runner
        torch.cuda.empty_cache()
        for it in range(1 + 3):
            flush.zero_()
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            res = S.solve(inst, "maxsum", {"stop_cycle": E2E_CYCLES}, precision=args.precision, device=dev, seed=0,
                          partition=part_owner if world > 1 else "auto",
                          halo=os.environ.get("PYDCOP_B200_HALO", "auto"))
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            assert res["status"] == "FINISHED" and res["cycle"] == E2E_CYCLES
            h2d, d2h = res["h2d_bytes"], res["d2h_bytes"]
            if it >= 1:
                times.append(dt * 1e3)
    e2e_ms = float(np.median(times)) if times else float("nan")
    if world > 1:
        t = torch.tensor([e2e_ms, float(h2d), float(d2h)], device=dev, dtype=torch.float64)
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        e2e_ms, h2d, d2h = float(tm[0].item()), int(t[1].item()), int(t[2].item())
    e2e = {"value": updates_per_step * E2E_CYCLES / (e2e_ms * 1e-3), "unit": UNIT,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "solve": f"pydcop_b200.solve.solve(arrays, 'maxsum', stop_cycle={E2E_CYCLES}): ingestion + layout packing on "
                    f"the host, engine construction + uploads, init, {E2E_CYCLES} cycles, assignment + device cost "
                    f"reduction back; median of 3 solves after 1 warm-up: {e2e_ms:.1f} ms per solve"
                    + (" (max over ranks; bytes summed over ranks)" if world > 1 else "")}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks, peak_kind = load_peaks()
    peak = float(peaks["hbm_gbs"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic_c2_f32.json")   # the final round-2 kernels (k_f2v_warp + k_v2f_warp)
    if world == 1 and args.precision == "f32" and args.vars_per_gpu == 100_000 and os.path.exists(tpath):
        traffic = json.load(open(tpath))["per_step_bytes"]   # from the committed ncu --set full capture
    per_gpu_bytes = alg_bytes / max(1, world)
    achieved = per_gpu_bytes / (ms_per_step * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": config, "clocks": clocks, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": ("constant from the committed ncu --set full capture profiles/r02_traffic_c2_f32.json "
                                        "(dram__bytes_read + dram__bytes_write of one launch of each kernel of this build), "
                                        "not a measurement of this run"
                                        if traffic is not None else None),
                     "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                     "algorithmic_bytes_per_step": int(per_gpu_bytes),
                     "bytes_per_update": alg_bytes / updates_per_step,
                     "kernel": "f2v + v2f kernels of one cycle (whole step; per-kernel split in "
                               "profiles/)"},
        "e2e": e2e,
    }
    if run_info:
        line["run"] = run_info
    if parity is not None:
        line["parity"] = parity
    if breakdown is not None:
        line["breakdown"] = breakdown
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(inst, L)
        # the UNMODIFIED reference's thread-mode solve on this host (BASELINE.md 3.1-3.2): reported next to the port
        line["cpu_baseline_reference_threadmode"] = reference_threadmode(int(os.environ.get("PYDCOP_B200_REF_SECONDS", "10")))
    print(json.dumps(line))


if __name__ == "__main__":
    main()
