#!/usr/bin/env python
"""bench.py — env-steps/sec of the batched CIM Env.step hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W           # our CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N ...           # the reference's own CPU path on the host cores
    python bench.py ... --dump-outputs DIR                  # also save the last timed step's outputs as DIR/<name>.npy

A bench "step" = one batched Env.step over all replicas of a rank (hashed random agent + step kernel).
Workload (config.workload): BASELINE.json configs[1] — CIM toy.4p_ssdd_l0.0, 1024 parallel envs per GPU,
1000 ticks, random actions; episodes are restarted (Env.reset, inside the timed region) when they end.

Printed JSON (rank 0, one line): see the keys at the bottom.  `value` = whole-job env-steps/s with state resident
in HBM, L2 flushed between timed steps, device-timed per step with CUDA events, max over ranks.  `e2e` = the same
metric through the host-buffer C-ABI call (maro_cim_step_pinned: actions in / decisions + metrics out through pinned
host buffers every step) with the agent evaluated on the host (tools/host_agent.c).  Extras on the same line:
`graph_mode` (agent + step pairs replayed from CUDA graphs), `rl_shaping` (device-side RL state / action / reward
shaping), `roofline`, `cpu_baseline`, `clocks`.

Other workloads (not the headline): --scenario citi_bike (BASELINE config #3), --scenario vm_scheduling (config #5 on the
synthetic azure.2019.10k-scale trace of tools/vm_trace_gen.py), --topology global_trade.22p_l0.8 --ticks 500 (config #4).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_DECLARED = {"toy.4p_ssdd_l0.0": 886}  # SURVEY.md §8: frame bytes per replica in the reference's declared dtypes


_JSON_FD = None


def emit(line: dict) -> None:
    """The one JSON line of the contract, written to the process's ORIGINAL stdout (see main)."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--replicas", type=int, default=1024, help="parallel envs per GPU")
    ap.add_argument("--ticks", type=int, default=1000)
    ap.add_argument("--topology", default="toy.4p_ssdd_l0.0")
    ap.add_argument("--scenario", default="cim", choices=["cim", "citi_bike", "vm_scheduling"],
                    help="citi_bike = BASELINE config #3 (frozen toy.3s_4t trace, greedy agent, snapshot_resolution 10); "
                         "vm_scheduling = config #5 (synthetic azure.2019.10k-scale trace, best-fit agent)")
    ap.add_argument("--vm-count", type=int, default=10000, help="vm_scheduling: VMs in the synthetic trace")
    ap.add_argument("--vm-query-agent", action="store_true", help="vm_scheduling e2e: the host agent makes the reference agent's snapshot "
                    "query every step (3.3 MB D2H) instead of reading the decision row's remaining-cores extension")
    ap.add_argument("--vm-trace-dir", default="", help="vm_scheduling: where the synthetic trace is written and reused (default: a fresh temporary directory, removed at exit)")
    ap.add_argument("--max-snapshots", type=int, default=0, help="0 = keep every frame (reference default)")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--graph-chunk", type=int, default=32, help="steps per CUDA-graph chunk of the extra graph-mode measurement (0: off)")
    ap.add_argument("--chunk", type=int, default=64, help="cim: env-steps fused into one resident-kernel launch (maro_cim_rollout_device)")
    ap.add_argument("--seeds", type=int, default=1, help="cim: distinct topology seeds in the batch (replica r runs seed 4096 + r %% seeds; "
                    "only noisy topologies differ by seed)")
    ap.add_argument("--launch-per-step", action="store_true", help="cim: time the one-launch-per-Env.step path as `value` instead of fused rollouts")
    ap.add_argument("--matrix", action="store_true", help="north-star measurement matrix: CIM toy.4p_ssdd_l0.0 and citi_bike toy.3s_4t at "
                    "1 k / 8 k / 64 k envs per GPU, short runs; the line's top-level keys are the first (headline) entry's")
    ap.add_argument("--matrix-sizes", default="1024,8192,65536")
    ap.add_argument("--skip-extras", action="store_true", help="cim: only the contract keys (value, e2e, roofline, cpu_baseline, clocks)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the timed path returned in its last step (decision rows, metrics) to DIR/<name>.npy as float64; "
                         "with --matrix, the headline entry's")
    return ap.parse_args()


DUMP_LIMIT = 64 << 20  # bytes of all --dump-outputs files together


def dump_outputs(out_dir, arrays, rank, world):
    """--dump-outputs: one float64 .npy per array (integer outputs convert exactly), rows indexed by replica.  Past
    DUMP_LIMIT a fixed, seeded sample of replica rows is kept, the same for every array, and its indices are written as
    replica_rows.npy.  Ranks other than 0 add _rank<r> to the names."""
    import numpy as np

    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values()) + 8
    keep = min(n, (DUMP_LIMIT // world - 128 * (len(arrays) + 1)) // row_bytes)  # (128: .npy header)
    if keep < n:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["replica_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if rank else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.001)

    def start(self):
        if self._nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------------------------- reference arm
def reference_built() -> bool:
    """oracle/_ref holds the reference's compiled package (oracle/build_ref.sh also stages its Python sources on their own,
    which cannot run the simulator)"""
    import glob

    return bool(glob.glob(os.path.join(ROOT, "oracle", "_ref", "maro", "backends", "frame*.so")))


def run_reference(args, rank, world):
    """The reference's own CPU implementation on the host cores: maro.vector_env.VectorEnv(batch_num=cpu_count)
    from oracle/_ref (the unmodified reference built by oracle/build_ref.sh) when present, else the C port."""
    if rank != 0:
        return
    import numpy as np

    ref_root = os.path.join(ROOT, "oracle", "_ref")
    cores = os.cpu_count() or 1
    line = {"metric": "env-steps/sec", "unit": "env-steps/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": f"CIM {args.topology}, {args.ticks} ticks, random actions", "replicas": cores}}
    if args.scenario == "vm_scheduling":
        return run_reference_vm(args, line, ref_root, cores)
    if args.scenario == "citi_bike":
        return run_reference_bike(args, line, ref_root, cores)
    if reference_built():
        os.environ["SKIP_DEPLOYMENT"] = "TRUE"
        os.environ.setdefault("DEFAULT_BACKEND_NAME", "dynamic")  # the Cython/C++ RawBackend the north-star names
        sys.path.insert(0, ref_root)
        sys.path.insert(1, os.path.join(ref_root, "_stubs"))
        from maro.simulator.scenarios.cim.common import Action, ActionType
        from maro.vector_env import VectorEnv

        from tools.workloads import cim_policy_random as policy_random

        with VectorEnv(batch_num=cores, scenario="cim", topology=args.topology, durations=args.ticks) as env:
            def agent(decisions, step):
                acts = {}
                for i, d in enumerate(decisions):
                    if d is None:
                        continue
                    row = [d.tick, d.port_idx, d.vessel_idx, d.action_scope.load, d.action_scope.discharge,
                           d.early_discharge]
                    v, p, q, t = policy_random(row, 0, i, step)
                    acts[i] = Action(v, p, q, ActionType.DISCHARGE if t else ActionType.LOAD)
                return acts

            def loop(n):
                nonlocal metrics, decisions, done, step, env_steps
                for _ in range(n):
                    if done:
                        env.reset()
                        metrics, decisions, done = env.step(None)
                        step = 0
                        env_steps += cores
                        continue
                    metrics, decisions, done = env.step(agent(decisions, step))
                    step += 1
                    env_steps += cores

            env_steps, step = 0, 0
            metrics, decisions, done = env.step(None)
            loop(args.warmup)
            env_steps = 0
            t0 = time.perf_counter()
            loop(args.steps)
            dt = time.perf_counter() - t0
        kind, sample = "reference", f"VectorEnv(batch_num={cores}) x {args.steps} steps, backend={os.environ['DEFAULT_BACKEND_NAME']}"
        value = env_steps / dt
    else:
        from maro_b200.scenarios.cim.topology import build_topology
        from oracle.cim_oracle import CimOracle

        topo = build_topology(args.topology, args.ticks)
        o = CimOracle(topo)
        env_steps, t0, ep = 0, time.perf_counter(), 0
        while env_steps < args.steps * 1024 and time.perf_counter() - t0 < 60:
            o.reset()
            n, _ = o.run_episode(1, 0, ep)
            env_steps += n
            ep += 1
        dt = time.perf_counter() - t0
        kind, sample, cores = "port", f"{ep} episodes of the C restatement, 1 thread", 1
        value = env_steps / dt
    line.update({"value": value, "ms_per_step": 1000.0 * dt / max(1, args.steps),
                 "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
                 "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    emit(line)


def run_reference_bike(args, line, ref_root, cores):
    """citi_bike: the unmodified reference (VectorEnv over every host core, greedy top-1 agent of
    examples/citi_bike/greedy/launcher.py) on the frozen toy.3s_4t trace; else the C port."""
    ticks = min(args.ticks, 2880) if args.ticks != 1000 else 1440
    line["config"] = {"workload": f"citi_bike toy.3s_4t (frozen trace), {ticks} ticks, greedy top-1 agent, snapshot_resolution 10",
                      "replicas": cores}
    if reference_built():
        os.environ["SKIP_DEPLOYMENT"] = "TRUE"
        sys.path.insert(0, ref_root)
        sys.path.insert(1, os.path.join(ref_root, "_stubs"))
        from maro.simulator.scenarios.citi_bike.common import Action, DecisionType
        from maro.vector_env import VectorEnv

        from tools.workloads import bike_greedy as greedy, bike_toy_config_dir

        with VectorEnv(batch_num=cores, scenario="citi_bike", topology=bike_toy_config_dir(), durations=ticks,
                       snapshot_resolution=10) as env:
            def agent(decisions):
                acts = {}
                for i, d in enumerate(decisions):
                    if d is None:
                        continue
                    v, cand = greedy(d)
                    acts[i] = (Action(d.station_idx, cand, int(v)) if d.type == DecisionType.Supply else Action(cand, d.station_idx, int(v)))
                return acts

            metrics, decisions, done = env.step(None)
            env_steps, t0 = 0, None
            for k in range(args.warmup + args.steps):
                if k == args.warmup:
                    t0, env_steps = time.perf_counter(), 0
                if done:
                    env.reset()
                    metrics, decisions, done = env.step(None)
                else:
                    metrics, decisions, done = env.step(agent(decisions))
                env_steps += cores
            dt = time.perf_counter() - t0
        kind, sample = "reference", f"VectorEnv(batch_num={cores}) x {args.steps} steps, static backend"
    else:
        from maro_b200.scenarios.citi_bike.data import build_bike_topology
        from oracle.bike_oracle import BikeOracle
        from tools.workloads import bike_toy_config

        o = BikeOracle(build_bike_topology(bike_toy_config(), 0, ticks, transfer_seed=128), 10)
        env_steps, ep, t0 = 0, 0, time.perf_counter()
        while env_steps < args.steps * 1024 and time.perf_counter() - t0 < 60:
            o.reset()
            env_steps += o.run_episode(1)[0]
            ep += 1
        dt = time.perf_counter() - t0
        kind, sample, cores = "port", f"{ep} episodes of oracle/bike_oracle.c, 1 thread", 1
    value = env_steps / dt
    line.update({"value": value, "ms_per_step": 1000.0 * dt / max(1, args.steps),
                 "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
                 "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    emit(line)


def run_reference_vm(args, line, ref_root, cores):
    """vm_scheduling: the unmodified reference (VectorEnv over every host core, best-fit agent of
    examples/vm_scheduling/rule_based_algorithm/best_fit.py) on the same synthetic trace; else the C port."""
    import numpy as np

    conf, ticks = vm_workload(args)
    line["config"] = {"workload": f"vm_scheduling synthetic azure.2019.10k-scale trace ({args.vm_count} VMs, 100 PMs, {ticks} ticks), best-fit agent",
                      "replicas": cores}
    line["dtype"] = "int32+f64"
    if reference_built():
        import yaml

        os.environ["SKIP_DEPLOYMENT"] = "TRUE"
        sys.path.insert(0, ref_root)
        sys.path.insert(1, os.path.join(ref_root, "_stubs"))
        from maro.simulator.scenarios.vm_scheduling import AllocateAction
        from maro.vector_env import VectorEnv

        cdir = os.path.dirname(conf["VM_TABLE"])
        with open(os.path.join(cdir, "config.yml"), "w") as fp:
            yaml.safe_dump(conf, fp, sort_keys=False)
        with VectorEnv(batch_num=cores, scenario="vm_scheduling", topology=cdir, durations=ticks) as env:
            def agent(decisions):
                acts = {}
                frames = env.frame_index
                for i, d in enumerate(decisions):
                    if d is None:
                        continue
                    info = env.snapshot_list["pms"][frames[i]:d.valid_pms:["cpu_cores_capacity", "cpu_cores_allocated"]][i]
                    info = np.asarray(info).reshape(-1, 2)
                    acts[i] = AllocateAction(vm_id=d.vm_id, pm_id=d.valid_pms[int(np.argmin(info[:, 0] - info[:, 1]))])
                return acts

            metrics, decisions, done = env.step(None)
            env_steps = 0
            t0 = None
            for k in range(args.warmup + args.steps):
                if k == args.warmup:
                    t0, env_steps = time.perf_counter(), 0
                if done:
                    env.reset()
                    metrics, decisions, done = env.step(None)
                else:
                    metrics, decisions, done = env.step(agent(decisions))
                env_steps += cores
            dt = time.perf_counter() - t0
        kind, sample = "reference", f"VectorEnv(batch_num={cores}) x {args.steps} steps of one episode, static backend"
    else:
        from maro_b200.scenarios.vm_scheduling.data import build_vm_topology
        from oracle.vm_oracle import VmOracle

        o = VmOracle(build_vm_topology(conf, 0, ticks), 1, 8)
        env_steps, ep, t0 = 0, 0, time.perf_counter()
        while env_steps < args.steps * 1024 and time.perf_counter() - t0 < 60:
            o.reset()
            env_steps += o.run_episode(1)[0]
            ep += 1
        dt = time.perf_counter() - t0
        kind, sample, cores = "port", f"{ep} episodes of oracle/vm_oracle.c, 1 thread", 1
    value = env_steps / dt
    line.update({"value": value, "ms_per_step": 1000.0 * dt / max(1, args.steps),
                 "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
                 "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    emit(line)


# ----------------------------------------------------------------------------------------------- our arm
def _all_cores(make_oracle, run_one, seconds):
    """`cores` host threads, each with its own oracle replica, run whole episodes for `seconds` (ctypes releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor

    cores = os.cpu_count() or 1
    oracles = [make_oracle() for _ in range(cores)]

    def work(k):
        o, steps, eps, t0 = oracles[k], 0, 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            o.reset()
            steps += run_one(o, k * 100003 + eps)
            eps += 1
        return steps, eps

    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        res = list(ex.map(work, range(cores)))
    dt = time.perf_counter() - t0
    return sum(r[0] for r in res) / dt, cores, sum(r[1] for r in res)


def _one_thread(make_oracle, run_one, seconds):
    o, steps, eps, t0 = make_oracle(), 0, 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        o.reset()
        steps += run_one(o, eps)
        eps += 1
    return steps / (time.perf_counter() - t0), eps, steps


def reference_inprocess(scenario, topology, ticks, seconds):
    """BASELINE.md §2: the unmodified reference's single in-process Env loop (no VectorEnv pipes), static and dynamic
    backends, one host core each; tools/ref_inprocess.py in a fresh process per backend (the backend is an import-time choice)."""
    import subprocess

    out = {}
    if not reference_built():
        return out
    for backend in ("static", "dynamic"):
        try:
            p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_inprocess.py"), scenario, topology, str(ticks),
                                str(seconds), backend], capture_output=True, text=True, timeout=120 + 4 * seconds)
            out[backend] = json.loads(p.stdout.strip().splitlines()[-1])
        except Exception as ex:  # pragma: no cover
            out[backend] = {"error": repr(ex)[:200]}
    return out


def _baseline(args, make_oracle, run_one, what, scenario, topology, ticks):
    """cpu_baseline object: `value` = the C port of the reference on ALL host cores (one replica per thread), next to the
    same port on one thread and the unmodified reference's in-process Env loop (static / dynamic backend, one core)."""
    if args.cpu_seconds <= 0:
        return None
    sec = max(0.2, args.cpu_seconds)
    v1, ep1, st1 = _one_thread(make_oracle, run_one, sec / 2)
    vall, cores, eps = _all_cores(make_oracle, run_one, sec)
    out = {"value": vall, "unit": "env-steps/s", "cores": cores, "kind": "port",
           "sample": f"{eps} full episodes of {what} in {sec:.1f} s, one replica per host thread ({cores} threads), same workload / policy",
           "one_thread": {"value": v1, "cores": 1, "sample": f"{ep1} full episodes ({st1} env-steps)"}}
    if args.cpu_seconds >= 2 and not args.matrix:
        out["reference_inprocess"] = reference_inprocess(scenario, topology, ticks, min(6.0, args.cpu_seconds))
    return out


def cpu_baseline_port(args, topo):
    from oracle.cim_oracle import CimOracle

    return _baseline(args, lambda: CimOracle(topo), lambda o, ep: o.run_episode(1, 0, ep)[0], "oracle/cim_oracle.c",
                     "cim", args.topology, args.ticks)


def cpu_baseline_bike(args, topo):
    from oracle.bike_oracle import BikeOracle
    from tools.workloads import bike_toy_config_dir

    return _baseline(args, lambda: BikeOracle(topo, 10), lambda o, ep: o.run_episode(1)[0], "oracle/bike_oracle.c",
                     "citi_bike", bike_toy_config_dir(), topo.max_tick)


_HOST_AGENT = None


def load_host_agent():
    """Compile (gcc) and load tools/host_agent.c — the host-side agent of the e2e leg.  The library is built in a
    temporary directory, so that the benchmark writes nothing into the source tree (which may be read-only)."""
    global _HOST_AGENT
    if _HOST_AGENT is not None:
        return _HOST_AGENT
    import ctypes
    import subprocess
    import tempfile

    src = os.path.join(ROOT, "tools", "host_agent.c")
    with tempfile.TemporaryDirectory(prefix="maro_b200_bench_") as d:
        out = os.path.join(d, "libhost_agent.so")
        subprocess.check_call(["gcc", "-O2", "-fopenmp", "-pthread", "-shared", "-fPIC", src, "-o", out])
        lib = ctypes.CDLL(out)  # stays mapped after the directory is removed
    lib.agent_random.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32]
    lib.agent_greedy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.agent_best_fit.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                   ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    lib.agent_best_fit_row.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    _HOST_AGENT = lib
    return lib


def vm_workload(args):
    """(config dict, ticks) of the vm_scheduling bench workload: tools/vm_trace_gen.py trace + azure.2019.10k topology."""
    import tempfile

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import vm_trace_gen

    ticks = 8638 if args.ticks == 1000 else args.ticks
    d = args.vm_trace_dir
    if not d:  # a fresh directory per process (and so per rank), removed at exit
        import atexit
        import shutil

        d = tempfile.mkdtemp(prefix="maro_b200_vm_trace_")
        atexit.register(shutil.rmtree, d, True)
    vm_path, cpu_path = vm_trace_gen.generate(d, args.vm_count, ticks)
    return vm_trace_gen.azure_like_config(vm_path, cpu_path), ticks


def cpu_baseline_vm(args, topo, max_snapshots):
    from oracle.vm_oracle import VmOracle

    saved, args.matrix = args.matrix, True  # (no in-process reference leg: the reference needs ~5 min per episode here)
    try:
        return _baseline(args, lambda: VmOracle(topo, 1, max_snapshots), lambda o, ep: o.run_episode(1)[0],
                         "oracle/vm_oracle.c", "vm_scheduling", "", 0)
    finally:
        args.matrix = saved


def host_policy_numpy(dec, seed, base, np):
    """numpy-vectorised twin of cim_policy_kernel (uint32 arithmetic)."""
    def h(x):
        x = x.astype(np.uint32)
        x ^= x >> np.uint32(16); x *= np.uint32(0x7FEB352D); x ^= x >> np.uint32(15)
        x *= np.uint32(0x846CA68B); x ^= x >> np.uint32(16)
        return x
    B = dec.shape[0]
    rid = (np.arange(B, dtype=np.uint32) + np.uint32(base))
    with np.errstate(over="ignore"):
        h1 = h(np.uint32(seed) ^ h(rid * np.uint32(0x9E3779B9) + dec[:, 7].astype(np.uint32) * np.uint32(0x85EBCA6B) + np.uint32(0x1234567)))
        h2 = h(h1 + np.uint32(0x68BC21EB))
    load, dis = dec[:, 3], dec[:, 4]
    to_dis = (dis > 0) & ((h1 & 1) == 1)
    scope = np.where(to_dis, dis, load)
    qty = np.where(scope > 0, h2 % (scope.astype(np.uint32) + np.uint32(1)), 0).astype(np.int32)
    act = np.empty((B, 1, 4), np.int32)
    act[:, 0, 0] = dec[:, 2]; act[:, 0, 1] = dec[:, 1]; act[:, 0, 2] = qty; act[:, 0, 3] = to_dis
    return act


def _rl_extras(torch, env, dec, topo, B, stream):
    """device-resident RL shaping kernels + rollout loop timings (extras of the CIM line; not part of `value`)"""
    from maro_b200.rl_shaping import CimShaper

    shaper = CimShaper(env)
    t_ticks = torch.clamp(dec[:, 0] - 120, min=0).contiguous()
    t_ports = torch.remainder(dec[:, 1], topo.n_ports).to(torch.int32).contiguous()
    for _ in range(3):
        shaper.states(dec); shaper.rewards(t_ticks, t_ports)
    t_model = torch.remainder(dec[:, 7], 21).to(torch.int32).contiguous()
    shaper.env_actions(dec, t_model)
    sev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    reps = 20
    sev[0].record(stream)
    for _ in range(reps):
        shaper.states(dec)
    sev[1].record(stream)
    for _ in range(reps):
        shaper.rewards(t_ticks, t_ports)
    sev[2].record(stream)
    for _ in range(reps):
        shaper.env_actions(dec, t_model)
    sev[3].record(stream)
    torch.cuda.synchronize()
    a_us = 1000.0 * sev[2].elapsed_time(sev[3]) / reps
    s_us, r_us = 1000.0 * sev[0].elapsed_time(sev[1]) / reps, 1000.0 * sev[1].elapsed_time(sev[2]) / reps
    shaping = {"state_dim": shaper.state_dim, "states_us": s_us, "states_per_s": B / (s_us * 1e-6),
               "state_gbs": B * shaper.state_dim * 12 / (s_us * 1e-6) / 1e9,  # 8 B written + 4 B gathered per element
               "actions_us": a_us, "rewards_us": r_us, "rewards_per_s": B / (r_us * 1e-6),
               "reward_gbs": B * (shaper.time_window * 2 * 4 + 4) / (r_us * 1e-6) / 1e9,
               "what": "examples/cim/rl shaping (look_back 7, 99-tick decayed reward) for all replicas, L2 warm"}

    # device-resident rollout with a small MLP policy (state -> 171x256x21 MLP -> argmax -> action -> step; rewards after)
    from maro_b200.rl_rollout import CimDeviceRollout

    torch.manual_seed(0)
    mlp = torch.nn.Sequential(torch.nn.Linear(shaper.state_dim, 256), torch.nn.ReLU(), torch.nn.Linear(256, 21)).cuda()
    ro = CimDeviceRollout(env, lambda st: mlp(st * 1e-4).argmax(1), shaper, store_states=False)
    ro.run_episode(max_steps=50)
    torch.cuda.synchronize()
    runs = []
    for _ in range(3):  # one episode each, wall clock; the best of three (the loop is host-enqueued: a busy host core shows)
        t0 = time.perf_counter()
        traj = ro.run_episode()
        torch.cuda.synchronize()
        runs.append(time.perf_counter() - t0)
    dt = min(runs)
    shaping["rollout"] = {"env_steps_per_s": float(traj["valid"].sum().item()) / dt, "steps": int(traj["valid"].shape[0]),
                          "seconds": dt, "seconds_all_runs": runs, "cuda_graph": ro._graph is not None, "graph_error": ro.graph_error,
                          "what": "BatchedCimEnvSampler.collect: one episode, MLP policy on the same GPU, sync-free fixed-length loop "
                                  "in CUDA-graph chunks, rewards in one launch (wall clock)"}
    return shaping


def _facade_e2e(args, device, B, base):
    """The literal drop-in surface, measured: maro_b200.vector_env.VectorEnv.step with a Python list of `Action` objects (one
    per env, built by a Python agent from the `DecisionEvent`s) + one `snapshot_list` query per step — what a caller of the
    reference's VectorEnv (maro/vector_env/vector_env.py:131-217) does.  Python object construction per env dominates."""
    from maro_b200.scenarios.cim.common import Action, ActionType
    from maro_b200.vector_env import VectorEnv
    from tools.workloads import cim_policy_random

    n_steps = 60 if B <= 2048 else 12
    with VectorEnv(batch_num=B, scenario="cim", topology=args.topology, durations=args.ticks, device=device,
                   max_snapshots=args.max_snapshots or None) as env:
        metrics, decisions, done = env.step(None)
        t_agent = t_query = 0.0
        t0 = time.perf_counter()
        for k in range(n_steps):
            ta = time.perf_counter()
            acts = []
            for i, d in enumerate(decisions):
                if d is None:
                    acts.append(None)
                    continue
                v, p, q, t = cim_policy_random((d.tick, d.port_idx, d.vessel_idx, d.action_scope.load, d.action_scope.discharge), 0, base + i, k)
                acts.append(Action(v, p, q, ActionType.DISCHARGE if t else ActionType.LOAD))
            t_agent += time.perf_counter() - ta
            tq = time.perf_counter()
            tick = next(d.tick for d in decisions if d is not None)
            states = env.snapshot_list["ports"][tick::["empty", "full", "shortage"]]
            t_query += time.perf_counter() - tq
            metrics, decisions, done = env.step(acts)
            if done:
                break
        dt = time.perf_counter() - t0
        n = k + 1
    return {"value": n * B / dt, "unit": "env-steps/s", "steps": n, "us_per_step": 1e6 * dt / n,
            "python_agent_us_per_step": 1e6 * t_agent / n, "query_us_per_step": 1e6 * t_query / n,
            "query_floats_per_step": int(sum(len(x) for x in states)),
            "api": "maro_b200.vector_env.VectorEnv.step(list of Action) + snapshot_list['ports'][tick::attrs] (one batched query) per step; "
                   "Python agent building one Action per env"}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fp:
            return json.load(fp)
    except Exception:
        return {}


def _traffic(key):
    """per-launch DRAM bytes of the dominant kernel from the committed ncu capture of this config, if any"""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fp:
                t = json.load(fp).get(key)
            if t:
                return t.get("bytes_per_launch"), name
        except Exception:
            pass
    return None, None


def run_cim(args, rank, local_rank, world):
    """CIM arm.  `value`: resident rollouts — maro_cim_rollout_device fuses `chunk` env-steps per launch with the hashed
    hello-world agent as a device callback (replica blocks stay in shared memory; snapshot rows stream to the HBM ring).
    `e2e`: the host-buffer call maro_cim_step_pinned (resident session: command rows / decision rows through mapped
    pinned memory) with the agent on the host.  Episode ends come from the oracle's episode length and are checked against
    the DONE status column the device returns."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from maro_b200.batch import CimBatch
    from maro_b200.scenarios.cim.topology import build_topology, load_config
    from oracle.cim_oracle import CimOracle  # episode length only

    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B = args.replicas
    conf = load_config(args.topology)
    n_seeds = max(1, min(args.seeds, B))
    topos = [build_topology(conf, args.ticks, seed=int(conf["seed"]) + k) for k in range(n_seeds)]
    rt = (np.arange(B) % n_seeds).astype(np.int32) if n_seeds > 1 else None
    env = CimBatch(topos, B, device=local_rank, max_snapshots=args.max_snapshots or None, replica_topology=rt)
    topo = topos[0]
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    env.set_stream(stream.cuda_stream)
    dec = torch.zeros((B, 8), dtype=torch.int32, device="cuda")
    met = torch.zeros((B, 3), dtype=torch.int64, device="cuda")
    act = torch.zeros((B, 1, 4), dtype=torch.int32, device="cuda")
    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    base = rank * B
    status = dec[:, 6]

    def all_done():  # the `done` the reference's step returns: every replica answered DONE / FINISHED
        return bool((status != 0).all().item())

    # An episode takes the same number of batched env-steps whatever the actions (one per decision event, plus the final
    # one); with several seeds the longest counts, shorter replicas idle at DONE until the reset.
    spe = max(CimOracle(t).run_episode(0)[0] for t in topos)
    pos = {"i": 0}  # batched env-steps into the current episode

    def next_episode():
        """Env.reset once the episode is over (the first env-step of an episode ignores its action: generator start)"""
        if pos["i"] < spe:
            return 0
        env.reset()
        pos["i"] = 0
        return 1

    def check_done():
        """the status column read back: every replica reports DONE exactly when the planned episode ends"""
        assert all_done() == (pos["i"] == spe), f"episode end at env-step {pos['i']}, the oracle's episode has {spe}"

    # ------------------------------------------------------------------ value: fused resident rollouts
    def timed_rollouts(total_steps, chunk, timed):
        """exactly `total_steps` batched env-steps in launches of <= chunk that end at episode ends at the latest (the
        kernel stops a launch at DONE); returns (device ms incl. resets, kernel ms, launches)"""
        evs, launches, left = [], 0, total_steps
        while left > 0:
            if flush is not None and timed:
                flush.fill_(1)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(stream)
            launches += next_episode()
            n = min(chunk, left, spe - pos["i"])
            e[1].record(stream)
            env.rollout_device(dec.data_ptr(), met.data_ptr(), n, 1, 0, base)
            e[2].record(stream)
            launches += 1
            evs.append(e)
            left -= n
            pos["i"] += n
            check_done()
        torch.cuda.synchronize()
        return sum(e[0].elapsed_time(e[2]) for e in evs), sum(e[1].elapsed_time(e[2]) for e in evs), launches

    def timed_launch_per_step(total_steps, timed):
        evs, launches = [], 0
        for k in range(total_steps):
            if flush is not None and timed:
                flush.fill_(1)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(stream)
            launches += next_episode()
            env.random_policy_device(dec.data_ptr(), act.data_ptr(), 0, base)
            e[1].record(stream)
            env.step_device(dec.data_ptr(), met.data_ptr(), act.data_ptr())
            e[2].record(stream)
            launches += 2
            evs.append(e)
            pos["i"] += 1
            if k % 16 == 15 or pos["i"] == spe:  # (read back every 16 steps and at each episode end)
                check_done()
        torch.cuda.synchronize()
        return sum(e[0].elapsed_time(e[2]) for e in evs), sum(e[1].elapsed_time(e[2]) for e in evs), launches

    chunk = max(1, min(args.chunk, args.steps))
    warm = max(args.warmup, 3)
    primary = (lambda n, t: timed_launch_per_step(n, t)) if args.launch_per_step else (lambda n, t: timed_rollouts(n, chunk, t))
    primary(warm, False)
    c0 = env.counters().sum(0)
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    wall0 = time.perf_counter()
    total_ms, kernel_ms, launches = primary(args.steps, True)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    if world > 1:
        dist.barrier()
    c1 = env.counters().sum(0)
    d_steps, d_ticks, d_events, d_snaps = (int(x) for x in (c1 - c0))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"decisions": dec.cpu(), "metrics": met.cpu()}, rank, world)

    extras = {}
    if not args.skip_extras and not args.launch_per_step:  # the one-launch-per-Env.step path, for comparison
        env.reset()
        dec.zero_()
        pos["i"] = 0
        n = min(args.steps, 500)
        timed_launch_per_step(warm, False)
        k0 = env.counters().sum(0)
        ms, kms, _ = timed_launch_per_step(n, True)
        k1 = env.counters().sum(0)
        extras["launch_per_step"] = {"value": float(k1[0] - k0[0]) / (ms / 1000.0), "unit": "env-steps/s", "steps": n,
                                     "us_per_step": 1000.0 * ms / n, "kernel_us": 1000.0 * kms / n,
                                     "what": "cim_policy_kernel + cim_step_kernel per Env.step (stage-in / write-back every step)"}
    if not args.skip_extras:
        try:  # extras never take the contract line down with them
            env.reset()
            dec.zero_()
            env.step_device(dec.data_ptr(), met.data_ptr())
            extras["rl_shaping"] = _rl_extras(torch, env, dec, topo, B, stream)
        except Exception as ex:  # pragma: no cover
            extras["rl_shaping"] = {"error": repr(ex)}

    if not args.skip_extras:
        try:
            extras["facade_e2e"] = _facade_e2e(args, local_rank, B, base)
        except Exception as ex:  # pragma: no cover
            extras["facade_e2e"] = {"error": repr(ex)[:300]}

    # ------------------------------------------------------------------ e2e: host buffers, agent on the host
    # The loop is user code in C on top of the C ABI (tools/host_agent.c:e2e_loop_cim): per sub-batch wait for the decision
    # rows, run the agent, submit the actions.  n_sub = 1 is the lock-step loop (one maro_cim_step_pinned per step); with more
    # sub-batches the agent's work on one overlaps the device's work and the PCIe latency of the others.
    e2e, e2e_variants, e2e_errors = None, {}, {}
    if not args.skip_e2e:
        import ctypes as C

        from maro_b200 import _native

        agent_lib = load_host_agent()
        L = _native.lib()
        env.reset()
        p_act, p_nact, p_active, p_dec, p_met = env.pinned()
        dec_ptr, act_ptr = p_dec.ctypes.data, p_act.ctypes.data
        env.step_pinned(use_actions=False)
        agent_lib.agent_random(dec_ptr, act_ptr, B, 1, 0, base)
        assert np.array_equal(p_act, host_policy_numpy(p_dec, 0, base, np))  # host agent == device agent
        gran = env.pinned_granularity()
        n_e2e = min(max(args.steps, 200), 3000)
        fptr = lambda f: C.cast(f, C.c_void_p)
        agent_lib.e2e_loop_cim_mt.argtypes = [C.c_void_p] * 6 + [C.c_int] * 5 + [C.c_uint32, C.c_uint32, C.c_void_p]
        out3 = (C.c_double * 3)()

        def run_loop(n_sub, n_threads, n_steps):
            env.reset()
            k0 = env.counters().sum(0)
            rc = agent_lib.e2e_loop_cim_mt(env._h, fptr(L.maro_cim_submit_pinned), fptr(L.maro_cim_wait_pinned), fptr(L.maro_cim_reset),
                                           dec_ptr, act_ptr, B, gran, n_sub, n_threads, n_steps, 0, base, out3)
            if rc:
                raise RuntimeError(L.maro_last_error().decode())
            k1 = env.counters().sum(0)
            return {"steps": int(k1[0] - k0[0]), "seconds": out3[0], "agent_seconds": out3[1], "resets": int(out3[2]),
                    "calls": n_steps, "n_sub": n_sub, "n_threads": n_threads}

        if gran > 0:
            run_loop(1, 1, 50)  # warm-up
            cores = os.cpu_count() or 1
            combos = [(1, 1)] + [(ns, nt) for ns, nt in ((2, 1), (4, 1), (8, 1), (8, 2), (8, 4), (16, 4), (16, 8), (32, 8), (32, 16))
                                 if B // gran >= 2 * ns and nt <= max(1, cores // 2)]
            e2e_errors = {}
            for n_sub, n_threads in combos:
                try:
                    r = run_loop(n_sub, n_threads, min(n_e2e, 600))
                    e2e_variants[f"{n_sub}x{n_threads}"] = r["steps"] / r["seconds"]
                except RuntimeError as ex:  # one combination failing must not take the line down
                    e2e_errors[f"{n_sub}x{n_threads}"] = str(ex)[:200]
                    print("e2e combo failed:", n_sub, n_threads, ex, file=sys.stderr)
            best = max(e2e_variants, key=e2e_variants.get)
            bs, bt = (int(x) for x in best.split("x"))
            e2e = run_loop(bs, bt, n_e2e)
        else:  # batch too large to stay resident: lock-step calls of maro_cim_step_pinned from Python
            env.reset()
            cc0 = env.counters().sum(0)
            st_col = p_dec[:, 6]
            t_agent, resets = 0.0, 0
            t0 = time.perf_counter()
            for k in range(n_e2e):
                ta = time.perf_counter()
                agent_lib.agent_random(dec_ptr, act_ptr, B, 1, 0, base)  # the first step of an episode ignores its action
                t_agent += time.perf_counter() - ta
                env.step_pinned()
                if st_col[0] != 0 and (st_col != 0).all():
                    env.reset()
                    resets += 1
            dt = time.perf_counter() - t0
            cc1 = env.counters().sum(0)
            e2e = {"steps": int(cc1[0] - cc0[0]), "seconds": dt, "agent_seconds": t_agent, "calls": n_e2e, "resets": resets, "n_sub": 0,
                   "n_threads": 1}

    t = torch.tensor([total_ms, kernel_ms, wall * 1000.0, (e2e or {}).get("seconds", 0.0) * 1000.0], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([d_steps, d_ticks, d_events, d_snaps, (e2e or {}).get("steps", 0)], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        from maro_b200.parallel import gather_metrics  # the path's single collective (SURVEY.md §8e)

        gathered = gather_metrics(met, world * B)
        assert gathered.shape == (world * B, 3)
    total_ms, kernel_ms, wall_ms, e2e_ms = (float(x) for x in t.cpu())
    g_steps, g_ticks, g_events, g_snaps, g_e2e_steps = (int(x) for x in cnt.cpu())

    line = None
    if rank == 0:
        peaks = _peaks()
        peak = float(peaks.get("hbm_gbs", 6650.0))
        F = F_DECLARED.get(args.topology, env.frame_words * 4)  # SURVEY.md §8 frame bytes
        n_snap, n_ev = g_snaps / max(1, g_steps), g_events / max(1, g_steps)
        bytes_per_step = 2 * F + n_snap * F + 32 * n_ev + 64
        achieved = bytes_per_step * g_steps / world / (kernel_ms / 1000.0) / 1e9  # per GPU
        value = g_steps / (total_ms / 1000.0)
        snaps = args.max_snapshots or "all"
        kname = "cim_step_kernel" if args.launch_per_step else "cim_resident_kernel"
        traffic, traffic_src = _traffic(f"cim/{args.topology}/{B}/{kname}")
        mode = ("one launch per Env.step" if args.launch_per_step else
                f"resident rollouts, {chunk} env-steps fused per launch, agent as a device callback")
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": (f"CIM {args.topology}, {B} parallel envs per GPU, {args.ticks} ticks, random actions (hashed "
                                    f"hello-world agent), snapshot_resolution 1, max_snapshots {snaps}"),
                       "replicas_per_gpu": B, "distinct_seeds": n_seeds, "mode": mode,
                       "l2": "state resident (no flush)" if args.no_flush else "flushed between timed launches (256 MiB write)"},
            "ticks_per_s": g_ticks / (total_ms / 1000.0), "events_per_s": g_events / (total_ms / 1000.0), "wall_ms": wall_ms,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": kname,
                         "bytes_per_env_step": bytes_per_step, "n_snap": n_snap, "n_ev": n_ev,
                         "kernel_us_per_step": 1000.0 * kernel_ms / args.steps,
                         "launch_us": 1000.0 * kernel_ms / max(1, launches),
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650"},
            "clocks": clocks, "gpu_launches": launches,
        }
        if e2e:
            line["e2e"] = {"value": g_e2e_steps / (e2e_ms / 1000.0), "unit": "env-steps/s",
                           # session: one 16-byte command row in, one 64-byte tagged result line out per replica and step
                           "h2d_bytes_per_step": B * 16, "d2h_bytes_per_step": B * (64 if e2e["n_sub"] else 8 * 4 + 3 * 8),
                           "api": ("maro_cim_submit_pinned / maro_cim_wait_pinned (pinned host buffers; resident session) driven by the C "
                                   "host loop tools/host_agent.c:e2e_loop_cim_mt, agent on the host" if e2e["n_sub"] else
                                   "maro_cim_step_pinned (pinned host buffers) + tools/host_agent.c on the host"),
                           "sub_batches": e2e["n_sub"], "host_threads": e2e["n_threads"], "us_per_batch_step": 1000.0 * e2e_ms / e2e["calls"],
                           "agent_us_per_batch_step": 1e6 * e2e["agent_seconds"] / e2e["calls"],
                           "batch_steps": e2e["calls"], "resets": e2e["resets"],
                           "by_sub_batches_x_host_threads": {str(k): v for k, v in e2e_variants.items()}}
            if e2e_errors:
                line["e2e"]["errors"] = e2e_errors
        line.update(extras)
        line["cpu_baseline"] = cpu_baseline_port(args, topo) if world == 1 else None
    env.close()
    return line if rank == 0 else None


def run_ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist

    from maro_b200.batch import CimBatch
    from maro_b200.scenarios.cim.topology import build_topology
    from oracle.cim_oracle import CimOracle  # checker / cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B = args.replicas
    bike = args.scenario == "citi_bike"
    vm = args.scenario == "vm_scheduling"
    met_words = 16 if vm else 3
    if vm:
        from maro_b200.batch import VmBatch
        from maro_b200.scenarios.vm_scheduling.data import build_vm_topology
        from oracle.vm_oracle import VmOracle  # checker / cpu_baseline leg only

        conf, ticks = vm_workload(args)
        topo = build_vm_topology(conf, 0, ticks)
        vm_snaps = args.max_snapshots or 8  # the reference default (every frame) is 51 MB per replica at this size
        steps_per_episode = VmOracle(topo, 1, vm_snaps).run_episode(1)[0]
        env = VmBatch(topo, B, 1, vm_snaps, device=local_rank)
        dec_words = env.dec_words
        life = topo.vm_attr[:, 4].astype("int64")
        vm_avg_live = float(np.minimum(np.where(life <= 0, ticks, life), ticks - topo.vm_attr[:, 3]).sum()) / ticks
    elif bike:
        from maro_b200.batch import BikeBatch
        from oracle.bike_oracle import BikeOracle  # checker / cpu_baseline leg only
        from tools.workloads import bike_toy_config
        from maro_b200.scenarios.citi_bike.data import build_bike_topology

        ticks = min(args.ticks, 2880) if args.ticks != 1000 else 1440
        topo = build_bike_topology(bike_toy_config(), 0, ticks, transfer_seed=128)
        steps_per_episode = BikeOracle(topo, 10).run_episode(1)[0]
        env = BikeBatch(topo, B, 10, args.max_snapshots or None, device=local_rank)
        dec_words = env.dec_words
    else:
        topo = build_topology(args.topology, args.ticks)
        steps_per_episode = CimOracle(topo).run_episode(0)[0]  # decisions + final step (static for a given stop table)
        env = CimBatch(topo, B, device=local_rank, max_snapshots=args.max_snapshots or None)
        dec_words = 8
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    env.set_stream(stream.cuda_stream)
    dec = torch.zeros((B, dec_words), dtype=torch.int32, device="cuda")

    def agent_device():
        if vm:
            env.best_fit_policy_device(dec.data_ptr(), act.data_ptr())
        elif bike:
            env.greedy_policy_device(dec.data_ptr(), act.data_ptr())
        else:
            env.random_policy_device(dec.data_ptr(), act.data_ptr(), 0, base)
    met = torch.zeros((B, met_words), dtype=torch.int64, device="cuda")
    act = torch.zeros((B, 1, 4), dtype=torch.int32, device="cuda")
    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    base = rank * B
    pos = {"i": 0}

    def one_step(ev=None, flush_l2=True):
        """agent + step; Env.reset at an episode boundary (synchronous; part of the job).  The first step of an episode
        ignores its action (generator start, core.py:128), so the agent kernel always runs."""
        if pos["i"] > 0 and pos["i"] % steps_per_episode == 0:
            env.reset()
        if flush is not None and flush_l2:
            flush.fill_(1)
        if ev:
            ev[0].record(stream)
        agent_device()
        if ev:
            ev[1].record(stream)
        env.step_device(dec.data_ptr(), met.data_ptr(), act.data_ptr())
        if ev:
            ev[2].record(stream)
        pos["i"] += 1

    # citi_bike / vm_scheduling: fused rollouts (maro_bike_rollout_device / maro_vm_rollout_device: the scenario's rule-based agent as
    # a device callback), like the CIM arm
    fused = (bike or vm) and not args.launch_per_step
    launches = 2 * args.steps

    def timed_rollouts(total_steps, chunk, timed):
        """exactly `total_steps` batched env-steps in launches of <= chunk (the rule-based agent as a device callback) that
        end at episode ends at the latest (the kernel stops a launch at DONE); Env.reset at each episode end.  Returns (device ms incl. resets, kernel ms, launches)."""
        evs, n_launch, left = [], 0, total_steps
        while left > 0:
            if flush is not None and timed:
                flush.fill_(1)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(stream)
            if pos["i"] > 0 and pos["i"] % steps_per_episode == 0:
                env.reset()
                n_launch += 1
            n = min(chunk, left, steps_per_episode - pos["i"] % steps_per_episode)
            e[1].record(stream)
            env.rollout_device(dec.data_ptr(), met.data_ptr(), n)
            e[2].record(stream)
            n_launch += 1
            evs.append(e)
            left -= n
            pos["i"] += n
            done = bool((dec[:, 6] != 0).all().item())  # every replica reports DONE exactly when the planned episode ends
            assert done == (pos["i"] % steps_per_episode == 0), f"episode end at env-step {pos['i']}, the oracle's has {steps_per_episode}"
        torch.cuda.synchronize()
        return sum(e[0].elapsed_time(e[2]) for e in evs), sum(e[1].elapsed_time(e[2]) for e in evs), n_launch

    if fused:
        chunk = max(1, min(args.chunk, args.steps))
        timed_rollouts(max(args.warmup, 3), chunk, False)
    else:
        for _ in range(max(args.warmup, 3)):
            one_step()
    torch.cuda.synchronize()
    c0 = env.counters().sum(0)
    events = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(0 if fused else args.steps)]
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    wall0 = time.perf_counter()
    if fused:
        total_ms, kernel_ms, launches = timed_rollouts(args.steps, chunk, True)
    else:
        for k in range(args.steps):
            one_step(events[k])
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    if world > 1:
        dist.barrier()
    if not fused:
        total_ms = sum(e[0].elapsed_time(e[2]) for e in events)
        kernel_ms = sum(e[1].elapsed_time(e[2]) for e in events)
    c1 = env.counters().sum(0)
    d_steps, d_ticks, d_events, d_snaps = (int(x) for x in (c1 - c0))
    if args.dump_outputs:
        m = met.cpu().numpy()
        if vm:  # these slots hold float64 bit patterns: decode them as the metrics dict does (_abi.vm_metrics)
            from maro_b200._abi import VM_METRIC_FLOAT

            m = m.astype(np.float64)
            m[:, VM_METRIC_FLOAT] = met.cpu().numpy()[:, VM_METRIC_FLOAT].view(np.float64)
        dump_outputs(args.dump_outputs, {"decisions": dec.cpu(), "metrics": m}, rank, world)
    if fused:  # the extra legs below drive the per-step path from a fresh episode
        env.reset()
        dec.zero_()
        pos["i"] = 0

    # ---- CUDA-graph mode (extra): chunks of `graph_chunk` (agent + step) pairs replayed from one graph; L2 flushed
    # between chunks.  This is how a device-resident RL loop would drive the env (no per-step launch cost).
    graph_info = None
    if args.graph_chunk > 0:
        env.reset()
        pos["i"] = 0
        n = args.graph_chunk
        for _ in range(3):
            one_step(flush_l2=False)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=stream):
            for _ in range(n):
                agent_device()
                env.step_device(dec.data_ptr(), met.data_ptr(), act.data_ptr())
        env.reset()
        done_in_ep = 0
        n_chunks = max(1, args.steps // n)
        gev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n_chunks)]
        torch.cuda.synchronize()
        g0 = env.counters().sum(0)
        for k in range(n_chunks):
            if done_in_ep + n > steps_per_episode:  # chunks never straddle an episode end
                env.reset()
                done_in_ep = 0
            if flush is not None:
                flush.fill_(1)
            gev[k][0].record(stream)
            gr.replay()
            gev[k][1].record(stream)
            done_in_ep += n
        torch.cuda.synchronize()
        g1 = env.counters().sum(0)
        gms = sum(a.elapsed_time(b) for a, b in gev)
        graph_info = {"steps": int(g1[0] - g0[0]), "ms": gms, "chunk": n}
        env.reset()
        pos["i"] = 0

    # ---- extra: device-resident RL state / reward shaping over the snapshot ring (SURVEY.md §8f rank 1), not part of `value`
    shaping = None
    if not bike and not vm:
        try:  # extras never take the contract line down with them
            shaping = _rl_extras(torch, env, dec, topo, B, stream)
        except Exception as ex:  # pragma: no cover
            shaping = {"error": repr(ex)}
        env.reset()
        pos["i"] = 0

    # ---- e2e: host-buffer C-ABI path, agent on the host, one episode-aligned run of min(steps, 2000) steps
    e2e = None
    if not args.skip_e2e:
        # Host-buffer path: the agent (tools/host_agent.c, gcc -fopenmp) reads the decision rows and writes the action
        # rows directly in the library's pinned staging buffers; maro_*_step_pinned moves them over PCIe (zero-copy
        # mapped memory for small batches, DMA copies for large ones) and runs the step kernel; every call synchronises.
        agent_lib = load_host_agent()
        p_act, p_nact, p_active, p_dec, p_met = env.pinned()
        dec_ptr, act_ptr = p_dec.ctypes.data, p_act.ctypes.data

        if vm:
            pm_nodes = np.arange(topo.n_pm)

        def host_agent():
            if vm and not args.vm_query_agent:  # best fit from the decision row's extension (remaining cores per valid PM)
                agent_lib.agent_best_fit_row(dec_ptr, act_ptr, B, 1, dec_words)
            elif vm:  # the reference agent's snapshot query (best_fit.py:38-44), batched over the replicas, then the argmin
                live = p_dec[:, 6] == 0
                frames = np.unique(p_dec[live, 2]).astype(np.int32) if live.any() else np.zeros(1, np.int32)
                q = env.query("pms", frames, pm_nodes, ["cpu_cores_capacity", "cpu_cores_allocated"])
                agent_lib.agent_best_fit(dec_ptr, act_ptr, B, 1, dec_words, q.ctypes.data, frames.ctypes.data, len(frames), topo.n_pm)
            elif bike:
                agent_lib.agent_greedy(dec_ptr, act_ptr, B, 1, dec_words)
            else:
                agent_lib.agent_random(dec_ptr, act_ptr, B, 1, 0, base)

        # cross-check the host agents against their twins once (the device agents are checked in tests/test_gpu_*)
        env.reset()
        env.step_pinned(use_actions=False)
        host_agent()
        if vm:
            chk = VmOracle(topo, 1, vm_snaps)
            _, od, _ = chk.step(None)
            assert p_act[0, 0].tolist() == chk.best_fit(od).tolist(), (p_act[0, 0], chk.best_fit(od))
        elif bike:
            from oracle.bike_oracle import policy_greedy
            assert p_act[0, 0].tolist() == policy_greedy(p_dec[0]).tolist()
        else:
            assert np.array_equal(p_act, host_policy_numpy(p_dec, 0, base, np))
        for k in range(3):
            env.step_pinned()
            host_agent()
        env.reset()
        n_e2e = min(args.steps, 2000)
        torch.cuda.synchronize()
        cc0 = env.counters().sum(0)
        t0 = time.perf_counter()
        i = 0
        t_agent = 0.0
        for k in range(n_e2e):
            if i == 0 and k > 0:
                env.reset()
            ta = time.perf_counter()
            host_agent()  # the first step of an episode ignores its action (generator start)
            t_agent += time.perf_counter() - ta
            env.step_pinned()
            i = (i + 1) % steps_per_episode
        dt = time.perf_counter() - t0
        cc1 = env.counters().sum(0)
        e2e = {"steps": int(cc1[0] - cc0[0]), "seconds": dt, "agent_seconds": t_agent}

    t = torch.tensor([total_ms, kernel_ms, wall * 1000.0, (e2e or {}).get("seconds", 0.0) * 1000.0,
                      (graph_info or {}).get("ms", 0.0)], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([d_steps, d_ticks, d_events, d_snaps, (e2e or {}).get("steps", 0),
                        (graph_info or {}).get("steps", 0)], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        # the path's single collective: collate per-replica episode metrics on every rank (SURVEY.md §8e)
        from maro_b200.parallel import gather_metrics

        gathered = gather_metrics(met, world * B)
        assert gathered.shape == (world * B, met_words)
    total_ms, kernel_ms, wall_ms, e2e_ms, graph_ms = (float(x) for x in t.cpu())
    g_steps, g_ticks, g_events, g_snaps, g_e2e_steps, g_graph_steps = (int(x) for x in cnt.cpu())

    line = None
    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fp:
                peaks = json.load(fp)
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        F = 180 if bike else F_DECLARED.get(args.topology, env.frame_words * 4)  # SURVEY.md §8 frame bytes
        n_snap = g_snaps / max(1, g_steps)
        n_ev = g_events / max(1, g_steps)
        bytes_per_step = 2 * F + n_snap * F + 32 * n_ev + 64
        if vm:
            # DESIGN.md §vm: per snapshot one frame row written; per tick every live VM's list entry (16 B) + its reading
            # (4 B + 1 B) read and the 5 dynamic PM attributes rewritten; per step the decision / metrics / action rows
            n_tick = g_ticks / max(1, g_steps)
            bytes_per_step = n_snap * F + n_tick * (21.0 * vm_avg_live + 20.0 * topo.n_pm) + dec_words * 4 + 128 + 16
        achieved = bytes_per_step * g_steps / world / (kernel_ms / 1000.0) / 1e9  # per GPU
        value = g_steps / (total_ms / 1000.0)
        snaps = args.max_snapshots or "all"
        traffic = None  # per-launch DRAM bytes of the dominant kernel from the committed ncu capture of this config, if any
        try:
            with open(os.path.join(ROOT, "profiles", "r1_traffic.json")) as fp:
                key = (f"vm_scheduling/azure-synth-{args.vm_count}/{B}" if vm else
                       f"{args.scenario}/{'toy.3s_4t' if bike else args.topology}/{B}")
                traffic = json.load(fp).get(key, {}).get("bytes_per_launch")
        except Exception:
            pass
        if vm:
            workload = (f"vm_scheduling synthetic azure.2019.10k-scale trace ({topo.n_vm} VMs, {topo.n_pm} PMs 32c/128G, {ticks} ticks; "
                        f"tools/vm_trace_gen.py), {B} parallel envs per GPU, best-fit agent, snapshot_resolution 1, max_snapshots {vm_snaps}")
        elif bike:
            workload = (f"citi_bike toy.3s_4t (frozen trace), {B} parallel envs per GPU, {topo.max_tick} ticks, greedy top-1 agent, "
                        f"snapshot_resolution 10, max_snapshots {snaps}")
        else:
            workload = (f"CIM {args.topology}, {B} parallel envs per GPU, {args.ticks} ticks, random actions (hashed hello-world "
                        f"agent), snapshot_resolution 1, max_snapshots {snaps}")
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32+f64" if vm else "int32", "data": "synthetic",
            "config": {"workload": workload,
                       "replicas_per_gpu": B, "l2": "state resident (no flush)" if args.no_flush else "flushed between timed steps (256 MiB write)",
                       "steps_per_episode": steps_per_episode},
            "ticks_per_s": g_ticks / (total_ms / 1000.0), "events_per_s": g_events / (total_ms / 1000.0),
            "wall_ms": wall_ms,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": ("vm_rollout_kernel" if fused else "vm_step_kernel") if vm else ("bike_step_kernel" if bike else "cim_step_kernel"), "bytes_per_env_step": bytes_per_step,
                         "n_snap": n_snap, "n_ev": n_ev, "kernel_us": 1000.0 * kernel_ms / args.steps,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650"},
            "clocks": clocks,
            "gpu_launches": launches,
        }
        if fused:
            line["config"]["mode"] = (f"fused rollouts, {chunk} env-steps per launch, "
                                      f"{'best-fit' if vm else 'greedy'} agent as a device callback")
        if e2e:
            line["e2e"] = {"value": g_e2e_steps / (e2e_ms / 1000.0), "unit": "env-steps/s",
                           "h2d_bytes_per_step": B * 16, "d2h_bytes_per_step": B * (dec_words * 4 + met_words * 8) + (B * topo.n_pm * 16 if vm and args.vm_query_agent else 0),
                           "api": (("maro_vm_step_pinned + maro_vm_query (the agent's snapshot query) + tools/host_agent.c on the host"
                                    if args.vm_query_agent else
                                    "maro_vm_step_pinned + tools/host_agent.c:agent_best_fit_row (decision-row extension) on the host") if vm else
                                   "maro_%s_step_pinned (pinned host buffers) + tools/host_agent.c on the host" % ("bike" if bike else "cim")),
                           "us_per_call": 1000.0 * e2e_ms / max(1, min(args.steps, 2000)),
                           "agent_us_per_call": 1e6 * e2e["agent_seconds"] / max(1, min(args.steps, 2000))}
        if shaping:
            line["rl_shaping"] = shaping
        if graph_info:
            line["graph_mode"] = {"value": g_graph_steps / (graph_ms / 1000.0), "unit": "env-steps/s",
                                  "chunk_steps": graph_info["chunk"], "us_per_step": 1000.0 * graph_ms / max(1, (args.steps // graph_info["chunk"]) * graph_info["chunk"]),
                                  "l2": "flushed between graph chunks"}
        line["cpu_baseline"] = (cpu_baseline_vm(args, topo, vm_snaps) if vm else
                                (cpu_baseline_bike(args, topo) if bike else cpu_baseline_port(args, topo))) if world == 1 else None
    env.close()
    return line if rank == 0 else None


def main():
    # Native libraries (NCCL's version banner, ...) write to file descriptor 1 behind Python's back.  Keep the original
    # stdout for the JSON line only and send everything else that targets fd 1 to stderr.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run = lambda a: run_cim(a, rank, local_rank, world) if a.scenario == "cim" else run_ours(a, rank, local_rank, world)
    if not args.matrix:
        line = run(args)
    else:
        # north-star matrix: {CIM toy.4p_ssdd_l0.0, citi_bike toy.3s_4t} x {1 k, 8 k, 64 k} envs per GPU; short runs of the same
        # legs as the default line (value / e2e / roofline / cpu_baseline); the first entry is the headline configuration
        import copy

        entries = []
        sizes = [int(x) for x in args.matrix_sizes.split(",") if x]
        for scenario in ("cim", "citi_bike"):
            for B in sizes:
                a = copy.copy(args)
                a.scenario, a.replicas, a.skip_extras, a.graph_chunk = scenario, B, True, 0
                a.topology, a.ticks = "toy.4p_ssdd_l0.0", 1000
                a.cpu_seconds = min(args.cpu_seconds, 3.0) if B == sizes[0] else 0.0
                a.dump_outputs = args.dump_outputs if (scenario, B) == ("cim", sizes[0]) else ""
                try:
                    ln = run(a)
                except Exception as ex:  # one configuration failing (e.g. out of memory) must not lose the others
                    ln = {"error": repr(ex)[:300], "config": {"workload": f"{scenario} {B} envs"}}
                if ln is not None:
                    ln["scenario"], ln["replicas_per_gpu"] = scenario, B
                    entries.append(ln)
        line = None
        if rank == 0:
            line = dict(entries[0])
            line["matrix"] = [{k: e.get(k) for k in ("scenario", "replicas_per_gpu", "value", "unit", "n_gpus", "ms_per_step", "e2e",
                                                     "roofline", "cpu_baseline", "config", "steps", "error") if k in e}
                              for e in entries]
    if line is not None:
        emit(line)
    if world > 1:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
