"""CPU: the Python façades (maro_b200.simulator.Env, maro_b200.vector_env.VectorEnv, SnapshotList) driven exactly like
the GPU suite drives them (tests/test_gpu_env_surfaces.py — reference-style tests), with the CUDA batch replaced by the
host emulation of the same device code (tests/emul_batch.py).  Covers the host logic of the drop-in surfaces: action
encoding, DecisionEvent / metrics decoding, status handling, snapshot_list slicing, reset / set_seed / keep_seed
bookkeeping, list / dict / broadcast stepping."""
import pytest

import test_gpu_bike as bike_surfaces
import test_gpu_env_surfaces as surfaces
import test_gpu_vm as vm_surfaces
from emul_batch import EmulBikeBatch, EmulCimBatch, EmulVmBatch


@pytest.fixture(autouse=True)
def emulated_batch(monkeypatch):
    import maro_b200.simulator.env as env_mod
    import maro_b200.vector_env.vector_env as venv_mod

    for mod in (env_mod, venv_mod):
        monkeypatch.setattr(mod, "CimBatch", EmulCimBatch)
        monkeypatch.setattr(mod, "BikeBatch", EmulBikeBatch)
        monkeypatch.setattr(mod, "VmBatch", EmulVmBatch)
    yield


def test_env_hello_world_null_policy_emulated():
    surfaces.test_env_hello_world_null_policy()


def test_env_actions_pickle_reset_and_seed_emulated():
    surfaces.test_env_actions_pickle_reset_and_seed()


def test_vector_env_like_reference_test_emulated():
    surfaces.test_vector_env_like_reference_test()


def test_env_reset_new_seed_matches_reference_emulated():
    surfaces.test_env_reset_new_seed_matches_reference()


def test_bike_env_surface_like_reference_tests_emulated(tmp_path):
    bike_surfaces.test_bike_env_surface_like_reference_tests(tmp_path)


def test_vm_env_surface_replays_reference_trace_emulated():
    vm_surfaces.test_vm_env_surface_replays_reference_trace()


def test_vm_vector_env_list_and_dict_stepping_emulated():
    vm_surfaces.test_vm_vector_env_two_envs_and_pinned_api(pinned=False)


def test_bike_vector_env_matches_the_env_facade_emulated(tmp_path):
    """VectorEnv("citi_bike") with two envs, list stepping with a greedy agent: every env's DecisionEvents / metrics equal the
    single-env façade's (and through it the reference trace the Env test replays)."""
    import os
    import shutil

    import yaml

    from maro_b200.scenarios.citi_bike.common import Action, DecisionType
    from maro_b200.simulator import Env
    from maro_b200.vector_env import VectorEnv

    src = os.path.join(bike_surfaces.GOLDEN, "bike_case_2")
    with open(os.path.join(src, "decision.yml")) as fp:
        conf = yaml.safe_load(fp)
    conf.update(trip_data=os.path.join(src, "trips.bin"), weather_data=os.path.join(src, "weathers.bin"),
                stations_init_data=os.path.join(src, "stations.csv"), distance_adj_data=os.path.join(src, "distance_adj.csv"))
    with open(tmp_path / "config.yml", "w") as fp:
        yaml.safe_dump(conf, fp)

    def agent(ev):
        best = max((kv for kv in ev.action_scope.items() if kv[0] != ev.station_idx), key=lambda kv: (kv[1], kv[0]), default=None)
        if best is None:
            return None
        return Action(ev.station_idx, best[0], best[1]) if ev.type == DecisionType.Supply else Action(best[0], ev.station_idx, best[1])

    env = Env("citi_bike", str(tmp_path), durations=30, options={"transfer_seed": 2})
    trace = []
    metrics, ev, done = env.step(None)
    while not done:
        trace.append((ev.tick, ev.station_idx, ev.frame_index, ev.type, dict(ev.action_scope), dict(metrics)))
        metrics, ev, done = env.step(agent(ev))
    final = dict(metrics)
    env.close()
    assert len(trace) > 5
    with VectorEnv(2, "citi_bike", str(tmp_path), durations=30, options={"transfer_seed": 2}) as venv:
        metrics, events, done = venv.step(None)
        for want in trace:
            assert not done
            for i in range(2):
                e = events[i]
                assert (e.tick, e.station_idx, e.frame_index, e.type, dict(e.action_scope), dict(metrics[i])) == want
                assert list(e.action_scope)[-1] == e.station_idx
            metrics, events, done = venv.step([agent(e) for e in events])
        assert done and events == [None, None] and [dict(m) for m in metrics] == [final, final]
        assert venv.step(None) == ([None, None], [None, None], True)


def test_vm_float_queries_are_lifted_to_the_reference_float64_values():
    """VmBatch.query: cpu_utilization / energy_consumption come back as the float64 values the reference's static backend
    holds (k / 100 and the energy model at k), not as the float32 words of the ring; unknown frames stay zero."""
    import numpy as np

    from vm_helpers import VM_CASES, load_vm_golden, vm_topology

    spec, gold = VM_CASES["synth_160_bestfit"], load_vm_golden("synth_160_bestfit")
    topo = vm_topology(spec)
    b = EmulVmBatch(topo, 1)
    b.step(None)
    for k in range(40):
        a = np.zeros((1, 1, 4), np.int32)
        a[0, 0] = gold["actions"][k]
        b.step(a, np.ones(1, np.int32))
    frames = b.snapshot_frames(0).tolist()[-3:]
    n = topo.n_pm
    q = b.query("pms", frames + [10 ** 6], np.arange(n), ["cpu_utilization", "pm_type", "energy_consumption"])[0].reshape(4, n, 3)
    assert (q[3] == 0).all()                                   # unknown frame -> zeros
    u = q[:3, :, 0]
    assert np.array_equal(u, np.rint(u * 100) / 100.0) and (u > 0).any()   # exact multiples of 0.01 in float64
    for f in range(3):
        for p in range(n):
            calib, busy, idle = topo.pmtype_power[int(q[f, p, 1])]
            x = min(1, u[f, p] / 100)
            assert q[f, p, 2] == ((idle + (busy - idle) * (2 * x - pow(x, calib))) / topo.ticks_per_hour) / 1000
    only_e = b.query("pms", frames, np.arange(n), ["energy_consumption"])[0].reshape(3, n)
    assert np.array_equal(only_e, q[:3, :, 2])                 # energy alone: utilisation fetched behind the scenes


def test_reference_examples_run_unchanged_on_the_shim_emulated():
    """maro import shim: hello_world/cim/hello.py and vector_env/hello.py, unmodified"""
    import test_gpu_shim as shim_cases

    if not shim_cases.HAVE_EXAMPLES:
        pytest.skip("oracle/_ref/examples not staged (oracle/build_ref.sh)")
    shim_cases.test_hello_world_cim_unchanged(emulate=True)
    shim_cases.test_vector_env_hello_unchanged(emulate=True)


def test_rl_toolkit_runs_unchanged_on_the_shim_emulated():
    """maro import shim: the maro.rl CIM sampler + DQN train step of examples/cim/rl, unmodified"""
    import test_gpu_shim as shim_cases

    if not (shim_cases.HAVE_RL and shim_cases.HAVE_EXAMPLES):
        pytest.skip("oracle/_ref (maro.rl + examples) not staged (oracle/build_ref.sh)")
    shim_cases.test_rl_toolkit_sampler_and_train_step_unchanged(emulate=True)


def test_vector_env_reset_reseeds_like_the_reference_processes_emulated():
    surfaces.test_vector_env_reset_reseeds_like_the_reference_processes()


def test_dynamic_backend_query_layout_matches_the_reference_emulated(monkeypatch):
    surfaces.test_dynamic_backend_query_layout_matches_the_reference(monkeypatch)


def test_frame_dump_is_byte_identical_to_the_reference_emulated(tmp_path):
    surfaces.test_frame_dump_is_byte_identical_to_the_reference(tmp_path)
