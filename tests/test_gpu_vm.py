"""GPU (-m gpu): the vm_scheduling CUDA path through the C ABI against reference traces, the oracle, and the
reference-facing Env / VectorEnv surfaces."""
import os
import tempfile

import numpy as np
import pytest

from vm_helpers import VM_CASES, assert_metrics_close, assert_vm_snapshots_equal, drive_vm, load_vm_golden, vm_topology

pytestmark = pytest.mark.gpu

EXACT_COLS = [0, 2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13]  # every metric except total_incomes (1) and total_profit (3)


def _row(dec, n_valid):
    """header + valid PM ids of a decision row; word 11 (offset of this build's remaining-cores extension) is not part of the
    reference's DecisionEvent and absent from the oracle's rows"""
    return list(dec[:11]) + list(dec[12:12 + n_valid])


@pytest.mark.parametrize("name", sorted(VM_CASES))
def test_vm_cuda_matches_reference_trace(name):
    from maro_b200.batch import VmBatch
    from oracle.vm_oracle import VmOracle

    spec = VM_CASES[name]
    topo = vm_topology(spec)
    gold = load_vm_golden(name)
    res, ms = spec.get("snapshot_resolution", 1), spec.get("max_snapshots")
    B = 3
    env = VmBatch(topo, B, res, ms, max_actions=2)

    def step_fn(act):
        if act is None:
            dec, met = env.step(None)
        else:
            a = np.zeros((B, 2, 4), np.int32)
            a[:, :1] = np.asarray(act, np.int32).reshape(1, 1, 4)
            dec, met = env.step(a, np.ones(B, np.int32))
        assert (dec == dec[0]).all() and (met == met[0]).all()
        return int(dec[0, 6]), dec[0].copy(), met[0].copy()

    rows, valid, mets, final, st, dec = drive_vm(step_fn, gold, topo.n_pm)
    assert rows.shape == gold["steps"].shape
    if not np.array_equal(rows, gold["steps"]):
        bad = np.argwhere(rows != gold["steps"])[0]
        raise AssertionError(f"step {bad[0]} col {bad[1]}: got {rows[bad[0]]} want {gold['steps'][bad[0]]}")
    assert np.array_equal(valid, gold["valid"])
    assert_metrics_close(mets, gold["metrics"], "per-step")
    assert_metrics_close(final, gold["final_metrics"], "final")
    assert env.ticks().tolist() == [int(gold["final_tick"])] * B and st == 1
    assert step_fn(None)[0] == 2
    assert env.snapshot_frames(B - 1).tolist() == gold["frames"].tolist()
    assert_vm_snapshots_equal(lambda f: env.snapshot_row(f, B - 1), gold, topo)
    # against the oracle: identical counters, frame words and energy metrics (float64 bit patterns)
    o = VmOracle(topo, res, ms)
    _, _, omets, ofinal, _, _ = drive_vm(lambda a: o.step(a), gold, topo.n_pm)
    assert np.array_equal(mets[:, EXACT_COLS], omets[:, EXACT_COLS])
    assert np.array_equal(final[EXACT_COLS], ofinal[EXACT_COLS])
    o.step(None)
    assert np.array_equal(env.counters()[B - 1], o.counters())
    assert np.array_equal(env.read_frame(B - 1), o.frame())
    env.close()


def test_vm_cuda_batch_best_fit_on_device_matches_oracle():
    """512 replicas, best-fit agent kernel, device-resident stepping; one replica replayed on the oracle."""
    import torch

    from maro_b200.batch import VmBatch
    from oracle.vm_oracle import VmOracle

    spec = VM_CASES["synth_160_tight_budget"]
    topo = vm_topology(spec)
    B = 512
    env = VmBatch(topo, B, 4, 16)
    env.set_stream(torch.cuda.current_stream().cuda_stream)
    dec = torch.zeros((B, env.dec_words), dtype=torch.int32, device="cuda")
    met = torch.zeros((B, 16), dtype=torch.int64, device="cuda")
    act = torch.zeros((B, 1, 4), dtype=torch.int32, device="cuda")
    o = VmOracle(topo, 4, 16)
    st, od, om = o.step(None)
    env.step_device(dec.data_ptr(), met.data_ptr())
    steps = 1
    while st == 0:
        d = dec.cpu().numpy()
        assert (d == d[0]).all()
        assert _row(d[0], od[10]) == _row(od, od[10]), steps
        env.best_fit_policy_device(dec.data_ptr(), act.data_ptr())
        a = act[0, 0].cpu().numpy()
        assert a.tolist() == o.best_fit(od).tolist()
        st, od, om = o.step(a.reshape(1, 4))
        env.step_device(dec.data_ptr(), met.data_ptr(), act.data_ptr())
        steps += 1
    torch.cuda.synchronize()
    m = met.cpu().numpy()
    assert (m == m[0]).all()
    assert np.array_equal(m[0][EXACT_COLS], om[EXACT_COLS])
    fm = m[0].view(np.float64)
    fo = om.view(np.float64)
    assert abs(fm[1] - fo[1]) <= 1e-9 * max(1.0, abs(fo[1])) and abs(fm[3] - fo[3]) <= 1e-9 * max(1.0, abs(fo[3]))
    assert dec.cpu().numpy()[:, 6].tolist() == [1] * B
    c = env.counters()
    assert (c == c[0]).all() and c[0].tolist() == o.counters().tolist() and c[0, 0] == steps
    assert np.array_equal(env.read_frame(B // 2), o.frame())
    env.close()


def _config_dir(spec):
    import yaml

    d = tempfile.mkdtemp()
    with open(os.path.join(d, "config.yml"), "w") as fp:
        yaml.safe_dump(spec["conf"], fp, sort_keys=False)
    return d


def test_vm_env_surface_replays_reference_trace():
    """maro.simulator.Env drop-in: AllocateAction / PostponeAction / DecisionEvent, metrics keys, snapshot_list query."""
    from maro_b200.scenarios.vm_scheduling import AllocateAction, DecisionEvent, PostponeAction
    from maro_b200.simulator import Env

    name = "synth_120_oversub_mixed"
    spec, gold = VM_CASES[name], load_vm_golden(name)
    env = Env("vm_scheduling", _config_dir(spec), durations=spec["durations"])
    assert env.agent_idx_list is None  # like the reference (its get_agent_idx_list has no body)
    assert env.summary["node_detail"]["pms"]["number"] == 8 and "cpu_utilization" in env.summary["node_detail"]["pms"]["attributes"]
    assert [p.cpu_cores_capacity for p in env.current_frame.pms] == [16] * 8 and env.current_frame.regions[0].total_machine_num == 8
    metrics, dec, done = env.step(None)
    k = 0
    while not done:
        assert isinstance(dec, DecisionEvent)
        g = gold["steps"][k]
        assert [env.tick, dec.vm_id, dec.frame_index, dec.vm_cpu_cores_requirement, dec.vm_memory_requirement, dec.vm_sub_id,
                int(dec.vm_category), dec.remaining_buffer_time, len(dec.valid_pms)] == g.tolist()
        assert dec.valid_pms == gold["valid"][k][:g[8]].tolist()
        assert metrics["total_vm_requests"] == int(gold["metrics"][k][0])
        assert metrics["total_latency"].due_to_agent == int(gold["metrics"][k][9])
        assert abs(metrics["total_energy_consumption"] - gold["metrics"][k][4]) <= 1e-12
        if k == 5:  # the pre-decision snapshot is queryable like the reference's (best_fit.py reads it)
            q = env.snapshot_list["pms"][env.frame_index:dec.valid_pms:["cpu_cores_capacity", "cpu_cores_allocated"]]
            want = np.stack([gold["pms/cpu_cores_capacity"], gold["pms/cpu_cores_allocated"]], -1)
            fi = gold["frames"].tolist().index(env.frame_index) if env.frame_index in gold["frames"].tolist() else None
            assert q.shape == (2 * len(dec.valid_pms),)
            assert (q.reshape(-1, 2)[:, 0] > 0).all()
            del want, fi
        a = gold["actions"][k]
        k += 1
        if a[1] < 0:
            action = None
        elif a[1] == 0:
            action = AllocateAction(vm_id=int(a[0]), pm_id=int(a[2]))
        else:
            action = PostponeAction(vm_id=int(a[0]), postpone_step=int(a[2]))
        metrics, dec, done = env.step(action)
    assert k == len(gold["steps"]) and env.tick == int(gold["final_tick"])
    fm = gold["final_metrics"]
    assert metrics["successful_allocation"] == int(fm[5]) and metrics["failed_allocation"] == int(fm[7])
    assert abs(metrics["total_profit"] - fm[3]) <= 1e-9
    assert env.step(None) == (None, None, True)
    with pytest.raises(Exception):
        env.reset()
        _, dec, _ = env.step(None)
        env.step(AllocateAction(vm_id=dec.vm_id + 99999, pm_id=0))
    env.close()


def test_vm_vector_env_two_envs_and_pinned_api(pinned=True):
    from maro_b200.scenarios.vm_scheduling import AllocateAction
    from maro_b200.vector_env import VectorEnv

    spec = VM_CASES["toy_5_first"]
    gold = load_vm_golden("toy_5_first")
    with VectorEnv(2, "vm_scheduling", _config_dir(spec), durations=spec["durations"]) as venv:
        metrics, events, done = venv.step(None)
        n = 0
        while not done:
            assert events[0].vm_id == events[1].vm_id == int(gold["steps"][n][1])
            n += 1
            metrics, events, done = venv.step([AllocateAction(e.vm_id, e.valid_pms[0]) for e in events])
        assert n == len(gold["steps"])
        assert_metrics_close([metrics[0][k] for k in ("total_vm_requests", "total_incomes", "energy_consumption_cost", "total_profit")],
                             gold["final_metrics"][:4])
        # dict stepping: only the named envs advance (vector_env.py:131-140)
        venv.reset()
        metrics, events, done = venv.step(None)
        first = [e.vm_id for e in events]
        metrics, events, done = venv.step({1: AllocateAction(events[1].vm_id, events[1].valid_pms[0])})
        assert len(events) == 1 and events[0].vm_id == int(gold["steps"][1][1])  # env 1 moved on, env 0 did not
        metrics, events, done = venv.step({0: AllocateAction(first[0], 0)})
        assert len(events) == 1 and events[0].vm_id == int(gold["steps"][1][1])
        assert events[0].valid_pms_remaining_cpu_cores is not None and len(events[0].valid_pms_remaining_cpu_cores) == len(events[0].valid_pms)
        if not pinned:  # (the CPU suite runs this test on the emulator-backed batch: no staging buffers there)
            return
        # zero-copy pinned staging buffers
        venv.reset()
        b = venv.batch
        actions, n_actions, active, decisions, mets = b.pinned()
        b.step_pinned(use_actions=False)
        assert decisions[:, 6].tolist() == [0, 0] and decisions[0, 1] == int(gold["steps"][0][1])
        actions[:, 0] = np.stack([[decisions[i, 1], 0, decisions[i, 12], 0] for i in range(2)])
        b.step_pinned(use_actions=True)
        assert decisions[0, 1] == int(gold["steps"][1][1]) and mets.shape == (2, 16)


def test_vm_cuda_full_size_episode_matches_oracle(tmp_path):
    """BASELINE config #5 size: 2 048 replicas, 10 000 VMs, 100 PMs, 8 638 ticks (synthetic azure.2019.10k-scale trace,
    tools/vm_trace_gen.py), best-fit agent kernel, the whole episode device-resident.  All replicas must agree, the
    request bookkeeping must balance, and the final metrics / frame / counters must equal the oracle's."""
    import sys

    import torch

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
    import vm_trace_gen

    from maro_b200.batch import VmBatch
    from maro_b200.scenarios.vm_scheduling.data import build_vm_topology
    from oracle.vm_oracle import VmOracle

    ticks = 8638
    vm_path, cpu_path = vm_trace_gen.generate(str(tmp_path), 10000, ticks)
    topo = build_vm_topology(vm_trace_gen.azure_like_config(vm_path, cpu_path), 0, ticks)
    assert topo.n_vm == 10000 and topo.n_pm == 100 and topo.error is None
    o = VmOracle(topo, 1, 8)
    n_steps, omet = o.run_episode(1)
    B = 2048
    env = VmBatch(topo, B, 1, 8)
    env.set_stream(torch.cuda.current_stream().cuda_stream)
    dec = torch.zeros((B, env.dec_words), dtype=torch.int32, device="cuda")
    met = torch.zeros((B, 16), dtype=torch.int64, device="cuda")
    act = torch.zeros((B, 1, 4), dtype=torch.int32, device="cuda")
    env.step_device(dec.data_ptr(), met.data_ptr())
    for k in range(n_steps - 1):
        env.best_fit_policy_device(dec.data_ptr(), act.data_ptr())
        env.step_device(dec.data_ptr(), met.data_ptr(), act.data_ptr())
        if k % 2500 == 0:
            d = dec.cpu().numpy()
            assert (d[:, 6] == 0).all() and (d == d[0]).all(), k
    torch.cuda.synchronize()
    d, m = dec.cpu().numpy(), met.cpu().numpy()
    assert d[:, 6].tolist() == [1] * B and (m == m[0]).all()
    assert np.array_equal(m[0][EXACT_COLS], omet[EXACT_COLS])
    fm, fo = m[0].view(np.float64), omet.view(np.float64)
    assert abs(fm[1] - fo[1]) <= 1e-9 * abs(fo[1]) and abs(fm[3] - fo[3]) <= 1e-9 * abs(fo[3])
    # every request ends up allocated or failed (none pending at the end of this trace); completions <= allocations
    assert m[0][0] == 10000 and m[0][5] + m[0][7] == m[0][0] and m[0][6] + m[0][8] <= m[0][5]
    c = env.counters()
    assert (c == c[0]).all() and c[0].tolist() == o.counters().tolist() and c[0, 0] == n_steps
    assert np.array_equal(env.read_frame(B - 1), o.frame())
    env.close()
    # ---- the same episode as fused rollouts (maro_vm_rollout_device: best-fit as a device callback), uneven launch lengths
    B2 = 296
    env2 = VmBatch(topo, B2, 1, 8)
    env2.set_stream(torch.cuda.current_stream().cuda_stream)
    dec2 = torch.zeros((B2, env2.dec_words), dtype=torch.int32, device="cuda")
    met2 = torch.zeros((B2, 16), dtype=torch.int64, device="cuda")
    done = 0
    for n in [1, 2, 777] + [2000] * 8:
        env2.rollout_device(dec2.data_ptr(), met2.data_ptr(), n)
        done += n
        if (dec2[:, 6] != 0).all().item():
            break
    assert done >= n_steps
    d2, m2 = dec2.cpu().numpy(), met2.cpu().numpy()
    assert d2[:, 6].tolist() == [1] * B2 and (m2 == m[0]).all()   # stopped at the DONE row, final metrics kept: bit-identical
    c2 = env2.counters()
    assert (c2 == c[0]).all()
    assert np.array_equal(env2.read_frame(B2 - 1), o.frame())
    assert env2.snapshot_frames(0).tolist() == env2.snapshot_frames(B2 - 1).tolist() and len(env2.snapshot_frames(0)) == 8
    env2.rollout_device(dec2.data_ptr(), met2.data_ptr(), 3)      # a further launch answers the all-zero FINISHED row
    assert (dec2.cpu().numpy()[:, 6] == 2).all() and (met2.cpu().numpy() == 0).all()
    env2.close()


def test_vm_cuda_large_hierarchy_of_the_reference_test_config():
    """The reference's own test topology (tests/data/vm_scheduling/config.yml shape: 2 regions / 2 zones / 3 data centres /
    8 clusters / 75 racks / 1130 PMs of two types) on the toy trace: CUDA path against the oracle, first-valid agent."""
    import yaml

    from maro_b200.batch import VmBatch
    from maro_b200.scenarios.vm_scheduling.data import build_vm_topology
    from oracle.vm_oracle import VmOracle
    from test_vm_oracle_golden import CONFIG_1130

    conf = yaml.safe_load(CONFIG_1130)
    conf["VM_TABLE"] = VM_CASES["toy_5_first"]["conf"]["VM_TABLE"]
    conf["CPU_READINGS"] = VM_CASES["toy_5_first"]["conf"]["CPU_READINGS"]
    topo = build_vm_topology(conf, 0, 5)
    assert topo.n_pm == 1130 and topo.error is None
    B = 6
    env, o = VmBatch(topo, B, 1, None), VmOracle(topo)
    (dec, met), (ost, odec, omet) = env.step(None), o.step(None)
    n = 0
    while ost == 0:
        assert (dec == dec[0]).all() and _row(dec[0], odec[10]) == _row(odec, odec[10]), n
        a = np.zeros((B, 1, 4), np.int32)
        a[:, 0] = [odec[1], 0, odec[12], 0]
        (dec, met), (ost, odec, omet) = env.step(a, np.ones(B, np.int32)), o.step(a[0])
        n += 1
    assert n > 0 and dec[:, 6].tolist() == [1] * B
    assert np.array_equal(met[0][EXACT_COLS], omet[EXACT_COLS])
    assert np.array_equal(env.read_frame(B - 1), o.frame())
    q = env.query("regions", [0], [0, 1], ["total_machine_num", "empty_machine_num"])[0].reshape(2, 2)
    assert q[:, 0].sum() == 1130
    env.close()
