"""GPU (-m gpu): the reference's example code runs UNCHANGED on the CUDA core through the ``maro`` import shim
(maro_b200/shim.py) — VERDICT r1 missing #8 / next #5.

Each case runs tests/run_reference_script.py with ``maro_b200.shim.install()`` in a fresh process and compares what the
scripts print / collect with what they did on the unmodified reference:
  * examples/hello_world/cim/hello.py  (Env; reset(keep_seed=False) before each episode; random agent) — episode metrics
  * examples/vector_env/hello.py       (VectorEnv dict / list stepping, snapshot_list, reset)            — tick reports
  * examples/cim/rl                     (CIMEnvSampler on maro.rl's AbsEnvSampler.sample + DQN TrainingManager.train_step,
                                         maro/rl/rollout/env_sampler.py:391-520) — experiences, states, rewards, trained weights
What the reference printed / collected is stored in tests/golden/examples_golden.json (recorded from the reference by
``python tests/run_reference_script.py --mode reference --what <key>``), and the shim runs are compared with it.  The
example scripts and maro.rl are the reference's own code: oracle/build_ref.sh stages them under oracle/_ref, the example
scripts and the reference's Python sources (maro.rl is pure Python, and the shim replaces the compiled simulator) before
it compiles the package.  Where the package is compiled, the hello cases are also run on the reference itself and
compared live."""
import glob
import json
import os
import re
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SCRIPT = os.path.join(HERE, "run_reference_script.py")
HAVE_EXAMPLES = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "examples"))
HAVE_RL = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "maro", "rl"))  # maro.rl is pure Python: staged sources suffice
HAVE_REF = bool(glob.glob(os.path.join(ROOT, "oracle", "_ref", "maro", "backends", "frame*.so")))  # the runnable reference

pytestmark = pytest.mark.gpu


def run(mode, what, emulate=False):
    cmd = [sys.executable, SCRIPT, "--mode", mode, "--what", what] + (["--emulate"] if emulate else [])
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=HERE)
    assert p.returncode == 0, p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


def numbers(lines):
    return [[int(x) for x in re.findall(r"-?\d+", re.sub(r"np\.int64\((\d+)\)", r"\1", ln))] for ln in lines]


def golden(what):
    with open(os.path.join(HERE, "golden", "examples_golden.json")) as fp:
        return json.load(fp)[what]


def check_hello(what, emulate=False):
    ours = run("shim", what, emulate)
    assert numbers(ours["lines"]) == numbers(golden(what)["lines"]) and len(ours["lines"]) > 0
    if HAVE_REF:
        ref = run("reference", what)
        assert numbers(ours["lines"]) == numbers(ref["lines"])
    return ours


@pytest.mark.skipif(not HAVE_EXAMPLES, reason="oracle/_ref/examples not staged (oracle/build_ref.sh)")
def test_hello_world_cim_unchanged(emulate=False):
    ours = check_hello("hello_cim", emulate)
    assert ours["summary_has_node_mapping"]


@pytest.mark.skipif(not HAVE_EXAMPLES, reason="oracle/_ref/examples not staged (oracle/build_ref.sh)")
def test_vector_env_hello_unchanged(emulate=False):
    check_hello("hello_vector", emulate)


@pytest.mark.skipif(not (HAVE_RL and HAVE_EXAMPLES), reason="oracle/_ref (maro.rl + examples) not staged (oracle/build_ref.sh)")
def test_rl_toolkit_sampler_and_train_step_unchanged(emulate=False):
    ours, ref = run("shim", "rl_cim", emulate), golden("rl_cim")
    assert ours["env_class"] == "maro_b200.simulator.env" and ref["env_class"] == "maro.simulator.core"
    for k in ("n_experiences", "ticks", "states", "actions", "env_metric", "rewards", "policy_state"):
        assert ours[k] == ref[k], k
    assert abs(ours["reward_sum"] - ref["reward_sum"]) <= 1e-6 * max(1.0, abs(ref["reward_sum"]))
    assert ours["n_experiences"] > 300


@pytest.mark.skipif(not (HAVE_RL and HAVE_EXAMPLES), reason="oracle/_ref (maro.rl + examples) not staged (oracle/build_ref.sh)")
def test_batched_sampler_equals_the_reference_sampler_and_feeds_its_trainers():
    """SURVEY.md §8f rank 2 / VERDICT r1 next #8: ``BatchedCimEnvSampler.sample()`` (device-resident collection for all
    replicas, ExpElements materialised from the columns) against ``AbsEnvSampler.sample()`` of the reference run on the
    reference Env with the same per-port DQN policies (exploration off in both): the same transitions — ticks, agents,
    states, per-agent next states, actions, rewards (1e-6), terminal flags, the reward_eval_delay cut-off — as the real
    ``maro.rl.rollout.ExpElement`` objects; ``TrainingManager.record_experiences`` + ``train_step`` run on them."""
    ours, ref = run("shim", "rl_cim_batched"), golden("rl_cim_greedy")
    assert ours["exp_class"] == ref["exp_class"] == "maro.rl.rollout.env_sampler"
    for k in ("n_experiences", "ticks", "agents", "states", "agent_states", "next_agent_states", "actions", "terminals", "env_metric",
              "trained"):
        assert ours[k] == ref[k], k
    assert len(ours["rewards"]) == len(ref["rewards"]) > 300
    for a, b in zip(ours["rewards"], ref["rewards"]):
        assert abs(a - b) <= 1e-6 * max(1.0, abs(b)), (a, b)
