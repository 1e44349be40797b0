"""CPU suite: pins the oracle's Python restatement (oracle/sawyer_env.py, oracle/tasks.py) to the REFERENCE's own
classes.  tests/golden/traj_*.npz were produced by the reference's `metaworld/envs/sawyer_*_v3.py` running
unmodified on oracle/refshim (tests/golden/make_reference_goldens.py: "reference glue on restated physics"); the
restatement must reproduce them to 1e-12 on observations, rewards, ALL 7 info keys and the physics state, for random,
policy-driven, partially-observable and full-500-step trajectories."""
import glob
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TASKS = [os.path.basename(p)[5:-4] for p in sorted(glob.glob(os.path.join(GOLD, "traj_*.npz")))]
KEYS = ("success", "near_object", "grasp_success", "grasp_reward", "in_place_reward", "obj_to_target", "unscaled_reward")
TOL = 1e-12


def _oracle_env(task, rv, partial=False):
    from oracle.tasks import TASKS as OT
    env = OT[task]()
    env.set_task_vec(np.asarray(rv, dtype=np.float64), partial)
    return env


def _replay(env, g, pre, k, nrv):
    o, _ = env.reset()
    assert np.abs(o - g[pre + "reset_obs"][k]).max() <= TOL
    assert np.abs(env.data.qpos - g[pre + "reset_qpos"][k]).max() <= TOL
    for t, a in enumerate(g[pre + "actions"][k]):
        o, r, term, trunc, info = env.step(a)
        assert np.abs(o - g[pre + "obs"][k, t]).max() <= TOL, (pre, k, t)
        assert abs(float(r) - g[pre + "reward"][k, t]) <= TOL, (pre, k, t)
        got = np.array([float(info[x]) for x in KEYS])
        assert np.abs(got - g[pre + "info"][k, t]).max() <= TOL, (pre, k, t, got, g[pre + "info"][k, t])
        assert bool(trunc) == bool(g[pre + "truncated"][k, t])
        assert np.abs(env.data.qpos - g[pre + "qpos"][k, t]).max() <= TOL and np.abs(env.data.qvel - g[pre + "qvel"][k, t]).max() <= TOL


@pytest.mark.parametrize("task", TASKS)
def test_oracle_restatement_equals_reference_goldens(task):
    from metaworld_b200.tasks import TASKS as SPEC
    g = np.load(os.path.join(GOLD, f"traj_{task}.npz"))
    assert bytes(g["source"]).decode().startswith("reference glue")
    nrv = SPEC[task].rand_vec_len if hasattr(SPEC[task], "rand_vec_len") else None
    for pre, partial in (("", False), ("p_", False), ("po_", True), ("l_", False)):
        for k in range(len(g[pre + "rand_vec"])):
            rv = g[pre + "rand_vec"][k]
            rv = rv[:nrv] if nrv else _trim(task, rv)
            _replay(_oracle_env(task, rv, partial), g, pre, k, nrv)
    assert g["l_truncated"][0, -1] and not g["l_truncated"][0, :-1].any()        # sawyer_xyz_env.py:634
    assert not g["po_obs"][0, :, 36:].any() and not g["po_reset_obs"][0, 36:].any()   # :521-522 goal zeroed


def _trim(task, rv):
    from oracle.tasks import TASKS as OT
    lo, _ = OT[task]().random_reset_space()
    return rv[: len(lo)]


def test_all_50_tasks_have_reference_goldens():
    from metaworld_b200.tasks import TASKS as SPEC
    assert set(TASKS) == set(SPEC) and len(TASKS) == 50

