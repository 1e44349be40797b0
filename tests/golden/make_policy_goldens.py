"""Writes tests/golden/scripted_policy_actions.npz: the actions the reference's scripted policies
(metaworld/policies/sawyer_*_policy.py) take when they drive the oracle restatement (oracle/tasks.py) closed loop, on
the five goals tests/test_oracle.py::test_reference_scripted_policy_succeeds_on_oracle uses.  Only episodes that reach
`success` are kept, up to and including the step that reaches it (an unsolved goal has no actions); the test replays
them open loop.

  python tests/golden/make_policy_goldens.py <reference checkout, the directory that holds the `metaworld` package>
"""
import os
import sys
import types
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(ROOT, "tests", "golden", "scripted_policy_actions.npz")
GOALS, SEED, MAX_STEPS = 5, 42, 500


def policies(reference_root):
    """The policies only, through a bare `metaworld` namespace (the package itself needs gymnasium / mujoco)."""
    pkg = types.ModuleType("metaworld")
    pkg.__path__ = [os.path.join(reference_root, "metaworld")]
    sys.modules["metaworld"] = pkg
    warnings.simplefilter("ignore")
    import metaworld.policies as MP
    return MP.ENV_POLICY_MAP


def record(task, policy):
    """-> one action array per goal, empty where the policy did not solve the goal within MAX_STEPS"""
    from oracle.tasks import TASKS
    from metaworld_b200 import benchmarks as B
    episodes = []
    for tk in B.make_tasks([task], False, seed=SEED, n_goals=GOALS):
        env = TASKS[task]()
        env.set_task_vec(tk.unpack()["rand_vec"], False)
        obs, _ = env.reset()
        actions = []
        for _ in range(MAX_STEPS):
            actions.append(np.clip(policy.get_action(obs.copy()), -1, 1).astype(np.float32))   # stored as float32
            obs, _, _, _, info = env.step(actions[-1])
            if info["success"]:
                break
        episodes.append(np.array(actions) if info["success"] else np.zeros((0, 4), np.float32))
    return episodes


def main(reference_root):
    sys.path.insert(0, ROOT)
    table = policies(reference_root)
    from oracle.tasks import TASKS
    out = {}
    for task in sorted(TASKS):
        eps = record(task, table[task]())
        out[task] = np.concatenate(eps)
        out[task + "/lengths"] = np.array([len(e) for e in eps], dtype=np.int64)
        print(f"{task}: {sum(len(e) > 0 for e in eps)}/{GOALS} goals solved, {len(out[task])} steps")
    np.savez_compressed(OUT, **out)


if __name__ == "__main__":
    main(os.path.abspath(sys.argv[1]))
