"""CPU suite: the REAL host code of `metaworld_b200` (benchmarks.make_tasks, MetaWorldVecEnv, evaluation) against the
REFERENCE's whole vector stack -- `gym.make_vec("Meta-World/MT10" | "ML10-train", ...)` from the reference package
running unmodified on oracle/refshim (gymnasium + mujoco stand-ins, see oracle/refshim/README.md).  Both sides step the
same float64 oracle physics (ours through tests/oracle_engine.py), so every difference is host logic: goal generation,
task selection streams, one-hot ids, TimeLimit / terminate-on-success, SAME_STEP autoreset, final_obs / final_info /
episode statistics, checkpoint format.

The reference is not part of this repository: what it returned to each test is stored under tests/golden/refstack/ and
replayed (tests/refreplay.py).  tests/golden/make_refstack_goldens.py re-records it from a reference checkout."""
import os
import types

import numpy as np
import pytest

KEYS = ("success", "near_object", "grasp_success", "grasp_reward", "in_place_reward", "obj_to_target", "unscaled_reward")
RECORD_FROM = os.environ.get("MW_REFSTACK_RECORD")      # a reference checkout: run it live and rewrite the recordings


@pytest.fixture
def ref(request):
    """`ref.gym` / `ref.metaworld`: the reference's gymnasium registry and metaworld package."""
    from refreplay import Session
    name = request.node.name.replace("[", "-").replace("]", "")
    if RECORD_FROM:
        from oracle import refshim
        metaworld = refshim.activate(RECORD_FROM)
        import gymnasium
        session = Session()
        yield session.root(types.SimpleNamespace(gym=gymnasium, metaworld=metaworld))
        session.save(name)
    else:
        session = Session.load(name)
        yield session.root()
        session.finish()


def _ours(kind, name, **kw):
    from metaworld_b200 import vector_env as V
    from metaworld_b200 import benchmarks as B
    from oracle_engine import OracleEngine
    names = {"MT10": B.MT10, "ML10": B.ML10["train"] * 2}.get(name, [name])
    eng = OracleEngine(list(dict.fromkeys(names)))
    return (V.make_mt_envs if kind == "mt" else V.make_ml_envs)(name, engine=eng, **kw)


def _compare_rollout(ref, ours, steps, seed, atol=2e-6):
    o1, i1 = ref.reset()
    o2, i2 = ours.reset()
    assert o1.shape == o2.shape and o1.dtype == o2.dtype and np.abs(o1 - o2).max() < atol
    n = o1.shape[0]
    rng = np.random.default_rng(seed)
    n_done = 0
    for t in range(steps):
        a = rng.uniform(-1, 1, size=(n, 4)).astype(np.float32)
        a[:, 3] = 1.0 if t % 7 > 3 else a[:, 3]
        r1 = ref.step(a)
        r2 = ours.step(a)
        assert r1[0].dtype == r2[0].dtype and np.abs(r1[0] - r2[0]).max() < atol, t
        assert r1[1].dtype == r2[1].dtype and np.abs(r1[1] - r2[1]).max() < 1e-5, t
        assert r1[2].dtype == r2[2].dtype and np.array_equal(r1[2], r2[2]) and np.array_equal(r1[3], r2[3]), t
        f1, f2 = r1[4], r2[4]
        assert set(f1) == set(f2), (t, sorted(f1), sorted(f2))
        for k in (KEYS if "success" in f1 else ()):
            assert np.abs(np.asarray(f1[k], dtype=np.float64) - f2[k]).max() < 1e-5 and np.array_equal(f1["_" + k], f2["_" + k])
        done = r1[2] | r1[3]
        assert ("final_obs" in f1) == ("final_obs" in f2) == bool(done.any())
        if done.any():
            n_done += int(done.sum())
            assert np.array_equal(f1["_final_obs"], f2["_final_obs"]) and np.array_equal(f1["_final_info"], f2["_final_info"])
            for e in np.nonzero(done)[0]:
                assert np.abs(f1["final_obs"][e] - f2["final_obs"][e]).max() < atol
            for e in np.nonzero(~done)[0]:
                assert f1["final_obs"][e] is None and f2["final_obs"][e] is None
            fi1, fi2 = f1["final_info"], f2["final_info"]
            for k in KEYS:
                assert np.abs(np.asarray(fi1[k], dtype=np.float64) - fi2[k]).max() < 1e-5 and np.array_equal(fi1["_" + k], fi2["_" + k])
            assert np.array_equal(fi1["episode"]["l"], fi2["episode"]["l"]) and np.allclose(fi1["episode"]["r"], fi2["episode"]["r"], atol=1e-3)
            assert np.array_equal(fi1["episode"]["_r"], fi2["episode"]["_r"]) and np.array_equal(fi1["_episode"], fi2["_episode"])
        # the task each sub-env is on (goal vector) follows the same stream
        rv1 = ref.get_attr("_last_rand_vec"); rv2 = ours.get_attr("_last_rand_vec")
        assert all(np.array_equal(x, y) for x, y in zip(rv1, rv2)), t
    return n_done


def test_mt10_one_hot_random_select_matches_reference_stack(ref):
    gym = ref.gym
    kw = dict(seed=42, use_one_hot=True, max_episode_steps=9, terminate_on_success=True, num_goals=3)
    ref = gym.make_vec("Meta-World/MT10", vector_strategy="sync", **kw)
    ours = _ours("mt", "MT10", **kw)
    assert ref.num_envs == ours.num_envs == 10
    assert ref.single_observation_space.shape == ours.single_observation_space.shape == (49,)
    assert ref.single_observation_space.dtype == ours.single_observation_space.dtype
    assert np.array_equal(ref.single_observation_space.low, ours.single_observation_space.low)
    assert ref.get_attr("task_name") is not None
    # goals (the _make_tasks legacy-RNG protocol, metaworld/__init__.py:114-179) are the reference's
    for tr, to in zip(ref.get_attr("tasks"), ours.get_attr("tasks")):
        assert len(tr) == len(to) == 3
        for a, b in zip(tr, to):
            from refreplay import unpickle
            assert np.array_equal(unpickle(a.data)["rand_vec"], b.unpack()["rand_vec"]) and a.env_name == b.env_name
    assert _compare_rollout(ref, ours, 30, seed=1) >= 30
    # evaluation protocol pieces used by metaworld/evaluation.py
    ref.call("toggle_terminate_on_success", False); ours.call("toggle_terminate_on_success", False)
    assert ref.get_attr("terminate_on_success") == ours.get_attr("terminate_on_success")
    _compare_rollout(ref, ours, 12, seed=2)
    # checkpoint: same ids, same keys, same task lists and RNG states; each side loads the other's
    c1, c2 = ref.call("get_checkpoint"), ours.call("get_checkpoint")
    for (id1, d1), (id2, d2) in zip(c1, c2):
        assert id1 == id2 and set(d1) <= set(d2) and d1["tasks"] != [] and d1["sample_tasks_on_reset"] == d2["sample_tasks_on_reset"]
        assert [t["env_name"] for t in d1["tasks"]] == [t["env_name"] for t in d2["tasks"]]
        assert d1["rng_state"] == d2["rng_state"] and d1["env_rng_state"]["np_random_state"] == d2["env_rng_state"]["np_random_state"]
    ours.call("load_checkpoint", list(c1))
    ref.call("load_checkpoint", list(c2))
    _compare_rollout(ref, ours, 12, seed=3)


def test_ml10_train_pseudorandom_partially_observable_matches_reference_stack(ref):
    gym = ref.gym
    metaworld = ref.metaworld
    kw = dict(seed=7, meta_batch_size=20, max_episode_steps=8)
    metaworld._N_GOALS = 4          # the ML entry points do not take num_goals (metaworld/__init__.py:631-654)
    ref = gym.make_vec("Meta-World/ML10-train", vector_strategy="sync", **kw)
    ours = _ours("ml", "ML10", split="train", num_goals=4, **kw)
    assert ref.num_envs == ours.num_envs == 20 and ref.single_observation_space.dtype == ours.single_observation_space.dtype == np.float64
    ref.call("sample_tasks"); ours.call("sample_tasks")
    assert ref.get_attr("sample_tasks_on_reset") == ours.get_attr("sample_tasks_on_reset") == tuple([False] * 20)
    _compare_rollout(ref, ours, 10, seed=5)
    for _ in range(3):          # no-collision cyclic sampling with reshuffle at wrap-around (wrappers.py:156-160)
        ref.call("sample_tasks"); ours.call("sample_tasks")
        assert all(np.array_equal(x, y) for x, y in zip(ref.get_attr("_last_rand_vec"), ours.get_attr("_last_rand_vec")))
    ref.call("toggle_sample_tasks_on_reset", True); ours.call("toggle_sample_tasks_on_reset", True)
    n = _compare_rollout(ref, ours, 18, seed=6)
    assert n >= 40
    o1, _ = ref.reset(); o2, _ = ours.reset()
    assert not o1[:, 36:].any() and not o2[:, 36:].any()


@pytest.mark.parametrize("extra", [dict(reward_normalization_method="gymnasium", normalize_observations=True),
                                   dict(recurrent_info_in_obs=True, normalize_observations=True, reward_normalization_method="exponential"),
                                   dict(recurrent_info_in_obs=True, normalize_reward_in_recurrent_info=False, reward_normalization_method="gymnasium")])
def test_normalisation_and_recurrent_wrappers_match_reference_stack(ref, extra):
    """The non-default per-sub-env wrappers of metaworld/__init__.py:437-446, autoresets included (the observation
    statistics see the terminal AND the reset observation of a finished env; the discounted return survives truncation)."""
    gym = ref.gym
    kw = dict(seed=11, use_one_hot=True, max_episode_steps=7, terminate_on_success=True, num_goals=2, **extra)
    ref = gym.make_vec("Meta-World/MT10", vector_strategy="sync", **kw)
    ours = _ours("mt", "MT10", **kw)
    assert ref.single_observation_space.shape == ours.single_observation_space.shape
    assert ref.single_observation_space.dtype == ours.single_observation_space.dtype
    # both sides run the same float64 physics, but ours passes observations through the engine interface as float32: the
    # 1e-7 rounding is amplified by 1 / sqrt(var) of slowly varying features
    assert _compare_rollout(ref, ours, 25, seed=4, atol=3e-4) >= 30


def test_mt1_single_task_vector_and_explicit_resets(ref):
    metaworld = ref.metaworld
    kw = dict(seed=3, max_episode_steps=6)
    metaworld._N_GOALS = 5
    # MT1 through the reference returns the single (wrapped) env of make_mt_envs; compare through our 1-env vector view
    renv = metaworld.make_mt_envs("door-open-v3", **kw)
    ours = _ours("mt", "door-open-v3", num_goals=5, **kw)
    o1, _ = renv.reset(); o2, _ = ours.reset()
    assert np.abs(o1 - o2[0]).max() < 2e-6
    rng = np.random.default_rng(0)
    for t in range(5):
        a = rng.uniform(-1, 1, 4).astype(np.float32)
        x1 = renv.step(a); x2 = ours.step(a[None])
        assert np.abs(x1[0] - x2[0][0]).max() < 2e-6 and abs(x1[1] - x2[1][0]) < 1e-5 and bool(x1[3]) == bool(x2[3][0])
    # explicit resets draw a new task each time, in the reference's order
    for _ in range(4):
        o1, _ = renv.reset(); o2, _ = ours.reset()
        assert np.abs(o1 - o2[0]).max() < 2e-6
        assert np.array_equal(renv.unwrapped._last_rand_vec, ours.get_attr("_last_rand_vec")[0])


def test_wrapped_single_env_across_truncations(ref):
    """gym.make("Meta-World/MT1") form (single=True): the TimeLimit step returns the terminal observation, stepping again
    raises, and reset() starts the task the reference's RandomTaskSelectWrapper draws -- three episodes, with and without
    the optional per-env wrappers (recurrent observation + exponential reward normalisation)."""
    metaworld = ref.metaworld
    metaworld._N_GOALS = 5
    for extra in ({}, dict(recurrent_info_in_obs=True, normalize_reward_in_recurrent_info=True), dict(use_one_hot=False, reward_normalization_method="exponential")):
        kw = dict(seed=11, max_episode_steps=5, **extra)
        renv = metaworld.make_mt_envs("drawer-open-v3", **kw)
        ours = _ours("mt", "drawer-open-v3", num_goals=5, single=True, **kw)
        o1, _ = renv.reset(); o2, _ = ours.reset()
        assert o1.shape == o2.shape and np.abs(o1 - o2).max() < 2e-6
        rng = np.random.default_rng(4)
        for ep in range(3):
            for t in range(5):
                a = rng.uniform(-1, 1, 4).astype(np.float32)
                x1 = renv.step(a); x2 = ours.step(a)
                assert np.abs(x1[0] - x2[0]).max() < 2e-6 and abs(x1[1] - x2[1]) < 1e-5, (extra, ep, t)
                assert bool(x1[2]) == x2[2] and bool(x1[3]) == x2[3] == (t == 4)
            with pytest.raises(ValueError):
                ours.step(a)
            o1, _ = renv.reset(); o2, _ = ours.reset()
            assert np.abs(o1 - o2).max() < 2e-6, (extra, ep)
            assert np.array_equal(renv.unwrapped._last_rand_vec, ours._last_rand_vec)


def test_bare_single_env_surface_matches_reference_class(ref):
    """`mt1.train_classes[name]()` + set_task / reset / step / evaluate_state and the attributes the reference's own tests
    read (tests/integration/test_new_api.py:18-45, tests/metaworld/envs/mujoco/sawyer_xyz/test_sawyer_xyz_env.py)."""
    metaworld = ref.metaworld
    from metaworld_b200 import benchmarks as B
    from metaworld_b200.single_env import SawyerXYZEnvB200
    from oracle_engine import OracleEngine
    metaworld._N_GOALS = 3
    name = "push-v3"
    rb = metaworld.MT1(name, seed=5)
    ob = B.MT1(name, seed=5, n_goals=3)
    assert list(rb.train_classes) == list(ob.train_classes) and repr(ob.train_classes[name]) == repr(rb.train_classes[name])
    renv = rb.train_classes[name]()
    oenv = SawyerXYZEnvB200(name, engine=OracleEngine([name]))
    assert oenv.task_name == renv.task_name and oenv.max_path_length == renv.max_path_length == 500
    assert oenv._partially_observable and renv._partially_observable
    with pytest.raises(RuntimeError):
        oenv.step(np.zeros(4, np.float32))
    with pytest.raises(RuntimeError):
        renv.step(np.zeros(4, np.float32))
    for rt, ot in zip(rb.train_tasks[:2], ob.train_tasks[:2]):
        renv.set_task(rt); oenv.set_task(ot)
        assert renv._partially_observable == oenv._partially_observable == False
        assert np.array_equal(renv.sawyer_observation_space.low, oenv.observation_space.low) and np.array_equal(renv.sawyer_observation_space.high, oenv.observation_space.high)
        o1, i1 = renv.reset(); o2, i2 = oenv.reset()
        assert o1.dtype == o2.dtype == np.float64 and np.abs(o1 - o2).max() < 2e-6 and i1 == i2 == {}
        assert np.array_equal(renv._last_rand_vec, oenv._last_rand_vec)
        assert np.abs(renv._target_pos - oenv._target_pos).max() < 1e-6 and np.abs(renv.obj_init_pos - oenv.obj_init_pos).max() < 1e-6
        rng = np.random.default_rng(1)
        for t in range(6):
            a = rng.uniform(-1, 1, 4).astype(np.float32)
            x1 = renv.step(a); x2 = oenv.step(a)
            assert np.abs(x1[0] - x2[0]).max() < 2e-6 and abs(x1[1] - x2[1]) < 1e-5 and x1[2] == x2[2] is False and x1[3] == x2[3]
            assert set(x1[4]) == set(x2[4]) and all(abs(float(x1[4][k]) - x2[4][k]) < 1e-5 for k in KEYS)
            assert renv.curr_path_length == oenv.curr_path_length == t + 1
        r1, f1 = renv.evaluate_state(x1[0], a); r2, f2 = oenv.evaluate_state(x2[0], a)
        assert abs(r1 - r2) < 1e-5 and all(abs(float(f1[k]) - f2[k]) < 1e-5 for k in KEYS)
    with pytest.raises(AssertionError):
        oenv.step(np.zeros(3, np.float32))


def test_goal_hidden_and_observable_envs_draw_the_reference_goal(ref):
    gymnasium = ref.gym
    from metaworld_b200.single_env import make_goal_env
    from oracle_engine import OracleEngine
    for observable, rid in ((False, "Meta-World/goal_hidden"), (True, "Meta-World/goal_observable")):
        renv = gymnasium.make(rid, env_name="drawer-open-v3", seed=11)
        oenv = make_goal_env("drawer-open-v3", seed=11, observable=observable, engine=OracleEngine(["drawer-open-v3"]))
        assert np.array_equal(renv._last_rand_vec, oenv._last_rand_vec) and renv._partially_observable == oenv._partially_observable == (not observable)
        a = np.array([0.3, -0.2, 0.1, 0.5], np.float32)
        x1 = renv.step(a); x2 = oenv.step(a)
        assert np.abs(x1[0] - x2[0]).max() < 2e-6 and (not x1[0][36:].any()) == (not observable)


def test_custom_mt_and_ml_entry_points_match_reference(ref):
    gym = ref.gym
    metaworld = ref.metaworld
    from metaworld_b200 import vector_env as V
    from oracle_engine import OracleEngine
    metaworld._N_GOALS = 3
    envs = ["reach-v3", "door-open-v3", "button-press-v3"]
    kw = dict(seed=9, use_one_hot=True, max_episode_steps=7)
    ref = gym.make_vec("Meta-World/custom-mt-envs", vector_strategy="sync", envs_list=envs, **kw)
    ours = V.make_custom_mt_envs(envs, engine=OracleEngine(envs), num_goals=3, **kw)
    assert _compare_rollout(ref, ours, 16, seed=4) >= 6
    tr, te = ["reach-v3", "push-v3"], ["door-open-v3"]
    kw = dict(seed=2, meta_batch_size=4, max_episode_steps=6)
    metaworld._N_GOALS = 4
    ref = gym.make_vec("Meta-World/custom-ml-envs", vector_strategy="sync", train_envs=tr, test_envs=te, **kw)
    ours = V.make_custom_ml_envs(tr, te, engine=OracleEngine(tr), num_goals=4, **kw)
    assert _compare_rollout(ref, ours, 14, seed=8) >= 8


def test_every_reference_id_has_an_entry_point(ref):
    """The ids the reference registers (metaworld/__init__.py:607-820) == the ids this package registers, and the entry
    points take the reference's argument names."""
    gym = ref.gym
    import metaworld_b200 as M
    from oracle_engine import OracleEngine
    ref_ids = {k.split("/", 1)[1] for k in gym.registry if k.startswith("Meta-World/")}
    table = M.entry_points()
    assert ref_ids == set(table), (sorted(ref_ids - set(table)), sorted(set(table) - ref_ids))
    for k, (single, vec) in table.items():
        spec = gym.registry["Meta-World/" + k]
        assert (single is not None) >= (spec.entry_point is not None) and (vec is not None) >= (spec.vector_entry_point is not None), k   # (MT1 additionally has a vector form here)
    v = table["MT10"][1](seed=1, use_one_hot=True, vector_strategy="sync", num_goals=2, engine=OracleEngine(M.MT10))
    assert v.num_envs == 10 and v.single_observation_space.shape == (49,)
    e = table["MT1"][0](env_name="reach-v3", seed=1, num_goals=2, engine=OracleEngine(["reach-v3"]))
    o, _ = e.reset()
    assert o.shape == (39,) and e.step(np.zeros(4, np.float32))[0].shape == (39,)
    ml = table["ML10-test"][1](seed=1, meta_batch_size=5, num_goals=2, engine=OracleEngine(M.ML10["test"]))
    assert ml.num_envs == 5 and ml.get_attr("terminate_on_success") == tuple([True] * 5)      # make_ml_envs_test (:603-605)
