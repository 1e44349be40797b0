"""CPU suite: the oracle (oracle/) against the reference's own importable pieces (committed golden vectors)
and against analytic invariants of the physics it restates.  No GPU."""
import copy
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gold():
    return json.load(open(os.path.join(GOLD, "reward_utils.json")))


def test_tolerance_matches_reference(gold):
    from oracle.sawyer_env import tolerance
    for x, lo, hi, m, sig, want in gold["tolerance"]:
        assert tolerance(x, (lo, hi), m, sig) == pytest.approx(want, rel=1e-12, abs=1e-15)


def test_hamacher_and_prism_match_reference(gold):
    from oracle.sawyer_env import hamacher_product, rect_prism_tolerance
    for a, b, want in gold["hamacher"]:
        assert hamacher_product(a, b) == pytest.approx(want, rel=1e-12, abs=1e-15)
    for c, z, o, want in gold["rect_prism"]:
        assert rect_prism_tolerance(np.array(c), np.array(z), np.array(o)) == pytest.approx(want, rel=1e-12)
    with pytest.raises(ValueError):
        hamacher_product(1.2, 0.5)


def test_quaternion_convention(gold):
    from oracle.sawyer_env import mat2quat_xyzw
    for R, q in gold["quat"]:
        assert np.allclose(mat2quat_xyzw(R), q, atol=1e-12)


def _free_model(dt):
    from metaworld_b200 import modelzoo
    m = copy.deepcopy(modelzoo.full_model("sawyer_reach_v3"))
    a = m.arrays
    a["dof_damping"][:] = 0
    a["geom_contype"][:] = 0
    a["geom_conaffinity"][:] = 0
    for k in ("eq_obj1id", "eq_obj2id", "eq_data", "eq_solref", "eq_solimp"):
        a[k] = a[k][:0]
    a["jnt_limited"][:] = 0
    a["actuator_kp"][:] = 0
    a["dof_armature"][:] = 0.001
    a["body_inertia"][m.names["body"].index("obj")] = [0.001, 0.002, 0.0005]
    m.opt["timestep"] = dt
    return m


def _energy_drift(dt, T=0.05):
    from oracle import mjphys as P
    m = _free_model(dt)
    a = m.arrays
    om = P.OModel(m)
    d = P.OData(om)

    def energy():
        P.mj_forward(om, d)
        M = d.qM.reshape(om.nv, om.nv)
        v = d.qvel
        return 0.5 * v @ M @ v + sum(a["body_mass"][b] * 9.81 * d.xipos.reshape(-1, 3)[b, 2] for b in range(om.nbody))

    rng = np.random.default_rng(0)
    d.qpos[:7] = rng.uniform(-1, 1, 7)
    d.qpos[1] = -1.5
    d.qvel[:] = rng.uniform(-1, 1, om.nv)
    d.qvel[9:12] = [0.3, 0.2, 1]
    d.qvel[12:15] = [3, -2, 1]
    e0 = energy()
    P.mj_step(om, d, int(round(T / dt)))
    return energy() - e0


def test_dynamics_energy_consistency():
    """Frictionless, undamped, unconstrained arm + tumbling free body: the energy error of the semi-implicit
    integrator must vanish linearly with dt (checks mass matrix, bias forces and free-joint integration together)."""
    d1, d2 = _energy_drift(2e-4), _energy_drift(1e-4)
    assert abs(d1) < 5e-3
    assert d1 / d2 == pytest.approx(2.0, rel=0.05)


def test_weld_tracks_mocap_and_object_rests():
    from oracle.tasks import TASKS
    env = TASKS["reach-v3"]()
    env.set_task_vec([0.05, 0.65, 0.02, -0.05, 0.85, 0.2], False)
    obs, _ = env.reset()
    assert np.allclose(obs[:3], [0, 0.6, 0.2], atol=5e-3)          # hand reached hand_init_pos
    assert np.allclose(obs[4:7], [0.05, 0.65, 0.02], atol=1e-9)    # object placed by _set_obj_xyz
    assert obs[36:39] == pytest.approx([-0.05, 0.85, 0.2])
    for _ in range(20):
        obs, r, term, trunc, info = env.step(np.zeros(4, np.float32))
    assert abs(obs[6] - 0.0194) < 1e-3                              # cylinder rests on the table (half height 0.02)
    f = [env.data.efc_force[c.efc_address] for c in env.data.contact if c.efc_address >= 0]
    assert len(f) >= 1 and abs(sum(f) - 0.75 * 9.81) < 1.5          # normal force ~ weight (rocking single contact)
    assert set(info) == {"success", "near_object", "grasp_success", "grasp_reward", "in_place_reward", "obj_to_target", "unscaled_reward"}


def test_reach_p_controller_succeeds():
    from oracle.tasks import TASKS
    env = TASKS["reach-v3"]()
    env.set_task_vec([0.0, 0.6, 0.02, 0.08, 0.88, 0.25], False)
    obs, _ = env.reset()
    ok = 0
    for _ in range(150):
        a = np.zeros(4, np.float32)
        a[:3] = np.clip((env._target_pos - obs[:3]) * 10, -1, 1)
        obs, r, term, trunc, info = env.step(a)
        ok = max(ok, info["success"])
    assert ok == 1.0 and r == pytest.approx(10.0)


def test_obs_layout_identities():
    """tests/helpers.py:4-33 of the reference: layout identities of the 39-vector."""
    from oracle.tasks import TASKS
    env = TASKS["reach-v3"]()
    env.set_task_vec([0.02, 0.62, 0.02, -0.08, 0.82, 0.1], False)
    prev, _ = env.reset()
    rng = np.random.default_rng(3)
    for _ in range(5):
        obs, *_ = env.step(rng.uniform(-1, 1, 4).astype(np.float32))
        assert np.all(obs[-3:] == env._target_pos)
        assert np.all(obs[:3] == env.get_endeff_pos())
        assert np.all(obs[4:7] == env._get_pos_objects()[:3])
        assert np.all(obs[18:36] == prev[:18])
        prev = obs
    with pytest.raises(ValueError):
        env.curr_path_length = 500
        env.step(np.zeros(4, np.float32))


def test_narrowphase_analytic_cases():
    """box-box / sphere-box / capsule-box / cylinder-box (GJK+EPA) against hand-computed configurations."""
    from metaworld_b200 import mjcf
    from oracle import mjphys as P
    import tempfile, textwrap
    xml = textwrap.dedent("""
    <mujoco><compiler angle="radian"/><option timestep="0.0025" cone="elliptic"/>
      <worldbody>
        <geom name="table" type="box" size="1 1 0.1" pos="0 0 -0.1" contype="0" conaffinity="1"/>
        <body name="b" pos="0 0 0.049"><freejoint/><geom name="bg" type="box" size="0.05 0.05 0.05" mass="1"/></body>
        <body name="s" pos="0.5 0 0.029"><freejoint/><geom name="sg" type="sphere" size="0.03" mass="1"/></body>
        <body name="c" pos="-0.5 0 0.019"><freejoint/><geom name="cg" type="capsule" size="0.02 0.1" euler="0 1.5707963267948966 0" mass="1"/></body>
        <body name="y" pos="0 0.5 0.039"><freejoint/><geom name="yg" type="cylinder" size="0.03 0.04" mass="1"/></body>
        <body mocap="true" name="mocap"/>
      </worldbody>
      <actuator><position joint="dummy1"/><position joint="dummy2"/></actuator>
    </mujoco>""")
    xml = xml.replace('<actuator><position joint="dummy1"/><position joint="dummy2"/></actuator>', "")
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "m.xml")
        open(p, "w").write(xml)
        m = mjcf.load(p)
    om = P.OModel(m)
    d = P.OData(om)
    P.mj_forward(om, d)
    cons = d.contact
    by = {}
    for c in cons:
        by.setdefault((m.names["geom"][c.geom1], m.names["geom"][c.geom2]), []).append(c)
    box = by[("table", "bg")]
    assert len(box) == 4 and all(abs(c.dist + 0.001) < 1e-9 for c in box)
    assert all(abs(abs(c.pos[0]) - 0.05) < 1e-9 and abs(abs(c.pos[1]) - 0.05) < 1e-9 for c in box)
    sph = by[("sg", "table")]
    assert len(sph) == 1 and abs(sph[0].dist + 0.001) < 1e-9 and abs(sph[0].frame[2] + 1) < 1e-9
    cap = by[("cg", "table")]
    assert len(cap) == 2 and all(abs(c.dist + 0.001) < 1e-9 for c in cap)
    assert sorted(round(c.pos[0], 6) for c in cap) == [-0.6, -0.4]
    cyl = by[("yg", "table")]
    assert len(cyl) == 1 and abs(cyl[0].dist + 0.001) < 1e-7 and abs(cyl[0].frame[2] + 1) < 1e-6
    assert abs(cyl[0].pos[0]) < 1e-6 and abs(cyl[0].pos[1] - 0.5) < 1e-6       # under the cylinder axis


def test_aligned_cylinder_fast_paths_agree_with_gjk_epa():
    """cyl_box_aligned / cyl_cyl_parallel (exact, used within 1.4 mrad of parallel) against the general GJK + EPA route on the
    same configuration tilted by 2 mrad (just outside the fast path): distance within r*tilt, normal within the tilt."""
    import ctypes as C
    from oracle import mjphys
    mjphys.build()
    L = C.CDLL(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "libmjphys.so"))
    dp = C.POINTER(C.c_double)

    def pair(t1, p1, R1, s1, t2, p2, R2, s2, margin=0.002):
        out = np.zeros(16 * 7); keep = [np.ascontiguousarray(x, dtype=np.float64) for x in (p1, R1.reshape(-1), s1, p2, R2.reshape(-1), s2)]
        L.om_narrowphase_pair.restype = C.c_int
        n = L.om_narrowphase_pair(C.c_int(t1), keep[0].ctypes.data_as(dp), keep[1].ctypes.data_as(dp), keep[2].ctypes.data_as(dp), None, C.c_int(0),
                                  C.c_int(t2), keep[3].ctypes.data_as(dp), keep[4].ctypes.data_as(dp), keep[5].ctypes.data_as(dp), None, C.c_int(0),
                                  C.c_double(margin), out.ctypes.data_as(dp))
        return out[: 7 * n].reshape(n, 7)

    def rot(ax, ang):
        ax = np.asarray(ax, float) / np.linalg.norm(ax)
        K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K

    CYL, BOX = 5, 6
    box = (np.array([0, 0, 0.05]), np.eye(3), [0.1, 0.06, 0.05])
    tilt = 2e-3
    cases = [((0.02, 0.01, 0.1 + 0.03 - 0.001), np.eye(3)),            # cap on the top face
             ((0.09, 0.0, 0.1 + 0.03 - 0.001), np.eye(3)),             # cap overhanging an edge
             ((0.1 + 0.02 - 0.0005, 0.0, 0.06), np.eye(3)),            # side against a vertical face
             ((0.0, 0.0, 0.1 + 0.02 - 0.001), rot([1, 0, 0], np.pi / 2)),   # lying on the top face
             ((0.03, 0.01, 0.08), np.eye(3))]                          # deep inside
    for pos, R in cases:
        a = pair(CYL, np.array(pos), R, [0.02, 0.03, 0], BOX, *box)
        b = pair(CYL, np.array(pos), rot([1, 0.7, 0], tilt) @ R, [0.02, 0.03, 0], BOX, *box)
        assert len(a) == 1 and len(b) == 1
        assert abs(a[0, 0] - b[0, 0]) < 0.03 * tilt + 2e-6 and np.abs(a[0, 4:] - b[0, 4:]).max() < 3 * tilt
    c1 = (np.array([0.3, 0, 0.25]), np.eye(3), [0.03, 0.03, 0])
    for pos in [(0.3, 0.0, 0.25 + 0.05 - 0.0008), (0.3 + 0.05 - 0.0005, 0, 0.25), (0.32, 0.01, 0.25 + 0.05 - 0.0008)]:
        a = pair(CYL, *c1, CYL, np.array(pos), np.eye(3), [0.02, 0.02, 0])
        b = pair(CYL, *c1, CYL, np.array(pos), rot([1, 0, 0], tilt), [0.02, 0.02, 0])
        assert len(a) == 1 and len(b) == 1
        assert abs(a[0, 0] - b[0, 0]) < 0.03 * tilt + 2e-6 and np.abs(a[0, 4:] - b[0, 4:]).max() < 3 * tilt


def _implemented():
    from oracle.tasks import TASKS
    return sorted(TASKS)


@pytest.mark.parametrize("task", _implemented())
def test_reference_scripted_policy_succeeds_on_oracle(task):
    """The reference's acceptance criterion for its physics+env stack (tests/metaworld/envs/mujoco/sawyer_xyz/
    test_scripted_policies.py:10-35: scripted policy success >= 80 %), applied to the oracle restatement.  The policies
    are the reference's and are not part of this repository: tests/golden/scripted_policy_actions.npz holds the actions
    they took driving the oracle closed loop on these goals (tests/golden/make_policy_goldens.py), for every goal they
    solved, and the oracle must reach `success` again on the last action of each."""
    from oracle.tasks import TASKS
    from metaworld_b200 import benchmarks as B
    if task == "basketball-v3":
        # Read literally, sawyer_basketball_v3.py:118-123 makes `_target_pos` a live view of data.site("goal").xpos and then
        # overwrites the site's LOCAL offset with that WORLD position, so the target the reward sees sits one hoop-offset away
        # from the hoop and the policy (which aims at the hoop) cannot trigger `success`.  The oracle follows the code as
        # written (DESIGN.md "Known reference quirks"); whether real MuJoCo bindings behave the same is part of "parity unpinned".
        pytest.xfail("basketball-v3: compounding goal-site write in the reference makes the scripted policy miss (see DESIGN.md)")
    with np.load(os.path.join(os.path.dirname(__file__), "golden", "scripted_policy_actions.npz")) as g:
        episodes = np.split(g[task], np.cumsum(g[task + "/lengths"])[:-1])
    wins = 0
    goals = B.make_tasks([task], False, seed=42, n_goals=5)
    for tk, actions in zip(goals, episodes):
        if not len(actions):        # the policy did not solve this goal
            continue
        env = TASKS[task]()
        env.set_task_vec(tk.unpack()["rand_vec"], False)
        obs, _ = env.reset()
        for a in actions:
            obs, r, _, _, info = env.step(a)
        wins += bool(info["success"])
    assert wins >= 4, f"{task}: scripted policy solved {wins}/5 goals on the oracle"


def _vee(S):
    return np.array([S[2, 1] - S[1, 2], S[0, 2] - S[2, 0], S[1, 0] - S[0, 1]]) / 2


def test_mass_matrix_equals_finite_difference_kinetic_energy():
    """qM against an independent construction: kinetic energy of every body from finite-differenced inertial-frame poses
    (door-open: hinge / slide joints only, so qpos can be perturbed directly)."""
    from oracle.tasks import TASKS
    from oracle import mjphys as P
    env = TASKS["door-open-v3"]()
    env.set_task_vec(np.array([0.05, 0.9, 0.15]), False)
    env.reset()
    rng = np.random.default_rng(0)
    q0 = np.array(env.data.qpos).copy()
    q0[:9] += rng.normal(size=9) * 0.2
    env.data.qpos = q0
    P.mj_forward(env.model, env.data)
    nv = len(env.data.qvel)
    M = np.array(env.data.qM).reshape(nv, nv)
    assert np.allclose(M, M.T, atol=1e-12) and np.linalg.eigvalsh(M).min() > 0
    from metaworld_b200 import modelzoo
    arr = modelzoo.full_model(env.xml).arrays
    mass = np.array(arr["body_mass"]); inertia = np.array(arr["body_inertia"]).reshape(-1, 3); armature = np.array(arr["dof_armature"])
    x0 = np.array(env.data.xipos).reshape(-1, 3).copy(); R0 = np.array(env.data.ximat).reshape(-1, 3, 3).copy()
    eps = 1e-6
    for _ in range(4):
        v = rng.normal(size=nv)
        env.data.qpos = q0 + eps * v
        P.mj_forward(env.model, env.data)
        x1 = np.array(env.data.xipos).reshape(-1, 3); R1 = np.array(env.data.ximat).reshape(-1, 3, 3)
        ke = 0.0
        for b in range(len(mass)):
            vc = (x1[b] - x0[b]) / eps
            w_world = _vee((R1[b] - R0[b]) @ R0[b].T) / eps
            w_body = R0[b].T @ w_world
            ke += 0.5 * mass[b] * vc @ vc + 0.5 * w_body @ (inertia[b] * w_body)
        ke += 0.5 * np.sum(armature * v * v)          # rotor inertia is part of qM but not of the bodies' motion
        assert abs(0.5 * v @ M @ v - ke) < 2e-5 * max(1.0, ke)


def test_constraint_solution_satisfies_dynamics_and_friction_cones():
    """At contact-rich states of the policy goldens: M qacc = qfrc_smooth + J^T f exactly (the solver's stationarity), contact
    normal forces are non-negative and friction stays inside the elliptic cone."""
    from oracle.tasks import TASKS
    from oracle import mjphys as P
    gold = os.path.join(os.path.dirname(__file__), "golden")
    checked = 0
    for task in ("pick-place-v3", "box-close-v3", "peg-insert-side-v3", "button-press-v3"):
        g = np.load(os.path.join(gold, f"traj_{task}.npz"))
        env = TASKS[task]()
        n = len(env.random_reset_space()[0])
        env.set_task_vec(g["p_rand_vec"][0][:n], False); env.reset()
        for t in range(20, g["p_qpos"].shape[1], 12):
            env.data.qpos = g["p_qpos"][0, t]; env.data.qvel = g["p_qvel"][0, t]; env.data.mocap_pos[0][:] = g["p_mocap"][0, t]
            a = g["p_actions"][0, t]; env.data.ctrl = (float(a[3]), -float(a[3]))
            P.mj_forward(env.model, env.data)
            nv, nefc = len(env.data.qvel), env.data.nefc
            M = np.array(env.data.qM).reshape(nv, nv)
            J = np.array(env.data.efc_J)[: nefc * nv].reshape(nefc, nv)
            f = np.array(env.data.efc_force)[:nefc]
            res = M @ np.array(env.data.qacc) - np.array(env.data.qfrc_smooth) - J.T @ f
            scale = max(1.0, np.abs(np.array(env.data.qfrc_smooth)).max(), np.abs(J.T @ f).max())
            assert np.abs(res).max() < 1e-6 * scale, (task, t, np.abs(res).max(), scale)
            for c in env.data.contact:
                if c.efc_address < 0:
                    continue
                fn = f[c.efc_address]
                assert fn >= -1e-9
                ft = f[c.efc_address + 1: c.efc_address + c.dim]
                fr = np.array(c.friction)[[0, 1, 2][: c.dim - 1]] if c.dim > 1 else np.zeros(0)
                if c.dim > 1 and fn > 0:
                    assert np.sqrt(np.sum((ft / np.maximum(fr, 1e-12)) ** 2)) <= fn * (1 + 1e-6) + 1e-9
                checked += 1
    assert checked > 50


def test_gravity_bias_equals_potential_gradient():
    """With qvel = 0 the bias force must be the gradient of the gravitational potential sum_b m_b g z_b (finite differences)."""
    from oracle.tasks import TASKS
    from oracle import mjphys as P
    from metaworld_b200 import modelzoo
    env = TASKS["drawer-open-v3"]()
    env.set_task_vec(np.array([0.0, 0.9, 0.0]), False); env.reset()
    mass = np.array(modelzoo.full_model(env.xml).arrays["body_mass"])
    rng = np.random.default_rng(1)
    q0 = np.array(env.data.qpos).copy(); q0[:9] += rng.normal(size=9) * 0.15
    nv = len(env.data.qvel)

    def potential(q):
        env.data.qpos = q; env.data.qvel = np.zeros(nv)
        P.mj_forward(env.model, env.data)
        return 9.81 * float(mass @ np.array(env.data.xipos).reshape(-1, 3)[:, 2])

    eps = 1e-6
    grad = np.array([(potential(q0 + eps * np.eye(nv)[i]) - potential(q0 - eps * np.eye(nv)[i])) / (2 * eps) for i in range(nv)])
    potential(q0)
    assert np.abs(np.array(env.data.qfrc_bias) - grad).max() < 1e-5 * max(1.0, np.abs(grad).max())


def test_contact_jacobian_is_the_rate_of_change_of_distance():
    """For every active contact: (J qvel)[normal row] = d(dist)/dt under the motion qvel, by finite differences on qpos
    (hinge / slide model); checks the contact frame orientation, the sign convention and the point Jacobians together."""
    from oracle.tasks import TASKS
    from oracle import mjphys as P
    gold = os.path.join(os.path.dirname(__file__), "golden")
    task = "button-press-topdown-v3"
    g = np.load(os.path.join(gold, f"traj_{task}.npz"))
    env = TASKS[task]()
    env.set_task_vec(g["p_rand_vec"][0][:3], False); env.reset()
    rng = np.random.default_rng(2)
    checked = 0
    for t in range(30, g["p_qpos"].shape[1], 10):
        q0 = g["p_qpos"][0, t].copy()
        env.data.qpos = q0; env.data.mocap_pos[0][:] = g["p_mocap"][0, t]
        P.mj_forward(env.model, env.data)
        nv, nefc = len(env.data.qvel), env.data.nefc
        J = np.array(env.data.efc_J)[: nefc * nv].reshape(nefc, nv).copy()
        base = {(c.geom1, c.geom2, tuple(np.round(c.pos, 4))): (c.dist, c.efc_address) for c in env.data.contact if c.efc_address >= 0}
        v = rng.normal(size=nv) * 0.5
        eps = 1e-7
        env.data.qpos = q0 + eps * v
        P.mj_forward(env.model, env.data)
        for c in env.data.contact:
            key = (c.geom1, c.geom2, tuple(np.round(c.pos, 4)))
            if key in base:
                d0, row = base[key]
                assert abs((c.dist - d0) / eps - J[row] @ v) < 2e-3 * max(1.0, np.abs(J[row]).sum()), (t, key)
                checked += 1
    assert checked >= 10


def test_drawer_close_golden_knife_edge():
    """Evidence for the drawer-close entry of tests/test_gpu.py::SENSITIVE_OPEN_LOOP.  Goal 0 of the committed golden rollout
    sits on a contact discontinuity: at step 2 the left claw (a box) grazes the drawer front (a box with exactly parallel
    faces) inside the 1 mm margin while moving at ~1 m/s, and which box-box feature pair fires - hence whether the full
    damping impulse is applied once more - flips back and forth under sub-micrometre displacements of the drawer.  The
    float64 oracle ITSELF answers displacements of 1e-7 .. 2e-6 m either with a change below 1e-7 or with a jump of
    1.08e-4 (measured here: +1.0e-7 -> -3e-9, +1.25e-7 -> +1.08e-4, +1.5e-7 -> -5e-9, +1e-6 -> +1.08e-4, +5e-6 -> -2e-7);
    float32 state noise (ulp 6e-8 at 0.6 m) cannot be expected to stay on the golden side."""
    from oracle.tasks import TASKS
    g = np.load(os.path.join(GOLD, "traj_drawer-close-v3.npz"))

    def drawer_y(dy):
        e = TASKS["drawer-close-v3"]()
        rv = g["rand_vec"][0][: len(e.random_reset_space()[0])].copy()
        rv[1] += dy
        e.set_task_vec(rv, False)
        e.reset()
        for t in range(3):
            o = e.step(g["actions"][0, t])[0]
        return o[5] - dy

    base = drawer_y(0.0)
    assert abs(base - g["obs"][0, 2][5]) < 1e-12
    resp = np.array([abs(drawer_y(d) - base) for d in np.geomspace(2e-8, 3e-6, 40)])
    assert (resp > 1e-4).sum() >= 3 and (resp < 2e-7).sum() >= 3         # both answers occur, interleaved (a jump already at 2e-8)
    assert not ((resp > 2e-7) & (resp < 1e-4)).any()                       # and nothing in between: a jump, not a slope
    assert abs(drawer_y(-1e-6) - base) < 1e-9                              # moving the drawer AWAY from the claw: no effect at all
