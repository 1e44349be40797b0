"""CPU suite: host logic (task generation, lowering, sharding) and the C-ABI library's exported symbols. No GPU."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_make_tasks_protocol():
    from metaworld_b200 import benchmarks as B
    a = B.MT1("reach-v3", seed=42)
    b = B.MT1("reach-v3", seed=42)
    c = B.MT1("reach-v3", seed=43)
    va = np.array([t.unpack()["rand_vec"] for t in a.train_tasks])
    vb = np.array([t.unpack()["rand_vec"] for t in b.train_tasks])
    vc = np.array([t.unpack()["rand_vec"] for t in c.train_tasks])
    assert va.shape == (50, 6) and np.array_equal(va, vb) and not np.array_equal(va, vc)
    assert len(np.unique(va, axis=0)) == 50                      # tests/integration/test_new_api.py: 50 unique goals
    assert np.all(np.linalg.norm(va[:, :2] - va[:, 3:5], axis=1) >= 0.15)   # rejection rule, sawyer_reach_v3.py:127
    lo, hi = np.array([-0.1, 0.6, 0.02, -0.1, 0.8, 0.05]), np.array([0.1, 0.7, 0.02, 0.1, 0.9, 0.3])
    assert np.all(va >= lo) and np.all(va <= hi)
    assert not a.train_tasks[0].unpack()["partially_observable"]
    assert B.ML1("reach-v3", seed=1).train_tasks[0].unpack()["partially_observable"]
    # the global NumPy RNG is left untouched (reference restores it, metaworld/__init__.py:175-177)
    st = np.random.get_state()[1].copy()
    B.MT1("reach-v3", seed=7)
    assert np.array_equal(st, np.random.get_state()[1])


def test_make_tasks_matches_legacy_stream():
    """Same draws as np.random.seed(seed); np.random.uniform(low, high, size) twice per goal."""
    from metaworld_b200 import benchmarks as B
    from metaworld_b200.tasks import TASKS
    spec = TASKS["reach-v3"]
    st0 = np.random.get_state()
    np.random.seed(5)
    want = []
    for _ in range(3):
        for p in range(2):
            v = np.random.uniform(spec.rand_low, spec.rand_high, size=6)
            while np.linalg.norm(v[:2] - v[3:5]) < 0.15:
                v = np.random.uniform(spec.rand_low, spec.rand_high, size=6)
        want.append(v)
    np.random.set_state(st0)
    got = [t.unpack()["rand_vec"] for t in B.make_tasks(["reach-v3"], False, seed=5, n_goals=3)]
    assert np.allclose(got, want, rtol=0, atol=0)


def test_benchmark_lists():
    from metaworld_b200 import benchmarks as B
    assert len(B.ALL_V3) == 50 and len(set(B.ALL_V3)) == 50
    assert B.MT10[0] == "reach-v3" and len(B.MT10) == 10 and len(B.MT25) == 25 and B.MT50 == B.ALL_V3
    assert len(B.ML45["train"]) == 45 and len(B.ML45["test"]) == 5 and not set(B.ML45["train"]) & set(B.ML45["test"])
    assert len(B.ML10["train"]) == 10 and len(B.ML10["test"]) == 5


def test_lowering_reach():
    from metaworld_b200 import lower, modelzoo
    from metaworld_b200.tasks import TASKS
    spec = TASKS["reach-v3"]
    m = modelzoo.full_model(spec.xml)
    lw = lower.lower(m, spec.movable, spec.frames)
    r = lw.rec
    assert int(r["nlink"]) == 10 and int(r["nv"]) == 15 and int(r["nq"]) == 16
    assert int(r["ngeom"]) == 12                                       # SURVEY appendix B: 12 active colliders
    total_mass = float(sum(m.arrays["body_mass"][b] for b in range(m.nbody) if m.arrays["body_weldid"][b] != 0))
    assert float(r["link_mass"][: int(r["nlink"])].sum()) == pytest.approx(total_mass, rel=1e-6)
    # dof masks: arm chain is nested, the free object only sees its own 6 dofs
    assert int(r["link_dofmask"][6]) == 0b1111111 and int(r["link_dofmask"][9]) == 0b111111 << 9
    assert lower.DTYPE.itemsize % 4 == 0
    hdr = lower.emit_header()
    assert f"sizeof(MwModel) == {lower.DTYPE.itemsize}" in hdr
    # flat-model kinematics equals full-model kinematics at a random configuration
    from metaworld_b200 import mjcf
    rng = np.random.default_rng(0)
    q = m.arrays["qpos0"].copy()
    q[:7] = rng.uniform(-1, 1, 7)
    q[7:9] = [0.02, -0.01]
    xpos, xquat = mjcf.kinematics(m, q, np.zeros(3), np.array([1.0, 0, 0, 0]))
    lpos, lquat = {}, {}
    for l in range(int(r["nlink"])):
        p = int(r["link_parent"][l])
        pp, pq = (np.zeros(3), np.array([1.0, 0, 0, 0])) if p < 0 else (lpos[p], lquat[p])
        pos = pp + mjcf.quat2mat(pq) @ r["link_pos"][l].astype(np.float64)
        quat = mjcf.quat_mul(pq, r["link_quat"][l].astype(np.float64))
        jt, qa = int(r["link_jtype"][l]), int(r["link_qadr"][l])
        if jt == mjcf.JNT_FREE:
            pos, quat = q[qa:qa + 3], mjcf.quat_norm(q[qa + 3:qa + 7])
        elif jt == mjcf.JNT_SLIDE:
            pos = pos + mjcf.quat2mat(quat) @ r["link_jaxis"][l] * q[qa]
        else:
            ax = r["link_jaxis"][l].astype(np.float64)
            qr = np.concatenate([[np.cos(q[qa] / 2)], np.sin(q[qa] / 2) * ax])
            anchor = pos + mjcf.quat2mat(quat) @ r["link_jpos"][l]
            quat = mjcf.quat_norm(mjcf.quat_mul(quat, qr))
            pos = anchor - mjcf.quat2mat(quat) @ r["link_jpos"][l]
        lpos[l], lquat[l] = pos, quat
        assert np.allclose(pos, xpos[lw.link_body[l]], atol=1e-6)
    f = lower.F_HAND
    hand = lpos[int(r["frame_link"][f])] + mjcf.quat2mat(lquat[int(r["frame_link"][f])]) @ r["frame_pos"][f]
    assert np.allclose(hand, xpos[m.names["body"].index("hand")], atol=1e-6)


def test_cabi_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "metaworld_b200.h")).read()
    names = set(re.findall(r"\b(mw_[a-z_0-9]+)\s*\(", hdr))
    assert {"mw_create", "mw_step", "mw_reset", "mw_build_snapshots", "mw_destroy"} <= names
    from metaworld_b200 import lower
    for so in ("libmwb200.so", "libmwb200_f64.so"):      # the float32 step engine and the float64 snapshot builder: same ABI, same records
        lib = ctypes.CDLL(os.path.join(ROOT, "metaworld_b200", so))
        for n in names:
            assert hasattr(lib, n), f"{n} declared in include/metaworld_b200.h but not exported by {so}"
        lib.mw_sizeof_envstate.restype = ctypes.c_int
        assert lib.mw_sizeof_envstate() == 512 and lib.mw_sizeof_snapshot() == 768
        assert lib.mw_sizeof_model() == lower.DTYPE.itemsize
        lib.mw_build_info.restype = ctypes.c_char_p
        assert (b"real=double" if "f64" in so else b"real=float") in lib.mw_build_info()
    # no CPU fallback: creating an engine without a CUDA device must fail loudly
    from metaworld_b200 import engine
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(engine.EngineError):
            engine.Engine(["reach-v3"])


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under metaworld_b200/ may reference it."""
    for dp, _, fs in os.walk(os.path.join(ROOT, "metaworld_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "oracle/" not in txt.replace("oracle/ ", ""), f


def test_sharding_partition():
    from metaworld_b200.sharding import env_type, shard_env_ids
    N, W, T = 4096, 8, 50
    allids = np.concatenate([shard_env_ids(N, r, W) for r in range(W)])
    assert sorted(allids.tolist()) == list(range(N))
    for r in range(W):
        types = env_type(shard_env_ids(N, r, W), T)
        cnt = np.bincount(types, minlength=T)
        assert cnt.min() >= 1 and cnt.max() - cnt.min() <= 2      # every rank sees every task type, balanced


_GLOO_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from metaworld_b200.sharding import shard_env_ids, gather_to_rank0
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
N = 101
ids = shard_env_ids(N, rank, world)
local = torch.stack([torch.tensor(ids, dtype=torch.float32), torch.full((len(ids),), float(rank))], dim=1)
out = gather_to_rank0(local, N, rank, world)
if rank == 0:
    assert out.shape == (N, 2)
    assert torch.equal(out[:, 0], torch.arange(N, dtype=torch.float32))
    assert torch.equal(out[:, 1], torch.cat([torch.zeros(51), torch.ones(50)]))
    print("GLOO_OK")
dist.destroy_process_group()
'''


def test_two_rank_gather_gloo(tmp_path):
    """world_size-2 run of the N>1 path on CPU (gloo): shard ownership + obs gather to rank 0."""
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", str(script), ROOT], capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0 and "GLOO_OK" in r.stdout, r.stdout + r.stderr


def test_task_registry_matches_oracle_classes():
    """The device's per-task constants (metaworld_b200/tasks.py, fed to the kernels through MwTaskConst) and the oracle's
    task classes (oracle/tasks.py) are two independent transcriptions of the 50 reference constructors: they must agree on
    the model file, hand / mocap workspace, initial hand position, reset space and goal space."""
    from metaworld_b200.tasks import TASKS
    from metaworld_b200 import benchmarks as B
    from oracle.tasks import TASKS as OT
    assert set(TASKS) == set(OT) == set(B.ALL_V3) and len(TASKS) == 50
    assert sorted(t.task_id for t in TASKS.values()) == list(range(50))
    for name, spec in TASKS.items():
        env = OT[name]()
        assert env.xml == spec.xml, name
        assert np.allclose(env.mocap_low, spec.hand_low) and np.allclose(env.mocap_high, spec.hand_high), name
        assert np.allclose(env.hand_init_pos, spec.hand_init_pos), name
        lo, hi = env.random_reset_space()
        assert np.allclose(lo, spec.rand_low) and np.allclose(hi, spec.rand_high), name
        assert np.allclose(env.goal_low, spec.goal_low) and np.allclose(env.goal_high, spec.goal_high), name


def test_bench_helpers():
    """bench.py host-side helpers: usable core count respects the cgroup quota; algorithmic bytes follow SURVEY 8(d)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = bench.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    names, total, kind = bench.benchmark_names("MT50")
    assert len(names) == total == 50 and kind == "mt"
    assert bench.benchmark_names("ML45-train")[0][0] == "assembly-v3" and len(bench.benchmark_names("ML45-test")[0]) == 5
    assert bench.METRIC == __import__("json").load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    v, sample, flops = bench.cpu_baseline(["reach-v3"], 1, 5)
    assert v > 0 and flops > 1e5          # oracle flop counter (oracle/mjphys.c FL): ~1.6 MFLOP per reach env step
    b = bench.algorithmic_bytes(["reach-v3"])
    assert b == 4 * (2 * 16 + 4 * 15 + 120)          # nq 16, nv 15 -> 848 B per env step
    assert abs(bench.algorithmic_bytes(names) - 792.32) < 0.5


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """--dump-outputs: every step_torch output as float32 .npy; above the size cap a seeded sample of env rows (the
    same rows every run) plus their indices, all within the cap."""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    out = dict(obs=torch.rand(1000, 89, generator=g), reward=torch.rand(1000, generator=g), terminated=torch.zeros(1000, dtype=torch.uint8),
               truncated=torch.ones(1000, dtype=torch.uint8), info=torch.rand(1000, 7, generator=g))
    bench.dump_outputs(str(tmp_path / "full"), out)
    for k, v in out.items():
        a = np.load(tmp_path / "full" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.float().numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 50_000)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), out)
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= 50_000
    rows = np.load(tmp_path / "s1" / "env_index.npy")
    assert np.array_equal(rows, np.load(tmp_path / "s2" / "env_index.npy")) and 0 < len(rows) < 1000
    assert np.array_equal(np.load(tmp_path / "s1" / "obs.npy"), out["obs"].numpy()[rows.astype(int)])
