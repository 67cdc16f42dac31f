"""CPU-only suite: the C-ABI library loads and exports every symbol include/mpe_b200.h declares,
shape-only handles answer the reference's shape table, descriptors match the property tables the
reference's make_world() produces (recorded in the golden fixtures), error behaviour, the drop-in
import surface, and the world_size-2 (gloo) shard/counter logic.  No compute call is made."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import CONFIGS, load_golden, make_product_env

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from multiagent_particle_envs_b200 import _lib
    header = open(os.path.join(ROOT, "include", "mpe_b200.h")).read()
    declared = set(re.findall(r"MPE_API[^;(]*?\b(mpe_[a-z_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    assert _lib.load().mpe_abi_version() == _lib.MPE_ABI_VERSION
    assert ctypes.sizeof(_lib.MpeDesc) == 480


# SURVEY.md 8(c) shapes table: n / action dims / obs dims / bytes per env-step (8(d))
SHAPES = {
    "simple": (1, [5], [4], 81),
    "simple_spread_n3": (3, [5, 5, 5], [18, 18, 18], 411),
    "simple_spread_n6": (6, [5] * 6, [36] * 6, 1254),
    "simple_tag": (4, [5] * 4, [16, 16, 16, 14], 492),
    "simple_world_comm": (6, [9, 5, 5, 5, 5, 5], [34, 34, 34, 34, 28, 28], 1182),
    "simple_adversary": (3, [5, 5, 5], [8, 10, 10], None),
    "simple_push": (2, [5, 5], [8, 19], None),
    "simple_speaker_listener": (2, [3, 5], [3, 11], None),
    "simple_reference": (2, [15, 15], [21, 21], None),
    "simple_crypto": (3, [4, 4, 4], [4, 8, 8], None),
}
N_GOALS = {"simple_adversary": 1, "simple_push": 1, "simple_speaker_listener": 1, "simple_reference": 2, "simple_crypto": 2}


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_shapes_spaces_and_descriptor(tag):
    from multiagent_particle_envs_b200 import MultiDiscrete
    env = make_product_env(tag)
    n, act, obs, nbytes = SHAPES[tag]
    g = load_golden(tag)
    assert env.n == n == len(env.agents)
    assert [s.shape for s in env.observation_space] == [(d,) for d in obs] == [(int(d),) for d in g["prop_obs_dims"]]
    sh = env.world.native_shapes()
    assert sh.act_dims == act == [int(d) for d in g["prop_act_dims"]]
    A, L, C = n, len(g["prop_landmark_size"]), int(g["prop_dim_c"])
    mov, sil = list(g["prop_agent_movable"]), list(g["prop_agent_silent"])
    unread = {"simple_crypto": 4 * A + 2 * L, "simple_speaker_listener": 4}.get(tag, 0)   # positions nobody needs
    formula = 4 * (4 * A + 2 * L + N_GOALS.get(tag, 0) + sum(act) + 4 * sum(mov) + sum(obs) + A
                   + C * sum(1 - x for x in sil) - unread) + A        # SURVEY.md 8(d), compulsory traffic
    assert sh.bytes_per_env_step == formula and (nbytes is None or nbytes == formula)
    assert sh.n_goals == N_GOALS.get(tag, 0)
    for i, sp in enumerate(env.action_space):
        if mov[i] and not sil[i]:
            assert isinstance(sp, MultiDiscrete) and list(sp.high - sp.low + 1) == [5, C]
        else:
            assert sp.n == (5 if mov[i] else C)
    assert env.shared_reward == bool(int(g["prop_shared_reward"]))
    assert env.discrete_action_space is True and env.discrete_action_input is False and env.time == 0
    d = env.world.descriptor()
    A, L = d.n_agents, d.n_landmarks
    assert d.dim_c == int(g["prop_dim_c"]) and d.dt == float(g["prop_dt"]) and d.damping == float(g["prop_damping"])
    assert d.contact_force == float(g["prop_contact_force"]) and d.contact_margin == float(g["prop_contact_margin"])
    assert list(d.agent_size)[:A] == list(g["prop_agent_size"]) and list(d.agent_mass)[:A] == list(g["prop_agent_mass"])
    assert list(d.agent_sens)[:A] == [5.0 if a < 0 else a for a in g["prop_agent_accel"]]
    assert list(d.agent_max_speed)[:A] == list(g["prop_agent_max_speed"])
    for field in ("movable", "collide", "silent", "adversary", "leader"):
        assert list(getattr(d, "agent_" + field))[:A] == list(g["prop_agent_" + field]), field
    assert list(d.landmark_size)[:L] == list(g["prop_landmark_size"])
    assert list(d.landmark_collide)[:L] == list(g["prop_landmark_collide"])
    assert not any(g["prop_landmark_movable"])


def test_error_codes_without_a_gpu():
    from multiagent_particle_envs_b200 import _lib
    lib = _lib.load()
    env = make_product_env("simple_spread_n3")
    d = env.world.descriptor()
    h = ctypes.c_void_p()
    assert lib.mpe_create(ctypes.byref(d), 0, -1, ctypes.byref(h)) == -1            # n_env <= 0
    d.abi_version = 99
    assert lib.mpe_create(ctypes.byref(d), 8, -1, ctypes.byref(h)) == -2
    d.abi_version = _lib.MPE_ABI_VERSION
    d.agent_silent[1] = 0                                                           # spread agents must be silent
    assert lib.mpe_create(ctypes.byref(d), 8, -1, ctypes.byref(h)) == -2
    d.agent_silent[1] = 1
    d.scenario = _lib.SCN_CRYPTO
    assert lib.mpe_create(ctypes.byref(d), 8, -1, ctypes.byref(h)) in (-2, -3)
    d.scenario = _lib.SCN_SPREAD
    assert lib.mpe_create(ctypes.byref(d), 8, -1, ctypes.byref(h)) == 0
    assert lib.mpe_num_envs(h) == 8 and lib.mpe_obs_dim(h, 0) == 18 and lib.mpe_obs_dim(h, 3) == -1
    # a shape-only handle refuses to launch
    assert lib.mpe_world_step(h, 16, 16, None, 16, None, None) == -5
    assert b"device" in lib.mpe_strerror(-5)
    assert lib.mpe_destroy(h) == 0
    assert lib.mpe_destroy(None) == -1
    with pytest.raises(_lib.MpeError):
        _lib.check(-3, "probe")


def test_no_cpu_fallback_and_loud_failures():
    import torch
    from multiagent_particle_envs_b200 import MultiAgentEnv, World, Agent
    from multiagent_particle_envs_b200.scenarios import simple_spread
    sc = simple_spread.Scenario()
    world = sc.make_world()
    with pytest.raises(NotImplementedError):      # arbitrary Python callbacks have no native program
        MultiAgentEnv(world, sc.reset_world, lambda a, w: 0.0, sc.observation)
    w2 = World()
    w2.agents = [Agent()]
    with pytest.raises(NotImplementedError):
        w2.descriptor()
    if not torch.cuda.is_available():
        env = make_product_env("simple")
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            env.reset()


def test_missing_extension_fails_loudly(tmp_path):
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from multiagent_particle_envs_b200 import _lib\n"
            "_lib.LIB_PATH = %r\n"
            "try:\n    _lib.load()\nexcept ImportError as e:\n    print('LOUD', e)\n") % (ROOT, str(tmp_path / "nope.so"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert "LOUD" in out.stdout and "no CPU fallback" in out.stdout


def test_drop_in_import_surface():
    """the imports an existing MADDPG train.py performs (make_env.py:33-36 of the reference)"""
    from multiagent.environment import MultiAgentEnv
    import multiagent.scenarios as scenarios
    from multiagent.core import World, Agent, Landmark  # noqa: F401
    from multiagent.scenario import BaseScenario
    from multiagent.multi_discrete import MultiDiscrete  # noqa: F401
    from make_env import make_env
    scenario = scenarios.load("simple_tag.py").Scenario()
    assert isinstance(scenario, BaseScenario)
    world = scenario.make_world()
    assert len(world.policy_agents) == 4 and world.scripted_agents == [] and len(world.entities) == 6
    env = MultiAgentEnv(world, scenario.reset_world, scenario.reward, scenario.observation)
    assert env.n == 4
    assert make_env("simple").n == 1
    with pytest.raises(FileNotFoundError):
        scenarios.load("no_such_scenario.py")
    with pytest.raises(NotImplementedError):
        BaseScenario().make_world()
    md = MultiDiscrete([[0, 4], [0, 3]])
    assert md.num_discrete_space == 2 and md.contains([4, 3]) and not md.contains([5, 0]) and md.shape == 2
    s = md.sample()
    assert len(s) == 2 and md.contains(s)


def test_shard_ranges():
    from multiagent_particle_envs_b200.sharding import shard_range
    for n in (1, 7, 8, 65536, 1000003):
        for ws in (1, 2, 3, 8):
            spans = [shard_range(n, r, ws) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(8, 2, 2)


def _gloo_worker(rank, world_size, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from multiagent_particle_envs_b200.sharding import aggregate_counters, shard_range
    from multiagent_particle_envs_b200 import make_env
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world_size)
    env = make_env("simple_spread", num_envs=1001, rank=rank, world_size=world_size)
    lo, hi = shard_range(1001, rank, world_size)
    assert env.world.batch_size == hi - lo and env.world.world_offset == lo
    total, tmax, per_rank = aggregate_counters(env.world.batch_size * 10, 0.5 + rank)
    q.put((rank, total, tmax, per_rank))
    dist.destroy_process_group()


def test_two_rank_gloo_sharding_and_counter():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, total, tmax, per_rank in res:
        assert total == 10010.0 and tmax == 1.5
        assert per_rank == [(5010.0, 0.5), (5000.0, 1.5)]


def test_headless_rasteriser_draws_circles():
    from multiagent_particle_envs_b200.raster import draw_world
    img = draw_world(np.array([[0.0, 0.0], [0.5, 0.5]]), [0.2, 0.1], [np.array([1.0, 0, 0]), np.array([0, 0, 1.0])], [1.0, 0.5])
    assert img.shape == (700, 700, 3) and img.dtype == np.uint8
    assert tuple(img[350, 350]) == (255, 0, 0)                    # opaque red disc at the origin
    assert tuple(img[175, 525]) == (128, 128, 255)                # half-transparent blue at (0.5, 0.5): y axis points up
    assert tuple(img[10, 10]) == (255, 255, 255)
    area = (img[:, :, 1] == 0).sum() / 700.0 ** 2 * 4.0           # red disc area in world units
    assert abs(area - np.pi * 0.2 ** 2) < 0.003


def test_custom_scenario_descriptor_and_shape_only_handle():
    """MPE_SCN_CUSTOM: any entity table is accepted; shapes come from the descriptor; observe / fused step are refused"""
    from multiagent_particle_envs_b200 import Agent, Landmark, TorchScenario, World, _lib

    class Scenario(TorchScenario):
        def make_world(self, num_envs=None, device=None):
            world = World()
            world.dim_c = 4
            world.agents = [Agent() for _ in range(7)]
            for i, ag in enumerate(world.agents):
                ag.name, ag.silent, ag.movable, ag.collide = 'agent %d' % i, i % 3 != 0, i != 6, i % 2 == 0
            world.landmarks = [Landmark() for _ in range(8)]
            return self._finish_world(world, num_envs, device)

    world = Scenario().make_world(num_envs=64)
    d = world.descriptor()
    assert d.scenario == _lib.SCN_CUSTOM and d.n_agents == 7 and d.n_landmarks == 8
    sh = world.native_shapes()
    assert sh.custom and sh.obs_dims == [] and sh.n_speakers == 3
    assert sh.act_dims == [9, 5, 5, 9, 5, 5, 4]
    lib = _lib.load()
    assert lib.mpe_obs_dim(sh.handle, 0) == _lib.ERR_UNSUPPORTED
    assert lib.mpe_observe(sh.handle, 16, 16, 16, None, None, 16, 16, None, 0, None) == _lib.ERR_UNSUPPORTED
    world.agents.append(Agent())
    world.agents.append(Agent())
    with pytest.raises(ValueError):          # more than 8 agents
        world.descriptor()


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver launches) prints exactly one JSON line with the contract's keys"""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "60", "--warmup", "5"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    r = json.loads(lines[0])
    assert r["impl"] == "reference" and r["metric"] == "env_steps_per_sec" and r["unit"] == "env-steps/s"
    assert r["n_gpus"] == 1 and r["steps"] == 60 and r["warmup"] == 5 and r["higher_is_better"] is True
    assert r["value"] > 100 and r["vs_baseline"] is None and r["data"] == "synthetic" and r["dtype"] == "f64"
    cb = r["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == r["value"] and "np_port" in cb["sample"]
    assert r["e2e"] == {"value": r["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert r["config"]["workload"].startswith("simple_spread N=3") and r["config"]["n_env_per_gpu"] == 65536
    # the CPU sample is decoupled from --steps: 60 bench steps x 100 calls = 6000 env.step calls per process
    assert r["steps_timed_per_process"] == 6000 and cb["warmup_per_process"] >= 100
    # the arm never loads CUDA or the product library: only the CPU oracle (its own infrastructure)
    assert r["native_so_in_process"] == ["oracle/_build/libmpe_oracle.so"], r["native_so_in_process"]
    # same config dict as the GPU arm builds for this workload (ring sized on input bytes: 132 B x 65536 x 123 > 8 x L2)
    assert r["config"]["ring_batches"] == 123 and r["config"]["bytes_per_env_step"] == 411
    # under torchrun every rank but 0 exits silently
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "10", "--warmup", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_bench_shape_formula_equals_library(tag):
    """bench.py's CPU arm computes the workload description without dlopening libmpe_b200.so; its restatement of
    mpe_bytes_per_env_step (and of the input bytes the ring is sized on) must equal what the library reports"""
    sys.path.insert(0, ROOT)
    import bench
    name, kw = CONFIGS[tag]
    w = bench.scenario_world(name, kw)
    act, obs, bpe, ibpe = bench.shapes_from_oracle(w.descriptor())
    sh = w.native_shapes()
    assert act == sh.act_dims and obs == sh.obs_dims and bpe == sh.bytes_per_env_step
    assert ibpe == bench.input_bytes_from_shapes(sh)        # what the GPU arm sizes its ring on
    R = bench.ring_size(ibpe, 65536)
    assert 0 < ibpe < bpe and (R == bench.MAX_RING or R * ibpe * 65536 > bench.L2_MULTIPLE * bench.L2_BYTES)
    assert bench.ring_size(ibpe, 1 << 26) == 3      # huge batches: the minimum ring


def test_bench_numa_pinning_degrades_gracefully():
    """without nvidia-smi / sysfs GPU entries (this container) the rank keeps its affinity and says so"""
    sys.path.insert(0, ROOT)
    import bench
    before = os.sched_getaffinity(0)
    orig, what = bench.pin_to_gpu_numa(0)
    try:
        assert orig == before and isinstance(what, str) and what
        assert os.sched_getaffinity(0) <= before
    finally:
        os.sched_setaffinity(0, before)


def test_bench_dump_outputs_arguments_and_sample():
    """--dump-outputs takes a directory; outputs over 64 MB are written as one fixed sample of worlds; a run must time
    at least one step"""
    sys.path.insert(0, ROOT)
    import bench
    assert bench.parse_args(["--steps", "7", "--dump-outputs", "out"]).dump_outputs == "out"
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        with pytest.raises(SystemExit):
            bench.parse_args(bad)
    assert bench.dump_sample(65536, 4 * (3 * 18 + 2 * 3)) is None          # the headline workload: every world
    rows = bench.dump_sample(1 << 20, 1024)
    assert rows.size == bench.DUMP_MAX_BYTES // 1024 and rows[-1] < 1 << 20 and (np.diff(rows) > 0).all()
    assert np.array_equal(rows, bench.dump_sample(1 << 20, 1024))
