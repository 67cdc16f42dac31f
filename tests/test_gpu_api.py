"""The reference-shaped Python surface, exercised on the GPU: entity state / action properties over the
device tensors, World.step(), scenario callbacks, MultiAgentEnv accessors, discrete_action_input, the
scalar (batch-1, NumPy) convention for every scenario, benchmark_data shapes, goal sampling at reset."""
import numpy as np
import pytest

from helpers import CONFIGS, NO_BENCHMARK, load_golden, make_product_env, split_cols

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RTOL, ATOL = 1e-5, 1e-6


def test_entity_properties_are_views_of_the_batch_state():
    n = 257
    env = make_product_env("simple_tag", num_envs=n)
    env.reset()
    world, nw = env.world, env.world.native
    ag, lm = world.agents[1], world.landmarks[0]
    p = ag.state.p_pos
    assert p.shape == (n, 2) and p.is_cuda and p.data_ptr() == nw.agent_pv[1].data_ptr()
    ag.state.p_pos = torch.full((n, 2), 0.25, device="cuda")             # assignment writes through
    ag.state.p_vel = np.array([0.5, -0.5])                                # broadcast of a reference-style 2-vector
    lm.state.p_pos = torch.zeros(n, 2, device="cuda")
    assert float(nw.agent_pv[1, :, 0:2].min()) == 0.25 and float(nw.agent_pv[1, 7, 3]) == -0.5
    assert float(nw.lm_p[0].abs().max()) == 0.0
    assert ag.state.c.shape == (n, 2) and float(ag.state.c.abs().max()) == 0.0          # silent agent
    assert lm.state.p_vel.shape == (n, 2)
    # World.step() consumes agent.action.u exactly like the reference (core.py:134-140)
    pv0 = nw.agent_pv.permute(1, 0, 2).cpu().numpy().astype(np.float64)
    lm0 = nw.lm_p.permute(1, 0, 2).cpu().numpy().astype(np.float64)
    u = np.random.RandomState(0).uniform(-3, 3, (n, 4, 2))
    for i, a in enumerate(world.agents):
        a.action.u = torch.as_tensor(u[:, i], dtype=torch.float32, device="cuda")
    world.step()
    from oracle import Oracle
    rpv, _ = Oracle(world.descriptor(), "f64").world_step(pv0, lm0, np.zeros((n, 4, 2)), u.astype(np.float32), np.zeros((n, 4, 2)))
    np.testing.assert_allclose(nw.agent_pv.permute(1, 0, 2).cpu().numpy(), rpv, rtol=RTOL, atol=ATOL)


def test_scenario_callbacks_and_env_accessors():
    n = 500
    env = make_product_env("simple_spread_n3", num_envs=n)
    env.reset()
    world = env.world
    sc = world.scenario
    acts = [torch.softmax(torch.randn(n, 5, device="cuda"), 1) for _ in range(3)]
    obs_n, rew_n, done_n, info_n = env.step(acts)
    for i, ag in enumerate(world.agents):
        assert torch.equal(sc.observation(ag, world), obs_n[i])          # callbacks == what step returned
        assert torch.equal(env._get_obs(ag), obs_n[i])
    per_agent = torch.stack([sc.reward(ag, world) for ag in world.agents])
    assert torch.allclose(per_agent.sum(0), rew_n[0], rtol=1e-6, atol=1e-5)   # env shares the SUM (environment.py:100-102)
    rew0, coll, mind, occ = sc.benchmark_data(world.agents[0], world)
    assert torch.equal(rew0, per_agent[0]) and float(coll.min()) >= 1.0
    assert env._get_done(world.agents[0]) is False and env._get_info(world.agents[0]) is not None
    # _set_action for a single agent decodes into agent.action.u (environment.py:173-181)
    a = torch.tensor([[0.0, 1.0, 0.0, 0.0, 0.0]], device="cuda").repeat(n, 1)
    env._set_action(a, world.agents[2], env.action_space[2])
    u = world.agents[2].action.u
    assert torch.allclose(u, torch.tensor([5.0, 0.0], device="cuda").expand(n, 2))
    frames = env.render('rgb_array')                                  # headless stand-in for the pyglet viewer
    assert len(frames) == 1 and frames[0].shape == (700, 700, 3) and frames[0].dtype == np.uint8
    assert (frames[0] != 255).any() and (frames[0] == 255).mean() > 0.5


@pytest.mark.parametrize("tag", ["simple_tag", "simple_world_comm", "simple_speaker_listener"])
def test_discrete_action_input(tag):
    """env.discrete_action_input = True: integer sub-actions (environment.py:161-167, 185-187)"""
    from oracle import Oracle
    from multiagent_particle_envs_b200 import _lib
    n = 1024
    env = make_product_env(tag, num_envs=n)
    env.discrete_action_input = True
    env.reset()
    nw, desc = env.world.native, env.world.descriptor()
    rng = np.random.RandomState(5)
    pv0 = nw.agent_pv.permute(1, 0, 2).cpu().numpy()
    lm0 = nw.lm_p.permute(1, 0, 2).cpu().numpy()
    goal = nw.goal.t().cpu().numpy() if nw.n_goals else None
    ints = []
    for i in range(desc.n_agents):
        cols = ([rng.randint(0, 5, n)] if desc.agent_movable[i] else []) + \
               ([rng.randint(0, desc.dim_c, n)] if not desc.agent_silent[i] else [])
        ints.append(np.stack(cols, 1))
    obs_n, rew_n, _, _ = env.step([torch.as_tensor(a, device="cuda") for a in ints])
    flat = np.concatenate(ints, 1).astype(np.float64)
    flags = _lib.FLAG_DISCRETE_ACTION_INPUT | (_lib.FLAG_SHARED_REWARD if env.shared_reward else 0)
    rpv, rcomm, robs, rrew, _, _ = Oracle(desc, "f64").step(pv0, lm0, np.zeros((n, desc.n_agents, desc.dim_c)), flat,
                                                            flags, goal=goal)
    np.testing.assert_allclose(np.concatenate([o.cpu().numpy() for o in obs_n], 1), robs, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(nw.agent_pv.permute(1, 0, 2).cpu().numpy(), rpv, rtol=RTOL, atol=ATOL)


def test_scalar_mode_with_integer_actions():
    """reference usage: env.discrete_action_input = True; env.step([2, 4, 0]) on a single world"""
    env = make_product_env("simple_spread_n3")
    env.discrete_action_input = True
    env.reset()
    for ag, p in zip(env.world.agents, ([-0.8, 0.0], [0.0, 0.8], [0.8, 0.0])):   # far apart: no contact forces
        ag.state.p_pos = np.array(p)
        ag.state.p_vel = np.zeros(2)
    obs_n, rew_n, done_n, info_n = env.step([1, 2, 4])
    assert all(isinstance(o, np.ndarray) and o.dtype == np.float64 and o.shape == (18,) for o in obs_n)
    assert all(isinstance(d, bool) for d in done_n) and isinstance(float(rew_n[0]), float)
    # index 1 -> u.x = -1, 2 -> +1, 4 -> u.y = +1 (environment.py:163-167), sensitivity 5, dt 0.1
    np.testing.assert_allclose([obs_n[0][0], obs_n[1][0], obs_n[2][1]], [-0.5, 0.5, 0.5], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_scalar_convention_replays_reference_world(tag):
    """make_env(name) with no batch: lists of float64 ndarrays / floats / bools, world 0 of the golden
    fixture injected through the reference's own attributes, 5 recorded steps replayed"""
    g = load_golden(tag)
    env = make_product_env(tag)
    env.reset()
    world = env.world
    nw = world.native
    for i, ag in enumerate(world.agents):
        ag.state.p_pos = g["pv0"][0, i, 0:2]
        ag.state.p_vel = g["pv0"][0, i, 2:4]
    for l, lm in enumerate(world.landmarks):
        lm.state.p_pos = g["lm"][0, l]
    if nw.n_goals:
        nw.goal.copy_(torch.as_tensor(g["goal"][0:1], dtype=torch.int32, device="cuda").t())
    adims = [int(x) for x in g["prop_act_dims"]]
    for t in range(5):
        obs_n, rew_n, done_n, info_n = env.step([a.copy() for a in split_cols(g["act"][0, t], adims)])
        assert isinstance(obs_n, list) and all(o.dtype == np.float64 and o.ndim == 1 for o in obs_n)
        assert all(isinstance(d, bool) and not d for d in done_n) and len(info_n["n"]) == env.n
        np.testing.assert_allclose(np.concatenate(obs_n), g["obs"][0, t], rtol=2e-5, atol=5e-6)
        np.testing.assert_allclose(np.array(rew_n, dtype=np.float64), g["rew"][0, t], rtol=2e-5, atol=2e-5)
    if tag not in NO_BENCHMARK:                     # benchmark_data comes back in the reference's shape
        item = info_n["n"][-1]
        ref = g["info"][0, 4, env.n - 1]
        got = np.concatenate([np.atleast_1d(np.asarray(x, dtype=np.float64)) for x in (item if isinstance(item, tuple) else (item,))])
        np.testing.assert_allclose(got, ref[:len(got)], rtol=2e-5, atol=2e-5)
    else:
        assert info_n["n"] == [{}] * env.n
    p = world.agents[0].state.p_pos
    assert isinstance(p, np.ndarray) and p.shape == (2,) and p.dtype == np.float64


def test_goal_indices_are_uniform_and_shard_independent():
    n = 120000
    env = make_product_env("simple_reference", num_envs=n, seed=9)
    env.reset()
    goal = env.world.native.goal
    assert goal.shape == (2, n) and int(goal.min()) == 0 and int(goal.max()) == 2
    for g in range(2):
        frac = torch.bincount(goal[g].long(), minlength=3).float() / n
        assert float((frac - 1 / 3).abs().max()) < 0.01
    assert float((goal[0] == goal[1]).float().mean()) < 0.36        # the two draws are independent
    sh = make_product_env("simple_reference", num_envs=n, seed=9, rank=1, world_size=3)
    sh.reset()
    assert torch.equal(sh.world.native.goal, goal[:, n // 3: 2 * n // 3])
    before = goal.clone()
    env.reset()
    assert not torch.equal(before, env.world.native.goal)            # new epoch, new draws


def test_graphed_rollout_matches_eager():
    """policy -> env.step x T captured in one CUDA graph == the same loop run eagerly"""
    from multiagent_particle_envs_b200.rollout import GraphedRollout
    n, T = 4096, 25
    torch.manual_seed(0)
    weights = [torch.randn(18, 5, device="cuda") * 0.5 for _ in range(3)]

    def policy(obs_n):
        return [torch.softmax(o @ w, dim=1) for o, w in zip(obs_n, weights)]

    env_g = make_product_env("simple_spread_n3", num_envs=n, seed=3)
    roll = GraphedRollout(env_g, policy, T)
    start_pv = env_g.world.native.agent_pv.clone()       # state after the warm-up / capture passes
    start_obs = [o.clone() for o in roll.obs]
    obs_g, rew_g = roll.run()
    torch.cuda.synchronize()
    env_e = make_product_env("simple_spread_n3", num_envs=n, seed=3)
    env_e.reset()
    env_e.world.native.agent_pv.copy_(start_pv)
    env_e.world.native.lm_p.copy_(env_g.world.native.lm_p)
    obs, tot = start_obs, torch.zeros(3, n, device="cuda")
    for _ in range(T):
        obs, rew_n, _, _ = env_e.step(policy(obs))
        tot += torch.stack(rew_n)
    for a, b in zip(obs_g, obs):
        assert torch.equal(a, b)
    assert torch.equal(rew_g, tot)


def test_graphed_rollout_with_resets_draws_fresh_episodes_on_replay():
    """a reset captured in the graph reads its epoch from device memory, so each replay starts new episodes"""
    from multiagent_particle_envs_b200.rollout import GraphedRollout
    n = 2048
    env = make_product_env("simple_spread_n3", num_envs=n, seed=5)
    roll = GraphedRollout(env, lambda obs_n: [torch.softmax(o[:, :5], 1) for o in obs_n], steps=10, reset_every=10)
    nw = env.world.native
    roll.run()
    torch.cuda.synchronize()
    first = nw.lm_p.clone()
    e1 = int(nw._epoch_dev.item())
    roll.run()
    torch.cuda.synchronize()
    assert int(nw._epoch_dev.item()) == e1 + 1
    assert not torch.equal(first, nw.lm_p)                      # new landmark draws after the replayed reset
    assert float(nw.agent_pv[:, :, 2:4].abs().max()) == 0.0      # ... and the episode really was reset
    env.reset()                                                  # eager resets keep advancing the same counter
    assert int(nw._epoch_dev.item()) == e1 + 2


@pytest.mark.parametrize("tag,n,T", [("simple_spread_n3", 2049, 25), ("simple_tag", 4096, 10), ("simple_world_comm", 1031, 7),
                                     ("simple_reference", 512, 6), ("simple_speaker_listener", 100, 5),
                                     ("simple_crypto", 333, 4), ("simple_adversary", 64, 9), ("simple", 33, 3)])
def test_open_loop_rollout_equals_repeated_steps(tag, n, T):
    """env.rollout (mpe_rollout: T steps in one launch, state in registers, next step's actions prefetched) is
    bit-identical to T calls of env.step on the same actions with the rewards summed in step order -- full tiles take
    the cp.async path, the ragged last tile the scalar one"""
    env_a = make_product_env(tag, num_envs=n, seed=5)
    env_b = make_product_env(tag, num_envs=n, seed=5)
    env_a.reset()
    env_b.reset()
    na, nb = env_a.world.native, env_b.world.native
    assert torch.equal(na.agent_pv, nb.agent_pv) and torch.equal(na.goal, nb.goal)
    g = torch.Generator(device="cuda").manual_seed(11)
    seqs = []
    for d, ag in zip(na.act_dims, env_a.agents):
        parts = [torch.softmax(2 * torch.randn(T, n, 5, device="cuda", generator=g), -1)] if ag.movable else []
        if d - (5 if ag.movable else 0) > 0:
            parts.append(torch.rand(T, n, d - (5 if ag.movable else 0), device="cuda", generator=g))
        seqs.append(torch.cat(parts, -1).contiguous())
    obs_r, rew_r, done_r, info_r, steps_r = env_a.rollout(seqs, per_step_rewards=True)
    rew_sum = torch.zeros(env_b.n, n, device="cuda")
    for t in range(T):
        obs_s, rew_s, done_s, _ = env_b.step([s[t] for s in seqs])
        rew_sum += torch.stack(list(rew_s))
        assert torch.equal(steps_r[t], torch.stack(list(rew_s))), t
    torch.cuda.synchronize()
    assert torch.equal(na.agent_pv, nb.agent_pv) and torch.equal(na.comm, nb.comm)
    for x, y in zip(obs_r, obs_s):
        assert torch.equal(x, y)
    assert torch.equal(torch.stack(list(rew_r)), rew_sum)
    assert not any(bool(d.any()) for d in done_r)
    # without the per-step record the result is the same
    env_c = make_product_env(tag, num_envs=n, seed=5)
    env_c.reset()
    obs_c, rew_c, _, _ = env_c.rollout(seqs)
    assert all(torch.equal(x, y) for x, y in zip(obs_c, obs_r)) and torch.equal(torch.stack(list(rew_c)), rew_sum)


@pytest.mark.parametrize("tag,n,T,H", [("simple_spread_n3", 2049, 12, 32), ("simple_spread_n3", 1000, 8, 64),
                                       ("simple_tag", 1031, 10, 32), ("simple_tag", 512, 5, 64), ("simple", 257, 6, 64)])
def test_closed_loop_policy_rollout(tag, n, T, H):
    """env.rollout_policy (mpe_rollout_policy: T steps in one launch, every agent's two-layer actor evaluated inside the
    kernel from observations that never leave the registers):
      (1) the actions it records, fed to T ordinary fused steps of a twin env, reproduce the final state, the final
          observations, every step's rewards and the reward sums BIT FOR BIT (physics / reward / observation parity);
      (2) every recorded action equals softmax(W2 relu(W1 obs + b1) + b2) evaluated in float64 on the twin's observations
          to 1e-5 (the fp32 perceptron, FMA accumulation in a fixed order)."""
    env_a = make_product_env(tag, num_envs=n, seed=9)
    env_b = make_product_env(tag, num_envs=n, seed=9)
    env_a.reset()
    obs_b = env_b.reset()
    na, nb = env_a.world.native, env_b.world.native
    assert torch.equal(na.agent_pv, nb.agent_pv)
    g = torch.Generator(device="cuda").manual_seed(3)
    policies = []
    for od in na.obs_dims:
        policies.append((torch.randn(H, od, device="cuda", generator=g) * 0.7, torch.randn(H, device="cuda", generator=g) * 0.3,
                         torch.randn(5, H, device="cuda", generator=g) * 0.5, torch.randn(5, device="cuda", generator=g) * 0.2))
    obs_r, rew_r, done_r, info_r, extras = env_a.rollout_policy(policies, T, record_actions=True, per_step_rewards=True)
    actions, rew_steps = extras["actions"], extras["rewards"]
    rew_sum = torch.zeros(env_b.n, n, device="cuda")
    for t in range(T):
        for i, (W1, b1, W2, b2) in enumerate(policies):          # (2) the actor, in float64, on the twin's observations
            o = obs_b[i].double()
            logits = torch.relu(o @ W1.double().t() + b1.double()) @ W2.double().t() + b2.double()
            want = torch.softmax(logits, -1)
            assert torch.allclose(actions[i][t].double(), want, rtol=1e-5, atol=1e-6), (t, i)
        obs_b, rew_s, done_s, _ = env_b.step([a[t] for a in actions])     # (1) replay the recorded actions
        rew_sum += torch.stack(list(rew_s))
        assert torch.equal(rew_steps[t], torch.stack(list(rew_s))), t
    torch.cuda.synchronize()
    assert torch.equal(na.agent_pv, nb.agent_pv)
    for x, y in zip(obs_r, obs_b):
        assert torch.equal(x, y)
    assert torch.equal(torch.stack(list(rew_r)), rew_sum)
    assert not any(bool(d.any()) for d in done_r)
    # nn.Module policies and no records: same result
    env_c = make_product_env(tag, num_envs=n, seed=9)
    env_c.reset()
    mods = []
    for W1, b1, W2, b2 in policies:
        m = torch.nn.Sequential(torch.nn.Linear(W1.shape[1], H), torch.nn.ReLU(), torch.nn.Linear(H, 5)).cuda()
        with torch.no_grad():
            m[0].weight.copy_(W1); m[0].bias.copy_(b1); m[2].weight.copy_(W2); m[2].bias.copy_(b2)
        mods.append(m)
    obs_c, rew_c, _, _, ex = env_c.rollout_policy(mods, T)
    assert ex["actions"] is None and all(torch.equal(x, y) for x, y in zip(obs_c, obs_r))
    assert torch.equal(torch.stack(list(rew_c)), rew_sum)
    # scenarios without the policy kernel refuse loudly
    env_w = make_product_env("simple_world_comm", num_envs=64)
    env_w.reset()
    from multiagent_particle_envs_b200._lib import MpeError
    with pytest.raises(MpeError):
        env_w.rollout_policy([(torch.zeros(32, od, device="cuda"), torch.zeros(32, device="cuda"), torch.zeros(5, 32, device="cuda"),
                               torch.zeros(5, device="cuda")) for od in env_w.world.native.obs_dims], 2)


def test_bench_dump_outputs_repeat_exactly(tmp_path):
    """bench.py --dump-outputs writes what the last timed step returned (per agent: obs, rew, done as float32), and two
    runs with the same arguments write the same arrays"""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = 4096
    dumps = []
    for r in range(2):
        d = tmp_path / str(r)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "30", "--warmup", "3",
                              "--num-envs", str(n), "--cpu-seconds", "0", "--e2e-steps", "3", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=root)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 30
        dumps.append({p.name[:-4]: np.load(p) for p in d.iterdir()})
    a, b = dumps
    assert sorted(a) == sorted("%s_%d" % (k, i) for k in ("obs", "rew", "done") for i in range(3))
    for k in a:
        assert a[k].dtype == np.float32 and a[k].shape[0] == n and np.array_equal(a[k], b[k]), k
        assert np.isfinite(a[k]).all(), k
    assert a["obs_0"].shape == (n, 18)
    assert np.array_equal(a["rew_0"], a["rew_1"]) and np.array_equal(a["rew_0"], a["rew_2"])     # shared reward
    assert set(np.unique(a["done_0"])) <= {0.0, 1.0}
