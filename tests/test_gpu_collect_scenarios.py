"""mpe_collect / env.rollout_policy in the scenarios whose agents speak or cannot move (simple_speaker_listener,
simple_reference, simple_crypto) and in simple_adversary / simple_push: per-head actors, the communication head's
exploration noise, the utterance state carried across steps.  CPU tests (no marker): which programs have the kernel,
the actor parser with action widths, the NumPy rebuild of the comm-head noise and its counters, argument checking on a
device-less crypto handle.  GPU tests (`gpu` marker): replay parity including the comm state, the float64 actor with
per-head softmax, continuation / sharding, the joint head distribution, the old entry point, refusals."""
import ctypes

import numpy as np
import pytest

from helpers import descriptor, make_product_env
from test_gpu_collect import MASK, exploration_uniforms, philox4x32_10

torch = pytest.importorskip("torch")

NEW = ("simple_adversary", "simple_push", "simple_speaker_listener", "simple_reference", "simple_crypto")
BUILT = ("simple", "simple_spread_n3", "simple_tag") + NEW
NOT_BUILT = ("simple_world_comm", "simple_spread_n6", "simple_tag_1v1", "simple_tag_2v1", "simple_tag_4v2",
             "simple_tag_6v2", "simple_adversary_n4")


def comm_uniforms(seed, worlds, step, agent, dim_c):
    """the dim_c u of the comm head of (global worlds [N], step, agent) as the kernel draws them: float64 [N, dim_c];
    logit q takes word q & 3 of block q >> 2 under the tag 0x40000100 | agent << 2 | block"""
    worlds = np.asarray(worlds, dtype=np.uint64)
    lo, hi = worlds & np.uint64(MASK), worlds >> np.uint64(32)
    key = (seed & MASK, seed >> 32)
    words = []
    for block in range((dim_c + 3) // 4):
        words += philox4x32_10((lo, hi, np.full_like(lo, step), np.full_like(lo, comm_tag(agent, block))), key)
    bits = np.stack(words[:dim_c], 1).astype(np.uint64)
    return (2.0 * (bits >> np.uint64(9)).astype(np.float64) + 1.0) * 2.0 ** -24


def comm_tag(agent, block):
    return 0x40000100 | (agent << 2) | block


def heads(nw, i):
    """column ranges of agent i's action heads: movement 0..4 if it moves, then dim_c comm logits if it speaks"""
    out, c = [], 0
    if nw.desc.agent_movable[i]:
        out.append((0, 5))
        c = 5
    if not nw.desc.agent_silent[i]:
        out.append((c, c + nw.dim_c))
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_collect_supported_on_device_less_handles():
    from multiagent_particle_envs_b200 import _lib
    from multiagent_particle_envs_b200.native import ShapeHandle
    lib = _lib.load()
    for tag in BUILT + NOT_BUILT:
        sh = ShapeHandle(descriptor(tag), 100, -1)
        want = 0 if tag in BUILT else _lib.ERR_UNSUPPORTED
        for depth in (1, 2):
            for H in (32, 64):
                assert sh.collect_supported(depth, H) == want, (tag, depth, H)
        assert sh.collect_supported(3, 64) == _lib.ERR_BAD_ARG
        assert sh.collect_supported(2, 48) == _lib.ERR_BAD_ARG
        sh.close()
    d = descriptor("simple_spread_n3")
    d.scenario = _lib.SCN_CUSTOM                                            # a user scenario with the same table
    sh = ShapeHandle(d, 100, -1)
    assert sh.custom and sh.collect_supported(1, 32) == _lib.ERR_UNSUPPORTED
    sh.close()
    assert lib.mpe_collect_supported(None, 1, 32) == _lib.ERR_BAD_ARG


def test_actor_parser_takes_the_action_widths():
    from multiagent_particle_envs_b200.environment import actor_parameters
    nn = torch.nn

    def seq(o, a, H=32, depth=2):
        mid = [nn.Linear(H, H), nn.ReLU()] if depth == 2 else []
        return nn.Sequential(nn.Linear(o, H), nn.ReLU(), *mid, nn.Linear(H, a))

    for od, ad in (([3, 11], [3, 5]), ([21, 21], [15, 15]), ([4, 8, 8], [4, 4, 4])):
        for depth in (1, 2):
            mods = [seq(o, a, depth=depth) for o, a in zip(od, ad)]
            got_depth, H, p = actor_parameters(mods, od, ad)
            assert (got_depth, H) == (depth, 32) and [tuple(t[-1].shape) for t in p] == [(a,) for a in ad]
            tup = [tuple(t.detach() for m in mod if isinstance(m, nn.Linear) for t in (m.weight, m.bias)) for mod in mods]
            assert actor_parameters(tup, od, ad)[:2] == (depth, 32)
            with pytest.raises(ValueError):                              # a 5-wide movement head only
                actor_parameters([seq(o, 5, depth=depth) for o in od], od, ad)
            with pytest.raises(ValueError):                              # one output too many on the last agent
                actor_parameters(mods[:-1] + [seq(od[-1], ad[-1] + 1, depth=depth)], od, ad)
    # act_dims=None: 5 for every agent, as before
    mods = [seq(18, 5) for _ in range(3)]
    assert actor_parameters(mods, [18] * 3)[:2] == actor_parameters(mods, [18] * 3, [5, 5, 5])[:2] == (2, 32)
    with pytest.raises(ValueError):
        actor_parameters([seq(18, 7) for _ in range(3)], [18] * 3)


def test_comm_noise_words_and_counters():
    """The NumPy rebuild of the comm-head uniforms, and the counter rule: comm tags never meet a movement tag or a
    counter of the reset stream (word 3 = a small block number or 0x80000000), for any agent, block or dim_c <= 16."""
    seed = 2 ** 37 + 3
    u = comm_uniforms(seed, np.arange(2000), 5, 1, 10)
    assert u.shape == (2000, 10) and u.min() > 0.0 and u.max() < 1.0
    assert np.all(u.astype(np.float32).astype(np.float64) == u)
    # q -> word q & 3 of block q >> 2: logits 4..7 are block 1 of the same (world, step, agent)
    w = philox4x32_10((np.arange(2000), 0, 5, comm_tag(1, 1)), (seed & MASK, seed >> 32))
    assert np.array_equal(u[:, 4], (2.0 * (w[0].astype(np.float64) // 512) + 1.0) * 2.0 ** -24)
    # different agents and the movement head draw different words
    assert not np.array_equal(u, comm_uniforms(seed, np.arange(2000), 5, 0, 10))
    assert not np.array_equal(u[:, :5], exploration_uniforms(seed, np.arange(2000), 5, 1))
    movement = {0x40000000 | (a << 1) | b for a in range(8) for b in (0, 1)}
    comm = {comm_tag(a, b) for a in range(8) for b in range(4)}
    reset = set(range(8)) | {0x80000000}
    assert len(movement) == 16 and len(comm) == 32
    assert not (movement & comm) and not (movement & reset) and not (comm & reset)


def test_collect_refuses_bad_arguments_on_a_crypto_handle():
    from multiagent_particle_envs_b200 import _lib
    from multiagent_particle_envs_b200.native import ShapeHandle
    sh = ShapeHandle(descriptor("simple_crypto"), 1031, -1)
    lib, h, A = sh.lib, sh.handle, sh.n_agents
    assert sh.act_dims == [4, 4, 4] and sh.n_speakers == 3
    arr = lambda: (ctypes.c_void_p * A)(*([256] * A))   # noqa: E731

    def call(comm=256, depth=2, hidden=64, w3=True, act=256, flags=16):
        w3_n = arr() if w3 else None
        return lib.mpe_collect(h, 256, 256, comm, 256, depth, hidden, arr(), arr(), arr(), arr(), w3_n,
                               arr() if w3 else None, 4, 1, 0, 0, arr(), 256, None,
                               (ctypes.c_void_p * A)(*([act] * A)), arr(), 256, flags, None)

    assert call() == _lib.ERR_NO_DEVICE                                      # well-formed: only the device is missing
    assert call(depth=1, w3=False) == _lib.ERR_NO_DEVICE
    assert call(comm=None) == _lib.ERR_BAD_ARG                               # speakers need the comm state
    assert call(comm=258) == _lib.ERR_BAD_ARG
    assert call(depth=1) == _lib.ERR_BAD_ARG                                 # depth 1 takes no W3
    assert call(w3=False) == _lib.ERR_BAD_ARG                                # depth 2 needs it
    assert call(hidden=48) == _lib.ERR_BAD_ARG
    assert call(act=258) == _lib.ERR_BAD_ARG                                 # misaligned action record
    assert sh.collect_supported(2, 64) == 0
    sh.close()


# ---------------------------------------------------------------------------------------------------------------- GPU
def _actors(nw, H, seed, depth=2):
    """torch-default-initialised actors with act_dim_i outputs, as 6- or 4-tuples on the GPU"""
    torch.manual_seed(seed)
    out = []
    for od, ad in zip(nw.obs_dims, nw.act_dims):
        layers = [torch.nn.Linear(od, H)] + ([torch.nn.Linear(H, H)] if depth == 2 else []) + [torch.nn.Linear(H, ad)]
        out.append(tuple(t.detach().cuda() for m in layers for t in (m.weight, m.bias)))
    return out


def _actor64(pol, obs):
    x = obs.double()
    n = len(pol) // 2
    for k in range(n):
        x = x @ pol[2 * k].double().t() + pol[2 * k + 1].double()
        if k < n - 1:
            x = torch.relu(x)
    return x


def _noise64(nw, i, seed, n, step):
    """the Gumbel terms of agent i's logits as the kernel draws them, float64 [n, act_dim_i]"""
    worlds = np.arange(n, dtype=np.uint64)
    parts = []
    if nw.desc.agent_movable[i]:
        parts.append(exploration_uniforms(seed, worlds, step, i))
    if not nw.desc.agent_silent[i]:
        parts.append(comm_uniforms(seed, worlds, step, i, nw.dim_c))
    u = np.concatenate(parts, 1)
    return torch.from_numpy(-np.log(-np.log(u))).cuda()


def _per_head_softmax(nw, i, logits):
    return torch.cat([torch.softmax(logits[:, lo:hi], -1) for lo, hi in heads(nw, i)], -1)


PARITY = ([(tag, 1031, 2, H, s) for tag in NEW for H in (32, 64) for s in (None, 11)]
          + [(tag, 65536, 2, 64, s) for tag in ("simple_reference", "simple_speaker_listener") for s in (None, 2 ** 33 + 5)]
          + [(tag, 1031, 1, 64 if k % 2 else 32, 7 if k % 2 else None) for k, tag in enumerate(NEW)])


@pytest.mark.gpu
@pytest.mark.parametrize("tag,n,depth,H,seed", PARITY)
def test_replay_parity_and_float64_actor(tag, n, depth, H, seed):
    """Per-head actors, deterministic and sampled, with every record on:
      (1) the recorded actions fed to T `env.step` calls of a twin env reproduce the agents' state, the comm state, the
          final observations, every step's rewards and the reward sums BIT FOR BIT, and observation record row t is
          bit-equal to what the twin returned before step t;
      (2) every recorded action equals the float64 actor with one softmax per head (sampled: plus the Gumbel terms
          rebuilt by the NumPy Philox, movement and comm words) to rtol 1e-5, atol 1e-6, and every head sums to 1."""
    T, step0 = 7, 3
    env_a = make_product_env(tag, num_envs=n, seed=9)
    env_b = make_product_env(tag, num_envs=n, seed=9)
    env_a.reset()
    obs_b = env_b.reset()
    na, nb = env_a.world.native, env_b.world.native
    if na.n_speakers:   # one ordinary step first: step 0 of the rollout then observes non-zero carried-in utterances
        g = torch.Generator(device="cuda").manual_seed(n)
        warm = [torch.rand(n, ad, device="cuda", generator=g) for ad in na.act_dims]
        env_a.step(warm)
        obs_b = env_b.step(warm)[0]
        assert bool((na.comm != 0).any())
    pols = _actors(na, H, seed=H + n + depth, depth=depth)
    obs_r, rew_r, done_r, _, ex = env_a.rollout_policy(pols, T, record_actions=True, per_step_rewards=True,
                                                       record_observations=True, explore_seed=seed,
                                                       explore_step=step0 if seed is not None else 0)
    actions, rew_steps, obs_rec = ex["actions"], ex["rewards"], ex["observations"]
    assert [tuple(a.shape) for a in actions] == [(T, n, ad) for ad in na.act_dims]
    rew_sum = torch.zeros(env_b.n, n, device="cuda")
    for t in range(T):
        for i, pol in enumerate(pols):
            assert torch.equal(obs_rec[i][t], obs_b[i]), (t, i)
            logits = _actor64(pol, obs_b[i])
            if seed is not None:
                logits = logits + _noise64(na, i, seed, n, step0 + t)
            want = _per_head_softmax(na, i, logits)
            assert torch.allclose(actions[i][t].double(), want, rtol=1e-5, atol=1e-6), (t, i)
            for lo, hi in heads(na, i):
                assert torch.allclose(actions[i][t][:, lo:hi].sum(-1), torch.ones(n, device="cuda"), atol=1e-5), (t, i)
        obs_b, rew_s, _, _ = env_b.step([a[t] for a in actions])
        rew_sum += torch.stack(list(rew_s))
        assert torch.equal(rew_steps[t], torch.stack(list(rew_s))), t
    torch.cuda.synchronize()
    assert torch.equal(na.agent_pv, nb.agent_pv)
    assert torch.equal(na.comm, nb.comm)
    assert all(torch.equal(x, y) for x, y in zip(obs_r, obs_b))
    assert torch.equal(torch.stack(list(rew_r)), rew_sum)
    assert not any(bool(d.any()) for d in done_r)


def _run(env, pols, T, seed, step):
    obs, rew, _, _, ex = env.rollout_policy(pols, T, record_actions=True, per_step_rewards=True, record_observations=True,
                                            explore_seed=seed, explore_step=step)
    return [o.clone() for o in obs], ex


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["simple_reference", "simple_crypto"])
def test_continuation_and_sharding_carry_the_comm_state(tag):
    """Sampled depth-2 rollouts of speaking agents: two calls (explore_step 0, then T/2) equal one call of T steps, and
    each rank of a two-rank sharded env reproduces its half of the full batch -- agents, utterances, records"""
    n, T, seed = 1031, 8, 123
    full = make_product_env(tag, num_envs=n, seed=2)
    full.reset()
    pols = _actors(full.world.native, 64, seed=5)
    obs_f, ex_f = _run(full, pols, T, seed, 0)
    pv_f, comm_f = full.world.native.agent_pv.clone(), full.world.native.comm.clone()
    env = make_product_env(tag, num_envs=n, seed=2)
    env.reset()
    _, ex1 = _run(env, pols, T // 2, seed, 0)
    obs2, ex2 = _run(env, pols, T // 2, seed, T // 2)
    assert torch.equal(env.world.native.agent_pv, pv_f) and torch.equal(env.world.native.comm, comm_f)
    assert all(torch.equal(x, y) for x, y in zip(obs2, obs_f))
    assert torch.equal(torch.cat([ex1["rewards"], ex2["rewards"]]), ex_f["rewards"])
    for key in ("actions", "observations"):
        assert all(torch.equal(torch.cat([a, b]), c) for a, b, c in zip(ex1[key], ex2[key], ex_f[key])), key
    from multiagent_particle_envs_b200.sharding import shard_range
    for r in range(2):
        lo, hi = shard_range(n, r, 2)
        sh = make_product_env(tag, num_envs=n, seed=2, rank=r, world_size=2)
        sh.reset()
        obs_s, ex_s = _run(sh, pols, T, seed, 0)
        assert torch.equal(sh.world.native.agent_pv, pv_f[:, lo:hi])
        assert torch.equal(sh.world.native.comm, comm_f[:, lo:hi])
        assert all(torch.equal(x, y[lo:hi]) for x, y in zip(obs_s, obs_f))
        assert torch.equal(ex_s["rewards"], ex_f["rewards"][:, :, lo:hi])
        for key in ("actions", "observations"):
            assert all(torch.equal(x, y[:, lo:hi]) for x, y in zip(ex_s[key], ex_f[key])), (r, key)


@pytest.mark.gpu
def test_joint_head_argmax_follows_the_product_of_head_softmaxes():
    """simple_reference, all weights zero and b3 = (movement logits | comm logits): by the Gumbel-max property the
    arg-max of each sampled head follows that head's softmax, and the two heads draw independent noise, so the 5 x 10
    table of joint arg-maxes follows softmax(movement) (x) softmax(comm).  Chi-square over every (world, step, agent)
    sample; the seed is fixed, so the test is deterministic."""
    from scipy.stats import chisquare
    n, T, H = 65536, 4, 32
    env = make_product_env("simple_reference", num_envs=n, seed=3)
    env.reset()
    mov = torch.tensor([0.3, -1.2, 1.0, 0.0, -0.4], device="cuda")
    com = torch.tensor([0.5, -0.3, 0.0, 0.8, -1.0, 0.2, -0.6, 0.4, 0.1, -0.2], device="cuda")
    z = lambda *s: torch.zeros(*s, device="cuda")   # noqa: E731
    pols = [(z(H, od), z(H), z(H, H), z(H), z(15, H), torch.cat([mov, com])) for od in env.world.native.obs_dims]
    _, _, _, _, ex = env.rollout_policy(pols, T, record_actions=True, explore_seed=77)
    a = torch.cat([x.reshape(-1, 15) for x in ex["actions"]])
    joint = a[:, :5].argmax(-1) * 10 + a[:, 5:].argmax(-1)
    counts = torch.bincount(joint, minlength=50).cpu().numpy()
    p = torch.outer(torch.softmax(mov.double(), 0), torch.softmax(com.double(), 0)).reshape(-1).cpu().numpy()
    assert chisquare(counts, p * counts.sum()).pvalue > 1e-3, counts
    # deterministic: each head is exactly its softmax
    _, _, _, _, ex_d = env.rollout_policy(pols, 2, record_actions=True)
    want = torch.cat([torch.softmax(mov, 0), torch.softmax(com, 0)]).expand(n, 15)
    assert torch.allclose(ex_d["actions"][1][0], want, rtol=1e-6, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["simple_adversary", "simple_push"])
def test_old_entry_point_serves_adversary_and_push(tag):
    """mpe_rollout_policy (5-wide actors, depth 1) equals depth-1 mpe_collect bit for bit"""
    from multiagent_particle_envs_b200 import _lib
    n, T, H = 1031, 6, 64
    env_a = make_product_env(tag, num_envs=n, seed=4)
    env_b = make_product_env(tag, num_envs=n, seed=4)
    env_a.reset()
    env_b.reset()
    na, nb = env_a.world.native, env_b.world.native
    pols = _actors(na, H, seed=1, depth=1)
    obs_a, rew_a, _, _, ex = env_a.rollout_policy(pols, T, record_actions=True, per_step_rewards=True)
    parts = [(W1.t().contiguous(), b1, W2, b2) for W1, b1, W2, b2 in pols]
    ptrs = [_lib.ptr_array([p[k].data_ptr() for p in parts]) for k in range(4)]
    out = nb.new_outputs()
    rew_steps = torch.empty((T, env_b.n, n), device="cuda")
    acts = [torch.empty((T, n, 5), device="cuda") for _ in range(env_b.n)]
    nb.rollout_policy(*ptrs, H, T, out, env_b._flags(), rew_steps, _lib.ptr_array([a.data_ptr() for a in acts]))
    torch.cuda.synchronize()
    assert torch.equal(na.agent_pv, nb.agent_pv) and torch.equal(ex["rewards"], rew_steps)
    assert all(torch.equal(x, y) for x, y in zip(obs_a, out.obs))
    assert all(torch.equal(x, y) for x, y in zip(ex["actions"], acts))
    assert torch.equal(torch.stack(list(rew_a)), out.rew)


@pytest.mark.gpu
def test_refusals():
    from multiagent_particle_envs_b200 import _lib
    from multiagent_particle_envs_b200._lib import MpeError
    env = make_product_env("simple_reference", num_envs=1031)
    env.reset()
    nw = env.world.native
    five = [(t[0], t[1], t[2], t[3], t[4][:5].contiguous(), t[5][:5].contiguous()) for t in _actors(nw, 64, seed=0)]
    with pytest.raises(ValueError):                                          # 5-wide last layer on 15-wide agents
        env.rollout_policy(five, 2)
    # the old entry point keeps its 5-wide contract: speaking agents are refused
    W = _actors(nw, 32, seed=0, depth=1)
    parts = [(W1.t().contiguous(), b1, W2, b2) for W1, b1, W2, b2 in W]
    ptrs = [_lib.ptr_array([p[k].data_ptr() for p in parts]) for k in range(4)]
    with pytest.raises(MpeError):
        nw.rollout_policy(*ptrs, 32, 2, nw.new_outputs())
    env6 = make_product_env("simple_spread_n6", num_envs=64)
    env6.reset()
    with pytest.raises(MpeError):
        env6.rollout_policy(_actors(env6.world.native, 32, seed=0), 2)
