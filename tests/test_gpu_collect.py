"""mpe_collect / env.rollout_policy as a source of training experience: two-hidden-layer actors, Gumbel-softmax
exploration from a Philox stream, and per-step observation records.  CPU tests (no marker): the NumPy Philox that the
GPU tests rebuild the noise with, argument checking of mpe_collect on a device-less handle, the actor parser.  GPU tests
(`gpu` marker): replay parity, float64 actor, the old entry point, continuation / sharding, the sampled distribution,
refusals."""
import ctypes

import numpy as np
import pytest

from helpers import descriptor, make_product_env

torch = pytest.importorskip("torch")

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123) on arrays: ctr = 4 arrays (or ints) of uint32 words, key = 2 words"""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in ctr]
    k0, k1 = np.uint64(key[0] & MASK), np.uint64(key[1] & MASK)
    for _ in range(10):
        p0, p1 = c[0] * np.uint64(M0), c[2] * np.uint64(M1)
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & np.uint64(MASK), (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & np.uint64(MASK)]
        k0, k1 = (k0 + np.uint64(W0)) & np.uint64(MASK), (k1 + np.uint64(W1)) & np.uint64(MASK)
    return [x.astype(np.uint32) for x in c]


def exploration_uniforms(seed, worlds, step, agent):
    """the five u of (global worlds [N], step, agent) as the kernel draws them: float64 [N, 5], exact"""
    worlds = np.asarray(worlds, dtype=np.uint64)
    lo, hi = worlds & np.uint64(MASK), worlds >> np.uint64(32)
    key = (seed & MASK, seed >> 32)
    words = []
    for block in (0, 1):
        tag = 0x40000000 | (agent << 1) | block
        words += philox4x32_10((lo, hi, np.full_like(lo, step), np.full_like(lo, tag)), key)
    bits = np.stack(words[:5], 1).astype(np.uint64)
    return (2.0 * (bits >> np.uint64(9)).astype(np.float64) + 1.0) * 2.0 ** -24


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_numpy_philox_reproduces_the_random123_known_answers():
    def hexs(ctr, key):
        return ["%08x" % int(v) for v in philox4x32_10(ctr, key)]
    assert hexs((0, 0, 0, 0), (0, 0)) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    assert hexs((MASK,) * 4, (MASK, MASK)) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert hexs((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]
    u = exploration_uniforms(2 ** 40 + 7, np.arange(1000), 3, 2)
    assert u.shape == (1000, 5) and u.min() > 0.0 and u.max() < 1.0
    assert np.all(u.astype(np.float32).astype(np.float64) == u)          # exact in fp32


def _collect_call(lib, h, A, depth=2, hidden=64, w1=True, n_steps=4, sample_step=0):
    """mpe_collect with well-formed (fake, aligned) pointers except where a test breaks one; no device is touched"""
    arr = lambda: (ctypes.c_void_p * A)(*([256] * A))   # noqa: E731
    w1_n = arr() if w1 else None
    w3 = arr() if depth == 2 else None
    return lib.mpe_collect(h, 256, 256, None, None, depth, hidden, w1_n, arr(), arr(), arr(), w3,
                           arr() if depth == 2 else None, n_steps, 1, sample_step, 0, arr(), 256, None, None, arr(),
                           256, 16, None)


def test_collect_refuses_bad_arguments_without_a_device():
    from multiagent_particle_envs_b200 import _lib
    from multiagent_particle_envs_b200.native import ShapeHandle
    sh = ShapeHandle(descriptor("simple_spread_n3"), 1031, -1)
    lib, h, A = sh.lib, sh.handle, sh.n_agents
    assert _collect_call(lib, h, A) == _lib.ERR_NO_DEVICE
    assert _collect_call(lib, h, A, depth=1) == _lib.ERR_NO_DEVICE
    assert _collect_call(lib, h, A, w1=False) == _lib.ERR_BAD_ARG
    assert _collect_call(lib, h, A, depth=3) == _lib.ERR_BAD_ARG
    assert _collect_call(lib, h, A, hidden=48) == _lib.ERR_BAD_ARG
    assert _collect_call(lib, h, A, n_steps=-1) == _lib.ERR_BAD_ARG
    assert _collect_call(lib, h, A, n_steps=4, sample_step=2 ** 32 - 4) == _lib.ERR_NO_DEVICE
    assert _collect_call(lib, h, A, n_steps=5, sample_step=2 ** 32 - 4) == _lib.ERR_BAD_ARG
    nulls = (ctypes.c_void_p * A)(*([256] * (A - 1) + [0]))                # one agent's W1 missing
    arr = lambda: (ctypes.c_void_p * A)(*([256] * A))   # noqa: E731
    assert lib.mpe_collect(h, 256, 256, None, None, 1, 32, nulls, arr(), arr(), arr(), None, None, 4, 0, 0, 0, arr(),
                           256, None, None, None, 256, 0, None) == _lib.ERR_BAD_ARG
    assert lib.mpe_collect(h, 256, 256, None, None, 1, 32, arr(), arr(), arr(), arr(), arr(), arr(), 4, 0, 0, 0, arr(),
                           256, None, None, None, 256, 0, None) == _lib.ERR_BAD_ARG     # depth 1 takes no W3
    sh.close()


def _linear(i, o):
    return torch.nn.Linear(i, o)


def test_actor_parser_accepts_and_rejects():
    from multiagent_particle_envs_b200.environment import actor_parameters
    nn = torch.nn
    od = [18, 18, 18]
    d1 = [nn.Sequential(_linear(o, 64), nn.ReLU(), _linear(64, 5)) for o in od]
    depth, H, p = actor_parameters(d1, od)
    assert (depth, H) == (1, 64) and len(p[0]) == 4 and p[0][2] is d1[0][2].weight
    d2 = [nn.Sequential(_linear(o, 32), nn.ReLU(), _linear(32, 32), nn.ReLU(), _linear(32, 5)) for o in od]
    depth, H, p = actor_parameters(d2, od)
    assert (depth, H) == (2, 32) and len(p[0]) == 6 and p[1][4] is d2[1][4].weight
    tup = [tuple(t.detach() for t in (m[0].weight, m[0].bias, m[2].weight, m[2].bias, m[4].weight, m[4].bias)) for m in d2]
    assert actor_parameters(tup, od)[:2] == (2, 32)
    tanh = [nn.Sequential(_linear(o, 32), nn.Tanh(), _linear(32, 32), nn.ReLU(), _linear(32, 5)) for o in od]
    with pytest.raises(ValueError):
        actor_parameters(tanh, od)
    with pytest.raises(ValueError):                                          # mixed depths
        actor_parameters(d2[:2] + [nn.Sequential(_linear(18, 32), nn.ReLU(), _linear(32, 5))], od)
    with pytest.raises(ValueError):                                          # mixed widths
        actor_parameters(d2[:2] + [nn.Sequential(_linear(18, 64), nn.ReLU(), _linear(64, 64), nn.ReLU(), _linear(64, 5))], od)
    with pytest.raises(ValueError):                                          # wrong observation width
        actor_parameters(d2, [18, 18, 16])
    with pytest.raises(ValueError):                                          # 5-tuple
        actor_parameters([t[:5] for t in tup], od)
    with pytest.raises(ValueError):                                          # W2 not square
        actor_parameters([(t[0], t[1], t[2][:, :16], t[3], t[4], t[5]) for t in tup], od)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _actors(obs_dims, H, seed, depth=2):
    """torch-default-initialised actors (logits of order one, as in training), as 6- or 4-tuples on the GPU"""
    torch.manual_seed(seed)
    out = []
    for od in obs_dims:
        layers = [_linear(od, H)] + ([_linear(H, H)] if depth == 2 else []) + [_linear(H, 5)]
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


def _gumbel64(seed, world_offset, n, step, agent):
    u = exploration_uniforms(seed, world_offset + np.arange(n, dtype=np.uint64), step, agent)
    return torch.from_numpy(-np.log(-np.log(u))).cuda()


PARITY = [(tag, n, H, s) for tag in ("simple_spread_n3", "simple_tag", "simple") for H in (32, 64) for s in (None, 11)
          for n in (1031,)] + [(tag, 65536, 64, s) for tag in ("simple_spread_n3", "simple_tag") for s in (None, 2 ** 33 + 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("tag,n,H,seed", PARITY)
def test_depth2_replay_parity_and_float64_actor(tag, n, H, seed):
    """Depth-2 actors, deterministic and sampled, with every record on:
      (1) the recorded actions fed to T `env.step` calls of a twin env reproduce the final state, final observations,
          every step's rewards and the reward sums BIT FOR BIT, and observation record row t is bit-equal to what the
          twin returned before step t;
      (2) every recorded action equals the float64 three-layer actor on the twin's observations (sampled: plus the
          Gumbel term -log(-log u) with u rebuilt by the NumPy Philox) to rtol 1e-5, atol 1e-6.  The fp32 noise adds at
          most ~2e-6 to a logit (|g| < 17: half an ulp of g and of logit + g, plus logf's 1-ulp error through the
          outer log, ~1e-7), which moves a probability p by at most p (1 - p) 2e-6 <= 5e-7: within the tolerance."""
    T, step0 = 7, 3
    env_a = make_product_env(tag, num_envs=n, seed=9)
    env_b = make_product_env(tag, num_envs=n, seed=9)
    env_a.reset()
    obs_b = env_b.reset()
    na, nb = env_a.world.native, env_b.world.native
    pols = _actors(na.obs_dims, H, seed=H + n)
    obs_r, rew_r, done_r, _, ex = env_a.rollout_policy(pols, T, record_actions=True, per_step_rewards=True,
                                                       record_observations=True, explore_seed=seed,
                                                       explore_step=step0 if seed is not None else 0)
    actions, rew_steps, obs_rec = ex["actions"], ex["rewards"], ex["observations"]
    assert [tuple(o.shape) for o in obs_rec] == [(T, n, od) for od in na.obs_dims]
    rew_sum = torch.zeros(env_b.n, n, device="cuda")
    for t in range(T):
        for i, pol in enumerate(pols):
            assert torch.equal(obs_rec[i][t], obs_b[i]), (t, i)
            logits = _actor64(pol, obs_b[i])
            if seed is not None:
                logits = logits + _gumbel64(seed, 0, n, step0 + t, i)
            want = torch.softmax(logits, -1)
            assert torch.allclose(actions[i][t].double(), want, rtol=1e-5, atol=1e-6), (t, i)
        obs_b, rew_s, _, _ = env_b.step([a[t] for a in actions])
        rew_sum += torch.stack(list(rew_s))
        assert torch.equal(rew_steps[t], torch.stack(list(rew_s))), t
    torch.cuda.synchronize()
    assert torch.equal(na.agent_pv, nb.agent_pv)
    assert all(torch.equal(x, y) for x, y in zip(obs_r, obs_b))
    assert torch.equal(torch.stack(list(rew_r)), rew_sum)
    assert not any(bool(d.any()) for d in done_r)


@pytest.mark.gpu
@pytest.mark.parametrize("tag,n,H", [("simple_spread_n3", 1031, 64), ("simple_tag", 65536, 32), ("simple", 1031, 32)])
def test_depth1_through_collect_matches_the_old_entry_point(tag, n, H):
    """depth 1, deterministic, through mpe_collect (env.rollout_policy) is bit-equal to mpe_rollout_policy"""
    from multiagent_particle_envs_b200 import _lib
    T = 6
    env_a = make_product_env(tag, num_envs=n, seed=4)
    env_b = make_product_env(tag, num_envs=n, seed=4)
    env_a.reset()
    env_b.reset()
    na, nb = env_a.world.native, env_b.world.native
    pols = _actors(na.obs_dims, H, seed=1, depth=1)
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


def _run(env, pols, T, seed, step):
    obs, rew, _, _, ex = env.rollout_policy(pols, T, record_actions=True, per_step_rewards=True, record_observations=True,
                                            explore_seed=seed, explore_step=step)
    return [o.clone() for o in obs], ex


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1031, 65536])
def test_continuation_sharding_and_seeds(n):
    """Sampled depth-2 rollouts: two calls (explore_step 0, then T/2) equal one call of T steps; each rank of a two-rank
    sharded env reproduces its half of the full batch; the same seed repeats exactly, another seed changes the actions."""
    tag, T, seed = "simple_spread_n3", 8, 123
    full = make_product_env(tag, num_envs=n, seed=2)
    full.reset()
    pols = _actors(full.world.native.obs_dims, 64, seed=5)
    obs_f, ex_f = _run(full, pols, T, seed, 0)
    pv_f = full.world.native.agent_pv.clone()
    # continuation
    env = make_product_env(tag, num_envs=n, seed=2)
    env.reset()
    _, ex1 = _run(env, pols, T // 2, seed, 0)
    obs2, ex2 = _run(env, pols, T // 2, seed, T // 2)
    assert torch.equal(env.world.native.agent_pv, pv_f)
    assert all(torch.equal(x, y) for x, y in zip(obs2, obs_f))
    assert torch.equal(torch.cat([ex1["rewards"], ex2["rewards"]]), ex_f["rewards"])
    for key in ("actions", "observations"):
        assert all(torch.equal(torch.cat([a, b]), c) for a, b, c in zip(ex1[key], ex2[key], ex_f[key])), key
    # sharding: rank r owns a contiguous range and draws with its global world indices
    from multiagent_particle_envs_b200.sharding import shard_range
    for r in range(2):
        lo, hi = shard_range(n, r, 2)
        sh = make_product_env(tag, num_envs=n, seed=2, rank=r, world_size=2)
        sh.reset()
        obs_s, ex_s = _run(sh, pols, T, seed, 0)
        assert torch.equal(sh.world.native.agent_pv, pv_f[:, lo:hi])
        assert all(torch.equal(x, y[lo:hi]) for x, y in zip(obs_s, obs_f))
        assert torch.equal(ex_s["rewards"], ex_f["rewards"][:, :, lo:hi])
        for key in ("actions", "observations"):
            assert all(torch.equal(x, y[:, lo:hi]) for x, y in zip(ex_s[key], ex_f[key])), (r, key)
    # same seed -> same actions; another seed -> different ones
    again = make_product_env(tag, num_envs=n, seed=2)
    again.reset()
    _, ex_r = _run(again, pols, T, seed, 0)
    assert all(torch.equal(x, y) for x, y in zip(ex_r["actions"], ex_f["actions"]))
    other = make_product_env(tag, num_envs=n, seed=2)
    other.reset()
    _, ex_o = _run(other, pols, T, seed + 1, 0)
    assert not torch.equal(ex_o["actions"][0][0], ex_f["actions"][0][0])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1031, 65536])
def test_sampled_argmax_follows_softmax_of_the_logits(n):
    """All weights zero and b3 = l, so the logits are l: by the Gumbel-max property the arg-max of the sampled action
    is distributed as softmax(l).  Chi-square goodness of fit over every (world, step, agent) sample; the seed is fixed,
    so the test is deterministic."""
    from scipy.stats import chisquare
    tag, T, H = "simple_spread_n3", 64 if n < 10000 else 4, 32
    env = make_product_env(tag, num_envs=n, seed=3)
    env.reset()
    ell = torch.tensor([0.3, -1.2, 1.0, 0.0, -0.4], device="cuda")
    z = lambda *s: torch.zeros(*s, device="cuda")   # noqa: E731
    pols = [(z(H, od), z(H), z(H, H), z(H), z(5, H), ell.clone()) for od in env.world.native.obs_dims]
    _, _, _, _, ex = env.rollout_policy(pols, T, record_actions=True, explore_seed=77)
    arg = torch.cat([a.reshape(-1, 5) for a in ex["actions"]]).argmax(-1)
    counts = torch.bincount(arg, minlength=5).cpu().numpy()
    expected = torch.softmax(ell.double(), 0).cpu().numpy() * counts.sum()
    assert chisquare(counts, expected).pvalue > 1e-3, (counts, expected)
    # and the deterministic path acts with softmax(l) exactly as before
    _, _, _, _, ex_d = env.rollout_policy(pols, 2, record_actions=True)
    assert torch.allclose(ex_d["actions"][0][0], torch.softmax(ell, 0).expand(n, 5), rtol=1e-6, atol=1e-7)


@pytest.mark.gpu
def test_collect_refusals():
    from multiagent_particle_envs_b200._lib import MpeError
    env_w = make_product_env("simple_world_comm", num_envs=64)
    env_w.reset()
    with pytest.raises(MpeError):
        env_w.rollout_policy(_actors(env_w.world.native.obs_dims, 32, seed=0), 2, explore_seed=1)
    env = make_product_env("simple_spread_n3", num_envs=1031)
    env.reset()
    od = env.world.native.obs_dims
    nn = torch.nn
    tanh = [nn.Sequential(_linear(o, 64), nn.ReLU(), _linear(64, 64), nn.Tanh(), _linear(64, 5)).cuda() for o in od]
    with pytest.raises(ValueError):
        env.rollout_policy(tanh, 2)
    mixed = _actors(od, 64, seed=0)[:2] + _actors(od, 64, seed=0, depth=1)[2:]
    with pytest.raises(ValueError):
        env.rollout_policy(mixed, 2)
    pols = _actors(od, 64, seed=0)
    with pytest.raises(ValueError):
        env.rollout_policy(pols, 4, explore_seed=1, explore_step=2 ** 32 - 4)
    env.rollout_policy(pols, 4, explore_seed=1, explore_step=2 ** 32 - 5)          # the last step that fits
