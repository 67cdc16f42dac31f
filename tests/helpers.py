"""shared test helpers (the oracle is imported HERE, in tests/, only as the checker)"""
import glob
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# golden tag -> (scenario name, scenario kwargs)
CONFIGS = {
    "simple": ("simple", {}),
    "simple_spread_n3": ("simple_spread", {}),
    "simple_spread_n6": ("simple_spread", {"num_agents": 6}),
    "simple_tag": ("simple_tag", {}),
    "simple_world_comm": ("simple_world_comm", {}),
    "simple_adversary": ("simple_adversary", {}),
    "simple_push": ("simple_push", {}),
    "simple_speaker_listener": ("simple_speaker_listener", {}),
    "simple_reference": ("simple_reference", {}),
    "simple_crypto": ("simple_crypto", {}),
}
# entity-count variants the reference hard-codes away (no goldens; checked against the generic oracle)
VARIANTS = {
    "simple_tag_1v1": ("simple_tag", {"num_adversaries": 1, "num_good_agents": 1, "num_landmarks": 2}),
    "simple_tag_2v1": ("simple_tag", {"num_adversaries": 2, "num_good_agents": 1, "num_landmarks": 2}),
    "simple_tag_4v2": ("simple_tag", {"num_adversaries": 4, "num_good_agents": 2, "num_landmarks": 2}),
    "simple_tag_6v2": ("simple_tag", {"num_adversaries": 6, "num_good_agents": 2, "num_landmarks": 3}),
    "simple_adversary_n4": ("simple_adversary", {"num_agents": 4}),
}
NO_BENCHMARK = ("simple", "simple_push", "simple_speaker_listener", "simple_reference")


# arrays of a fixture with one row per recorded world; the rest (prop_*, flags) describe the whole scenario
PER_WORLD = ("pv0", "lm", "comm0", "goal", "act", "pv", "comm", "obs", "rew", "done", "info")


def load_golden(tag):
    """one fixture; a fixture stored as <tag>.part<k>.npz (each file stays below 1 MB) is joined along the worlds"""
    path = os.path.join(GOLDEN, tag + ".npz")
    if os.path.exists(path):
        return dict(np.load(path))
    parts = [dict(np.load(p)) for p in sorted(glob.glob(os.path.join(GOLDEN, tag + ".part*.npz")))]
    if not parts:
        raise FileNotFoundError(path)
    g = parts[0]
    for k in PER_WORLD:
        g[k] = np.concatenate([p[k] for p in parts])
    return g


def make_product_env(tag, **kw):
    from multiagent_particle_envs_b200 import make_env
    name, skw = CONFIGS[tag] if tag in CONFIGS else VARIANTS[tag]
    kw.update(skw)
    return make_env(name, benchmark=(name not in NO_BENCHMARK), **kw)


def descriptor(tag):
    from multiagent_particle_envs_b200 import scenarios
    name, kw = CONFIGS[tag] if tag in CONFIGS else VARIANTS[tag]
    return scenarios.load(name).Scenario(**kw).make_world().descriptor()


def step_flags(tag_or_golden):
    from multiagent_particle_envs_b200 import _lib
    g = load_golden(tag_or_golden) if isinstance(tag_or_golden, str) else tag_or_golden
    f = 0
    if int(g["prop_shared_reward"]):
        f |= _lib.FLAG_SHARED_REWARD
    if int(g["force_discrete"]):
        f |= _lib.FLAG_FORCE_DISCRETE_ACTION
    return f


def random_states(desc, n, rng, mode="mixed"):
    """seeded synthetic worlds in the oracle layout: reset-like, squeezed (contacts), fast/outside"""
    A, L, C = desc.n_agents, desc.n_landmarks, desc.dim_c
    pv = np.zeros((n, A, 4))
    pv[:, :, 0:2] = rng.uniform(-1, 1, (n, A, 2))
    lm = rng.uniform(-0.9, 0.9, (n, L, 2))
    kind = rng.randint(0, 4, n) if mode == "mixed" else np.zeros(n, int)
    sq = kind == 1
    pv[sq, :, 0:2] *= 0.3
    lm[sq] *= 0.3
    fast = kind == 2
    pv[fast, :, 0:2] *= 1.25
    pv[fast, :, 2:4] = rng.uniform(-1.5, 1.5, (int(fast.sum()), A, 2))
    tight = kind == 3
    pv[tight, :, 0:2] = rng.uniform(-0.12, 0.12, (int(tight.sum()), A, 2))
    comm = np.zeros((n, A, C))
    for i in range(A):
        if not desc.agent_silent[i]:
            comm[:, i, :] = rng.uniform(0, 1, (n, C)) * (rng.uniform(0, 1, (n, 1)) > 0.1)
        if not desc.agent_movable[i]:
            pv[:, i, 2:4] = 0.0
    return pv, lm, comm


def random_goals(n_goals, n_landmarks, n, rng):
    return rng.randint(0, max(n_landmarks, 1), (n, n_goals)).astype(np.int32)


def random_actions(act_dims, n, rng, temperature=2.0, movable=None):
    """probability vectors as MADDPG emits (softmax of logits) + uniform comm"""
    parts = []
    for i, d in enumerate(act_dims):
        mov = True if movable is None else bool(movable[i])
        if mov:
            logits = temperature * rng.randn(n, 5)
            p = np.exp(logits - logits.max(axis=1, keepdims=True))
            p /= p.sum(axis=1, keepdims=True)
            parts.append(p)
            d -= 5
        if d > 0:
            parts.append(rng.uniform(0, 1, (n, d)) * (rng.uniform(0, 1, (n, 1)) > 0.1))
    return np.concatenate(parts, axis=1)


def split_cols(a, dims):
    out, c = [], 0
    for d in dims:
        out.append(a[..., c:c + d])
        c += d
    return out


# ---- accounting for contact-indicator mismatches between fp32 and fp64 ---------------------------------
# Rewards / benchmark_data contain indicator terms ([dist < size_a + size_b], [min dist < 0.1]).  An fp32
# evaluation may legitimately flip one when the fp64 distance sits within rounding of its threshold.  Every
# mismatch must be explained that way: (1) the difference is an integer multiple of the scenario's contact
# quantum and (2) some entity pair of that world is within `margin` of a threshold in the fp64 reference state.
CONTACT_QUANTUM = {"simple_spread": 1.0, "simple_tag": 10.0, "simple_world_comm": 1.0}   # world_comm: 5a + 2b
INFO_QUANTUM = 1.0                                                                       # counts


def scenario_of(tag):
    for name in ("simple_spread", "simple_tag", "simple_world_comm"):
        if tag.startswith(name):
            return name
    return tag


def threshold_margin(scn, pv_post, lm, a_size, l_size):
    """per world: min over entity pairs of |dist - threshold| in the given (fp64) post-step state"""
    p = np.asarray(pv_post, dtype=np.float64)[:, :, 0:2]
    lm = np.asarray(lm, dtype=np.float64)
    n, A = p.shape[:2]
    best = np.full(n, np.inf)
    for i in range(A):
        for j in range(i + 1, A):
            d = np.sqrt(((p[:, i] - p[:, j]) ** 2).sum(-1))
            best = np.minimum(best, np.abs(d - (a_size[i] + a_size[j])))
        for l in range(lm.shape[1]):
            d = np.sqrt(((p[:, i] - lm[:, l]) ** 2).sum(-1))
            best = np.minimum(best, np.abs(d - (a_size[i] + l_size[l])))
            if scn == "simple_spread":
                best = np.minimum(best, np.abs(d - 0.1))      # occupied_landmarks (simple_spread.py:56-57)
    return best


def explain_flag_mismatches(tag, rew, ref_rew, info, ref_info, pv_post64, lm64, a_size, l_size,
                            rtol=1e-5, atol=5e-6, margin=2e-6):
    """assert that every reward / info mismatch is a flipped contact indicator; returns #worlds with one"""
    scn = scenario_of(tag)
    ok = np.isclose(rew, ref_rew, rtol=rtol, atol=atol)
    bad = ~ok.all(axis=1)
    oki = None
    if info is not None and info.size:
        oki = np.isclose(info, ref_info, rtol=rtol, atol=atol)
        bad |= ~oki.reshape(oki.shape[0], -1).all(axis=1)
    if not bad.any():
        return 0
    q = CONTACT_QUANTUM.get(scn)
    assert q is not None, "%s has no contact indicators: reward mismatch in worlds %s" % (tag, np.where(bad)[0][:8])
    m = threshold_margin(scn, pv_post64, lm64, a_size, l_size)
    assert (m[bad] < margin).all(), "unexplained mismatch: worlds %s have no pair within %g of a threshold (margins %s)" % (
        np.where(bad)[0][:8], margin, m[bad][:8])
    d = (np.asarray(rew, np.float64) - ref_rew)[~ok] / q
    assert (np.abs(d - np.round(d)) < 1e-3).all() and (np.round(d) != 0).all(), "reward difference is not a multiple of %g: %s" % (q, d[:8])
    if oki is not None:
        di = (np.asarray(info, np.float64) - ref_info)[~oki]
        # counts differ by integers; simple_spread's info[0] is the reward itself (quantum 1 as well)
        assert (np.abs(di - np.round(di)) < 1e-3).all(), di[:8]
    return int(bad.sum())
