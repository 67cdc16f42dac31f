"""Generates the golden fixtures in this directory by running the UNMODIFIED Python reference
(/root/reference, imported through oracle/refshim.py) -- run in the build container only:

    python tests/golden/make_golden.py

For every BASELINE.json scenario it records W worlds x T steps of `MultiAgentEnv.step`
(environment.py:80-104): initial state, the actions fed, and after every step the state, the
observations, rewards, dones and benchmark_data.  Initial states come from the reference's own
reset_world; odd worlds are then squeezed (positions scaled) so that contacts are frequent, and
some worlds start outside the arena so that tag's bound() penalty is exercised.  `kat.npz` holds
the known-answer trajectories of SURVEY.md section 8(c) (np.random.seed(0); reset; 2 steps).

The fixtures pin oracle/mpe_oracle.c (tests/test_oracle_golden.py) and, through it and directly,
the CUDA kernels (tests/test_gpu_parity.py).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
sys.path.insert(0, os.path.join(HERE, ".."))
import refshim  # noqa: E402
from helpers import PER_WORLD  # noqa: E402

MAX_FILE_BYTES = 1000000   # a fixture that would be larger is stored as <tag>.part<k>.npz, split along the worlds

# (scenario, entity-count override, worlds W, recorded steps T): W x T >= 1536 reference steps per scenario
CONFIGS = [
    ("simple_adversary", None, 256, 6),
    ("simple_push", None, 256, 6),
    ("simple_speaker_listener", None, 256, 6),
    ("simple_reference", None, 256, 6),
    ("simple_crypto", None, 256, 6),
    ("simple", None, 256, 6),
    ("simple_spread", 3, 256, 8),
    ("simple_spread", 6, 256, 6),
    ("simple_tag", None, 256, 8),
    ("simple_world_comm", None, 256, 6),
]
PREROLL = 50   # worlds 4..7 (mod 8) first run this many unrecorded reference steps: contact equilibria,
#                clustered agents pushing against each other, prey pinned against obstacles


SEEDS = {"simple": 1, "simple_spread_n3": 2, "simple_spread_n6": 3, "simple_tag": 4, "simple_world_comm": 5,
         "simple_adversary": 11, "simple_push": 12, "simple_speaker_listener": 13, "simple_reference": 14,
         "simple_crypto": 15}


def act_dim(space):
    return int(space.n) if hasattr(space, "n") else int(np.sum(space.high - space.low + 1))


def world_props(world):
    """entity properties as make_world() left them (pins the product's descriptors)"""
    ag, lm = world.agents, world.landmarks
    return dict(
        dim_c=world.dim_c, dt=world.dt, damping=world.damping, contact_force=world.contact_force,
        contact_margin=world.contact_margin,
        agent_size=[a.size for a in ag], agent_mass=[a.mass for a in ag],
        agent_accel=[-1.0 if a.accel is None else a.accel for a in ag],
        agent_max_speed=[-1.0 if a.max_speed is None else a.max_speed for a in ag],
        agent_movable=[int(a.movable) for a in ag], agent_collide=[int(a.collide) for a in ag],
        agent_silent=[int(a.silent) for a in ag],
        agent_adversary=[int(getattr(a, "adversary", False)) for a in ag],
        agent_leader=[int(getattr(a, "leader", False)) for a in ag],
        landmark_size=[l.size for l in lm], landmark_collide=[int(l.collide) for l in lm],
        landmark_movable=[int(l.movable) for l in lm],
        collaborative=int(getattr(world, "collaborative", False)),
    )


def snapshot(world):
    pv = np.array([np.concatenate([a.state.p_pos, a.state.p_vel]) for a in world.agents])
    comm = np.array([np.asarray(a.state.c, dtype=np.float64) for a in world.agents]).reshape(len(world.agents), world.dim_c)
    return pv, comm


def goals_of(name, world):
    """per-world goal indices chosen by reset_world (np.random.choice(world.landmarks))"""
    lms = world.landmarks
    idx = lambda e: [i for i, l in enumerate(lms) if l is e][0]  # noqa: E731
    if name in ("simple_adversary", "simple_push"):
        return [idx(world.agents[0].goal_a)]
    if name == "simple_speaker_listener":
        return [idx(world.agents[0].goal_b)]
    if name == "simple_reference":
        return [idx(world.agents[0].goal_b), idx(world.agents[1].goal_b)]
    if name == "simple_crypto":
        return [idx(world.agents[0].goal_a), int(np.argmax(world.agents[2].key))]
    return []


def flatten_info(name, info_n):
    out = []
    for item in info_n["n"]:
        if isinstance(item, dict):
            out.append([])
        elif isinstance(item, tuple):
            out.append([float(v) for part in item for v in np.atleast_1d(part)])
        else:
            out.append([float(item)])
    width = max(len(r) for r in out)
    return np.array([r + [0.0] * (width - len(r)) for r in out], dtype=np.float64)   # ragged rows zero-padded


def run_config(name, n, W, T, seed, force_discrete=False, discrete_input=False):
    rng = np.random.RandomState(seed)
    rec = dict(pv0=[], lm=[], comm0=[], goal=[], act=[], pv=[], comm=[], obs=[], rew=[], done=[], info=[])
    props = None
    for w in range(W):
        np.random.seed(seed * 1000 + w)
        env = refshim.make_reference_env(name, n)
        env.force_discrete_action = force_discrete
        env.discrete_action_input = discrete_input      # integer actions (environment.py:161-167)
        env.reset()
        world = env.world
        if props is None:
            props = world_props(world)
            props["obs_dims"] = [int(s.shape[0]) for s in env.observation_space]
            props["act_dims"] = [act_dim(s) for s in env.action_space]
            props["shared_reward"] = int(env.shared_reward)
        mode = w % 4
        preroll = PREROLL if (w % 8) >= 4 else 0
        if mode == 1:      # squeezed: many contacts
            for e in world.entities:
                e.state.p_pos = e.state.p_pos * 0.3
        elif mode == 2:    # agents near / beyond the arena edge, moving fast
            for a in world.agents:
                a.state.p_pos = a.state.p_pos * 1.25
                a.state.p_vel = rng.uniform(-1.5, 1.5, 2)
        elif mode == 3:    # very tight cluster: deep penetrations
            for a in world.agents:
                a.state.p_pos = rng.uniform(-0.12, 0.12, 2)
        pv0, comm0 = snapshot(world)
        rec["goal"].append(np.array(goals_of(name, world), dtype=np.int32))
        rec["pv0"].append(pv0)
        rec["comm0"].append(comm0)
        rec["lm"].append(np.array([l.state.p_pos for l in world.landmarks]))
        steps = {k: [] for k in ("act", "pv", "comm", "obs", "rew", "done", "info")}
        temperature = [1.0, 3.0, 0.3, 6.0][mode]
        drift = rng.randn(env.n, 5)
        for t in range(-preroll, T):
            acts = []
            for i, sp in enumerate(env.action_space):
                d = act_dim(sp)
                if discrete_input:
                    acts.append(np.array([float(rng.randint(0, d))]))
                    continue
                if not world.agents[i].movable:          # speaker-only agents: the comm chunk
                    a = rng.uniform(0, 1, d) * (rng.uniform() > 0.15)   # sometimes an all-zero utterance
                else:
                    logits = temperature * rng.randn(5)
                    logits += 2.0 * drift[i] if mode in (2, 3) else 0.0
                    p = np.exp(logits - logits.max())
                    a = np.concatenate([p / p.sum(), rng.uniform(0, 1, d - 5)]) if d > 5 else p / p.sum()
                acts.append(a)
            if t == 0 and preroll:      # the recorded trajectory starts from the equilibrated state
                rec["pv0"][-1], rec["comm0"][-1] = snapshot(world)
            obs_n, rew_n, done_n, info_n = env.step([int(a[0]) for a in acts] if discrete_input else [a.copy() for a in acts])
            if t < 0:
                continue
            pv, comm = snapshot(world)
            steps["act"].append(np.concatenate(acts))
            steps["pv"].append(pv)
            steps["comm"].append(comm)
            steps["obs"].append(np.concatenate(obs_n))
            steps["rew"].append(np.array(rew_n, dtype=np.float64))
            steps["done"].append(np.array(done_n, dtype=np.uint8))
            steps["info"].append(flatten_info(name, info_n))
        for k, v in steps.items():
            rec[k].append(np.array(v))
    out = {k: np.array(v) for k, v in rec.items()}
    for k, v in props.items():
        out["prop_" + k] = np.array(v)
    out["force_discrete"] = np.array(int(force_discrete))
    out["discrete_input"] = np.array(int(discrete_input))
    return out


def kat():
    """SURVEY.md 8(c): np.random.seed(0); env = make_env(name); env.reset(); two steps with
    one-hot actions (agent i presses index i+1; `simple` presses index 2)."""
    out = {}
    for name in ("simple", "simple_spread", "simple_tag", "simple_world_comm"):
        np.random.seed(0)
        env = refshim.make_reference_env(name)
        env.reset()
        pv0, comm0 = snapshot(env.world)
        lm = np.array([l.state.p_pos for l in env.world.landmarks])
        acts = []
        for i, sp in enumerate(env.action_space):
            d = act_dim(sp)
            a = np.zeros(d)
            a[2 if name == "simple" else min(i + 1, 4)] = 1.0
            acts.append(a)
        for _ in range(2):
            obs_n, rew_n, done_n, info_n = env.step([a.copy() for a in acts])
        pv, comm = snapshot(env.world)
        out[name + "/pv0"], out[name + "/lm"], out[name + "/comm0"] = pv0, lm, comm0
        out[name + "/act"] = np.concatenate(acts)
        out[name + "/pv"], out[name + "/comm"] = pv, comm
        out[name + "/obs"] = np.concatenate(obs_n)
        out[name + "/rew"] = np.array(rew_n, dtype=np.float64)
        out[name + "/done"] = np.array(done_n, dtype=np.uint8)
    return out


def save(tag, data):
    path = os.path.join(HERE, tag + ".npz")
    np.savez_compressed(path, **data)
    parts = -(-os.path.getsize(path) // (MAX_FILE_BYTES * 9 // 10))      # 10 % headroom: parts differ in size
    if parts == 1:
        return
    os.remove(path)
    bounds = np.linspace(0, len(data["pv0"]), parts + 1).astype(int)
    for k in range(parts):
        part_path = os.path.join(HERE, "%s.part%d.npz" % (tag, k))
        np.savez_compressed(part_path, **{key: v[bounds[k]:bounds[k + 1]] if key in PER_WORLD else v for key, v in data.items()})
        assert os.path.getsize(part_path) < MAX_FILE_BYTES, part_path


def main():
    only = sys.argv[1:]
    for idx, (name, n, W, T) in enumerate(CONFIGS):
        if only and name not in only:
            continue
        tag = name + ("_n%d" % n if n else "")
        data = run_config(name, n, W, T, seed=SEEDS[tag])
        save(tag, data)
        print(tag, {k: v.shape for k, v in data.items() if not k.startswith("prop_")})
    if only:
        return
    data = run_config("simple_tag", None, 64, 8, seed=77, force_discrete=True)
    save("simple_tag_force_discrete", data)
    data = run_config("simple_tag", None, 64, 8, seed=78, discrete_input=True)
    save("simple_tag_discrete_input", data)
    for counts, tag in (((1, 1, 2), "simple_tag_1v1"), ((4, 2, 2), "simple_tag_4v2"), ((6, 2, 3), "simple_tag_6v2")):
        data = run_config("simple_tag", counts, 64, 6, seed=80 + counts[0])     # entity-count variants
        save(tag, data)
    np.savez_compressed(os.path.join(HERE, "kat.npz"), **kat())


if __name__ == "__main__":
    main()
