#!/usr/bin/env python
"""Collecting training experience: T closed-loop steps of obs -> per-agent actor -> (exploration) -> env.step with the
replay-buffer records (actions, per-step rewards, observations), as
  (a) ONE launch of mpe_collect (env.rollout_policy: actors inside the kernel, state in registers),
  (b) the same actors as torch modules + env.step captured in one CUDA graph (rollout.GraphedRollout), with Gumbel
      noise from torch.rand and the actions, rewards and observations copied into record buffers inside the graph.
One JSON line per configuration: device time per step of each (CUDA events over --reps calls after warm-up), env-steps/s,
their ratio, and the card's name and power limit."""
import argparse
import itertools
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return {"name": torch.cuda.get_device_name(0), "power_limit": limit}


def actors(obs_dims, act_dims, H, depth, dev):
    import torch
    nn = torch.nn
    torch.manual_seed(0)
    mods = []
    for od, ad in zip(obs_dims, act_dims):
        layers = [nn.Linear(od, H), nn.ReLU()] + ([nn.Linear(H, H), nn.ReLU()] if depth == 2 else []) + [nn.Linear(H, ad)]
        mods.append(nn.Sequential(*layers).to(dev))
    return mods


def action_heads(nw):
    """per agent, the column ranges of its action heads: 5 movement logits if it moves, then dim_c if it speaks"""
    heads = []
    for i in range(nw.n_agents):
        h, c = [], 0
        if nw.desc.agent_movable[i]:
            h.append((0, 5))
            c = 5
        if not nw.desc.agent_silent[i]:
            h.append((c, c + nw.dim_c))
        heads.append(h)
    return heads


def time_calls(fn, reps, stream=None):
    import torch
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s = stream or torch.cuda.current_stream()
    with torch.cuda.stream(s):
        e0.record(s)
        for _ in range(reps):
            fn()
        e1.record(s)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def measure(scenario, n, T, depth, H, sample, record, reps, dev):
    import torch
    from multiagent_particle_envs_b200 import make_env
    from multiagent_particle_envs_b200.rollout import GraphedRollout
    env = make_env(scenario, num_envs=n, device=dev)
    env.reuse_buffers = True
    env.reset()
    nw = env.world.native
    mods = actors(nw.obs_dims, nw.act_dims, H, depth, dev)
    heads = action_heads(nw)
    kw = dict(record_actions=record, per_step_rewards=record, record_observations=record)
    if sample:
        kw["explore_seed"] = 1
    sec_a = time_calls(lambda: env.rollout_policy(mods, T, **kw), reps) / T

    env2 = make_env(scenario, num_envs=n, device=dev)
    env2.reset()
    A = len(mods)
    rec = None
    if record:
        rec = dict(act=[torch.empty(T, n, ad, device=dev) for ad in nw.act_dims],
                   obs=[torch.empty(T, n, od, device=dev) for od in nw.obs_dims],
                   rew=torch.empty(T, A, n, device=dev))
    clock = {"t": 0}

    def policy(obs_n):
        t = clock["t"] % T
        clock["t"] += 1
        acts = []
        for i, (m, o) in enumerate(zip(mods, obs_n)):
            logits = m(o)
            if sample:
                u = torch.rand_like(logits)
                logits = logits - torch.log(-torch.log(u))
            if len(heads[i]) == 1:
                a = torch.softmax(logits, -1)
            else:     # one Gumbel-softmax per head, as MADDPG samples a MultiDiscrete action
                a = torch.cat([torch.softmax(logits[:, lo:hi], -1) for lo, hi in heads[i]], -1)
            if rec is not None:
                rec["obs"][i][t].copy_(o)
                rec["act"][i][t].copy_(a)
            acts.append(a)
        return acts

    if record:   # every step's rewards go to the record as well (the policy call of step t has just advanced the clock)
        step = env2.step

        def recording_step(action_n):
            out = step(action_n)
            rec["rew"][(clock["t"] - 1) % T].copy_(torch.stack(list(out[1])))
            return out
        env2.step = recording_step
    ro = GraphedRollout(env2, policy, steps=T)
    sec_b = time_calls(ro.run, reps, ro.stream) / T
    return {"config": {"scenario": scenario, "n_env": n, "T": T, "depth": depth, "hidden": H, "sample": sample,
                       "records": record},
            "collect": {"us_per_step": 1e6 * sec_a, "env_steps_per_sec": n / sec_a},
            "graphed_torch": {"us_per_step": 1e6 * sec_b, "env_steps_per_sec": n / sec_b},
            "speedup": sec_b / sec_a}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", default="simple_spread,simple_tag",
                    help="comma-separated, any of simple, simple_spread, simple_tag, simple_adversary, simple_push, "
                         "simple_speaker_listener, simple_reference, simple_crypto")
    ap.add_argument("--num-envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=25)
    ap.add_argument("--hidden", type=int, default=64)
    ap.add_argument("--depths", default="1,2")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("collect_bench.py measures on a CUDA device; none is available")
    import __graft_entry__ as g
    g.build(quiet=True)
    dev = torch.device("cuda", 0)
    info = card()
    for sc, depth, sample, record in itertools.product(args.scenarios.split(","), [int(d) for d in args.depths.split(",")],
                                                       (False, True), (False, True)):
        res = measure(sc, args.num_envs, args.steps, depth, args.hidden, sample, record, args.reps, dev)
        res["card"] = info
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
