#!/usr/bin/env python
"""bench.py -- env-steps/sec of the multiagent-particle-envs hot path on B200.

    python bench.py --gpus N --steps K --warmup W                    # this repo (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm: the reference path on the host cores

A "step" is one pass of the hot path (MultiAgentEnv.step: action decode -> World.step -> observation /
reward / done, environment.py:80-104) over ONE batch of `n_env` worlds = one fused-kernel launch.
Workload (BASELINE.json configs[1]): simple_spread N=3, 65 536 worlds per GPU.  Under torchrun every
rank steps its own shard (weak scaling, no data-path collective); the only exchange is one all-gather of
the (env_steps, seconds) counters.  Other BASELINE configs: --scenario / --num-envs / --num-agents.

Timing hygiene
  * the timed steps rotate over a ring of R independent batches.  R is sized on the INPUT bytes (state +
    actions, what a step re-reads): R x input bytes > 2 x 126 MB L2, so nothing a step reads can still be
    L2-resident from its previous visit ("inputs larger than L2"); the outputs are write-only;
  * EXACTLY the K requested steps are timed, all of them replayed from CUDA graphs captured before the timed
    region (whole units of R x 25 steps + one graph holding the remainder), whatever K is;
  * a spin kernel queued in front of the start event keeps the stream busy while the host enqueues the event
    records and graph launches, so host launch latency is not inside the region even for K = 20;
  * W >= 3 warm-up steps (+ one untimed replay of every captured graph); CUDA events on the launching
    stream, barrier + synchronize on both sides, max over ranks; nvidia-smi clocks sampled during the region;
  * episodes are reset every 25 steps of each batch (MADDPG's episode length), resets inside the region.

value      device-resident throughput: inputs already in HBM, strictly serialized launches on one stream
e2e        the same metric through the public API `env.step(pinned host tensors)`: H2D of the actions, the
           fused step, D2H of observations / rewards / dones, stream synchronize -- every step
roofline   achieved = algorithmic bytes per launch (SURVEY.md 8(d)) / mean launch time; `traffic` = DRAM bytes
           per launch measured in steady state with ncu (tools/traffic.py, profiles/traffic.json), null if this
           config was not measured; `kernel_ns` = one isolated launch (cold L2) between two events;
           `size_matched_stream` = a pure streaming kernel with the same read / write byte counts in the same harness
cpu_baseline  the reference path on the host cores beside the GPU number (N=1): oracle/np_port.py, the per-world
           NumPy port at the reference's granularity (kind "port"), or the unmodified reference itself when a
           reference install is present under baseline/_ref (kind "reference")

--dump-outputs DIR writes what the last timed step computed, as its caller receives it, to DIR/*.npy.  Inputs are
seeded, so two builds run with the same arguments can be compared output for output.  Run from a tree that
__graft_entry__.build() has built, the benchmark writes nothing into it (it may be read-only); DIR is the only
place it writes to.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the CPU arms run one world per process: keep NumPy / torch thread pools from oversubscribing the host
for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
    os.environ.setdefault(_v, "1")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

EPISODE = 25
L2_BYTES = 126 * 1024 * 1024
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
REF_CHUNK = 100     # reference arm: one bench "step" = REF_CHUNK env.step calls in each process's world
DUMP_MAX_BYTES = 64 * 1024 * 1024   # --dump-outputs: larger outputs are written as a seeded sample of worlds


# ------------------------------------------------------------------------------------------------
# workload description (identical for both arms, computed without touching the CUDA library)
# ------------------------------------------------------------------------------------------------
def scenario_world(scenario, kw):
    from multiagent_particle_envs_b200 import scenarios
    return scenarios.load(scenario + ".py").Scenario(**kw).make_world()


def shapes_from_oracle(desc):
    """(act_dims, obs_dims, algorithmic bytes per env-step, input bytes per env-step) from the descriptor and
    the CPU oracle's shape functions -- the formula of mpe_bytes_per_env_step (csrc/mpe_kernels.cu), restated
    here so that the CPU arm never has to dlopen libmpe_b200.so; tests/test_cpu_host_logic.py keeps them equal."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import Oracle
    o = Oracle(desc, "f64")
    A, L, C = desc.n_agents, desc.n_landmarks, desc.dim_c
    S = sum(0 if desc.agent_silent[i] else 1 for i in range(A))
    G = {4: 1, 5: 1, 6: 1, 7: 2, 8: 2}.get(int(desc.scenario), 0)
    unread = {8: 4 * A + 2 * L, 6: 4}.get(int(desc.scenario), 0)
    mov = sum(4 for i in range(A) if desc.agent_movable[i])
    floats = 4 * A + 2 * L + G + A + S * C - unread + sum(o.act_dims) + sum(o.obs_dims) + mov
    in_floats = 4 * A + 2 * L + G - unread + sum(o.act_dims)
    return list(o.act_dims), list(o.obs_dims), 4 * floats + A, 4 * in_floats


MAX_RING = 256      # tiny batches (< ~8k worlds) would need thousands of ring slots; they are launch-bound anyway
L2_MULTIPLE = 8     # ring inputs >= 8 x L2.  Measured (profiles/traffic.json): with the contract's minimum of 2 x L2 the
#                     126 MB L2 still served ~60 % of the input reads, because the evict-first observation stores leave
#                     the input lines resident and the replacement is not LRU; 8 x L2 + a read-flush before the region


def input_bytes_from_shapes(sh):
    """bytes a step READS per world (state it looks at + goal indices + actions), from a library shape handle"""
    from multiagent_particle_envs_b200 import _lib
    A, L = sh.n_agents, sh.n_landmarks
    unread = {_lib.SCN_CRYPTO: 4 * A + 2 * L, _lib.SCN_SPEAKER_LISTENER: 4}.get(int(sh.desc.scenario), 0)
    return 4 * (4 * A + 2 * L + sh.n_goals - unread + sum(sh.act_dims))


def ring_size(input_bytes_per_env, n_env, requested=0, cap=MAX_RING, l2_multiple=L2_MULTIPLE):
    need = int(l2_multiple * L2_BYTES / (input_bytes_per_env * n_env)) + 1
    return max(3, min(need, cap), requested or 0)


def dump_sample(n_env, bytes_per_world, max_bytes=DUMP_MAX_BYTES):
    """worlds --dump-outputs writes: None (all of them) when they fit max_bytes, else the same seeded sorted sample on
    every run, so that two builds can be compared array for array"""
    if n_env * bytes_per_world <= max_bytes:
        return None
    import numpy as np
    return np.sort(np.random.RandomState(0).choice(n_env, max_bytes // bytes_per_world, replace=False))


def workload_config(scenario, kw, n_env, n_agents, bytes_per_env, input_bytes_per_env, n_gpus, ring):
    headline = (scenario == "simple_spread" and n_env == 65536 and not kw)
    return {"workload": ("simple_spread N=3 agents/landmarks, batch=65536 worlds per GPU (BASELINE configs[1])" if headline
                         else "%s %s, batch=%d worlds per GPU" % (scenario, kw or "", n_env)),
            "scenario": scenario, "scenario_kwargs": kw, "n_env_per_gpu": n_env, "global_n_env": n_env * n_gpus,
            "agents": n_agents, "episode_length": EPISODE, "ring_batches": ring,
            "bytes_per_env_step": bytes_per_env, "input_bytes_per_env_step": input_bytes_per_env,
            "l2_policy": "inputs larger than L2 AND L2 flushed: steps rotate over %d independent batches; their INPUTS alone "
                         "(state + actions, %.1f MB per batch) total %.0f MB %s %d x 126 MB L2 (all bytes %.0f MB), and a "
                         "512 MB read-only sweep evicts the L2 right before every timed region; address translations are "
                         "then re-warmed by touching one word per 32 KB of the ring (a trainer reuses its buffers; cold-TLB "
                         "first touches cost 0.5 us per step at K = 20, profiles/r2d_*)"
                         % (ring, input_bytes_per_env * n_env / 1e6, ring * input_bytes_per_env * n_env / 1e6,
                            ">=" if ring * input_bytes_per_env * n_env >= L2_MULTIPLE * L2_BYTES else "(ring capped) <",
                            L2_MULTIPLE, ring * bytes_per_env * n_env / 1e6),
            "actions": "softmax of N(0,1) logits (+ uniform utterances), pre-generated per batch, resident in HBM",
            "parallelism": "dp%d (independent shards, no data-path collective)" % n_gpus}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_key(scenario, kw, n_env):
    return "%s%s:%d" % (scenario, "".join(",%s=%s" % (k, kw[k]) for k in sorted(kw)), n_env)


def measured_traffic(scenario, kw, n_env):
    """steady-state DRAM bytes per launch of THIS config from profiles/traffic.json (tools/traffic.py + ncu), or None"""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tp)).get("steady_state", {}).get(traffic_key(scenario, kw, n_env))
    except Exception:  # noqa: BLE001
        return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows[-3:]]
        sm = sorted(float(r[1]) for r in rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in rows if len(r) >= 9 for k in range(4) if r[5 + k].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(rows[0][2]) if rows and len(rows[0]) > 2 else None,
                "power_w_max": max([float(r[3]) for r in rows if len(r) > 3 and r[3].replace(".", "").isdigit()] or [0.0]),
                "samples": len(rows), "reasons": reasons}


# ------------------------------------------------------------------------------------------------
# CPU arm (test / baseline infrastructure under oracle/):
#   the unmodified reference   when a reference install exists under baseline/_ref (kind "reference")
#   np_port.py                 per-world NumPy float64 at the reference's own granularity, one world per process --
#                              the stand-in that can travel to the GPU box (kind "port"); next to the real reference in
#                              the build container it is 1.1-1.5x FASTER (profiles/r1_cpu_reference_vs_port.json)
#   mpe_oracle.c               the C checker, ~300x faster than the reference; reported alongside (headline config)
# ------------------------------------------------------------------------------------------------
def reference_install():
    p = os.path.join(ROOT, "baseline", "_ref")
    return p if os.path.isfile(os.path.join(p, "multiagent", "environment.py")) else None


def _ref_worker(args):
    """one process = one world of the UNMODIFIED reference (baseline/_ref), same action distribution as np_port"""
    ref_root, name, n_agents, seed, warmup, steps = args
    import numpy as np
    os.environ["MPE_REFERENCE_ROOT"] = ref_root
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refshim
    np.random.seed(seed)
    env = refshim.make_reference_env(name, n_agents if name == "simple_spread" else None)
    env.reset()
    dims = [int(s.n) if hasattr(s, "n") else int(sum(s.high - s.low + 1)) for s in env.action_space]
    mov = [bool(a.movable) for a in env.world.agents]
    rng = np.random.RandomState(seed)

    def acts():
        out = []
        for d, m in zip(dims, mov):
            parts = []
            if m:
                z = rng.randn(5)
                e = np.exp(z - z.max())
                parts.append(e / e.sum())
            if d - (5 if m else 0) > 0:
                parts.append(rng.uniform(0, 1, d - (5 if m else 0)))
            out.append(np.concatenate(parts))
        return out

    for _ in range(warmup):
        env.step(acts())
    t0 = time.perf_counter()
    for t in range(steps):
        if t % EPISODE == 0:
            env.reset()
        env.step(acts())
    return steps / (time.perf_counter() - t0)


def _cpu_throughput(desc, scenario, kw, procs, warmup, steps, shared_reward):
    """aggregate env-steps/s of `procs` processes x one world each; (total, kind)"""
    ref = reference_install()
    if ref is not None:
        import multiprocessing as mp
        n_agents = kw.get("num_agents")
        with mp.get_context("fork").Pool(procs) as pool:
            rates = pool.map(_ref_worker, [(ref, scenario, n_agents, 100 + p, warmup, steps) for p in range(procs)])
        return float(sum(rates)), "reference"
    import np_port
    total, _ = np_port.timed_throughput(desc, procs, warmup, steps, shared_reward=shared_reward)
    return total, "port"


def _best_process_count(desc, scenario, kw, shared):
    """`os.sched_getaffinity` can exceed what the container may really use (CPU quota, SMT): probe a few process
    counts briefly and keep the one with the highest aggregate throughput -- "all the host threads it can use"."""
    cores = len(os.sched_getaffinity(0))
    cands = sorted({max(1, cores // 8), max(1, cores // 4), max(1, cores // 2), cores})
    best = (0.0, cores)
    for p in cands:
        rate, _ = _cpu_throughput(desc, scenario, kw, p, 20, 300, shared)
        if rate > best[0]:
            best = (rate, p)
    return best[1], best[0]


def cpu_reference_path(desc, scenario, kw, shared, steps, warmup, max_seconds):
    """times the reference path: `steps` env.step calls per process after `warmup` (both may shrink to fit
    max_seconds of wall time, never below 500 / 50)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    procs, probe = _best_process_count(desc, scenario, kw, shared)
    per_proc = max(probe / procs, 1.0)
    steps = int(max(500, min(steps, max_seconds * per_proc)))
    warmup = int(max(50, min(warmup, 0.25 * max_seconds * per_proc)))
    t0 = time.perf_counter()
    total, kind = 0.0, "port"
    for _ in range(2):      # the better of two timed repetitions: gives the CPU arm its best shot, damps box noise
        rate, kind = _cpu_throughput(desc, scenario, kw, procs, warmup, steps, shared)
        total = max(total, rate)
    dt = time.perf_counter() - t0
    cpu_model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                cpu_model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    what = ("the UNMODIFIED reference (baseline/_ref, MultiAgentEnv.step, environment.py:80-104)" if kind == "reference"
            else "oracle/np_port.py (per-world NumPy float64 restatement at the reference's granularity)")
    return {"value": total, "unit": UNIT, "cores": procs, "kind": kind, "cpu_model": cpu_model,
            "sample": "%d processes (best of the probed counts; affinity reports %d CPUs) x %d env.step calls of one %s "
                      "world each after %d warm-up calls (better of two repetitions), through %s; softmax actions, reset every 25 steps; %.1f s wall"
                      % (procs, len(os.sched_getaffinity(0)), steps, scenario, warmup, what, dt),
            "per_process": total / procs, "steps_timed_per_process": steps, "warmup_per_process": warmup, "seconds": dt}


def cpu_c_oracle(desc, budget_s, n_sample=65536):
    """env-steps/s of oracle/mpe_oracle.c (fp64) stepping n_sample simple_spread worlds split over all host threads;
    the step loop runs inside C (ctypes releases the GIL).  Headline config only."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import Oracle
    cores = len(os.sched_getaffinity(0))
    rng = np.random.RandomState(0)
    A, L = 3, 3
    per = (n_sample + cores - 1) // cores
    chunks = []
    for c in range(cores):
        m = min(per, n_sample - c * per)
        if m <= 0:
            break
        pv = np.zeros((m, A, 4))
        pv[:, :, :2] = rng.uniform(-1, 1, (m, A, 2))
        logits = rng.randn(m, A, 5)
        act = np.ascontiguousarray((np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)).reshape(m, 15))
        chunks.append((Oracle(desc, "f64"), pv, rng.uniform(-1, 1, (m, L, 2)), np.zeros((m, A, 2)), act))
    pool = ThreadPoolExecutor(len(chunks))

    def run(steps):
        t0 = time.perf_counter()
        list(pool.map(lambda ch: ch[0].rollout(ch[1], ch[2], ch[3], ch[4], steps, 1), chunks))
        return time.perf_counter() - t0

    run(1)
    one = run(2) / 2
    steps = int(max(2, min(5000, budget_s / max(one, 1e-6))))
    dt = run(steps)
    pool.shutdown()
    return {"value": n_sample * steps / dt, "unit": UNIT, "cores": len(chunks), "kind": "port",
            "sample": "%d steps x %d worlds through oracle/mpe_oracle.c (fp64 C restatement, step loop in C, one thread "
                      "per core); %.1f s" % (steps, n_sample, dt)}


def cpu_baseline_block(desc, scenario, kw, shared, seconds, headline):
    cb = cpu_reference_path(desc, scenario, kw, shared, steps=20000, warmup=100, max_seconds=seconds)
    out = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu_model", "per_process",
                              "steps_timed_per_process")}
    if headline:
        c = cpu_c_oracle(desc, 5.0)
        out["c_oracle"] = {k: c[k] for k in ("value", "unit", "cores", "sample")}
    return out


def run_reference_arm(args, rank, world):
    """The reference's CPU path on this box's host cores, one world per process on every core.  One bench "step"
    of this arm = REF_CHUNK env.step calls in each process's world (a bounded sample of the n_env-world batch):
    `--steps 20 --warmup 5` times 2000 calls per process after 500 warm-up calls.  Loads neither CUDA nor
    libmpe_b200.so: shapes come from the descriptor and the CPU oracle."""
    if rank != 0:
        return
    t_all = time.perf_counter()
    import __graft_entry__ as g
    g.build_oracle(quiet=True)
    w = scenario_world(args.scenario, args.scenario_kw)
    desc = w.descriptor()
    shared = bool(getattr(w, "collaborative", False))
    act_dims, obs_dims, bpe, ibpe = shapes_from_oracle(desc)
    ring = ring_size(ibpe, args.num_envs, args.ring)
    res = cpu_reference_path(desc, args.scenario, args.scenario_kw, shared,
                             steps=max(2000, args.steps * REF_CHUNK), warmup=max(100, args.warmup * REF_CHUNK),
                             max_seconds=90.0)
    cb = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu_model", "per_process",
                              "steps_timed_per_process", "warmup_per_process")}
    headline = args.scenario == "simple_spread" and not args.scenario_kw
    if headline:
        c = cpu_c_oracle(desc, 5.0)
        cb["c_oracle"] = {k: c[k] for k in ("value", "unit", "cores", "sample")}
    cores = res["cores"]
    per_step_calls = res["steps_timed_per_process"] / float(args.steps)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "steps_timed_per_process": res["steps_timed_per_process"],
            "ms_per_step": 1e3 * per_step_calls * cores / res["value"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.scenario, args.scenario_kw, args.num_envs, desc.n_agents, bpe, ibpe, args.gpus, ring),
            "cpu_baseline": cb, "agent_steps_per_sec": desc.n_agents * res["value"],
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_all,
            "native_so_in_process": sorted({ln.split()[-1][len(ROOT) + 1:] for ln in open("/proc/self/maps")
                                            if ln.rstrip().endswith(".so") and ROOT in ln}),
            "note": "reference arm = the reference's CPU path on the host cores (%s): %d processes, one world each, %d "
                    "env.step calls per process = %d bench steps of %.0f calls; it does not scale with --gpus"
                    % ("the unmodified reference from baseline/_ref" if res["kind"] == "reference" else
                       "oracle/np_port.py, the per-world NumPy port -- the Python reference itself cannot travel to the GPU box",
                       cores, res["steps_timed_per_process"], args.steps, per_step_calls)}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def pin_to_gpu_numa(local_rank):
    """Bind this rank to the CPUs of its GPU's NUMA node BEFORE CUDA starts and before any pinned slab is allocated
    (first touch puts the staging buffers on that node; torch.distributed.run does not bind).  Returns the original
    affinity (restored for the CPU baseline) and a description."""
    orig = os.sched_getaffinity(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=20).stdout
        bus = None
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local_rank]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else local_rank
        for ln in out.splitlines():
            idx, b = [x.strip() for x in ln.split(",")]
            if int(idx) == phys:
                bus = b.lower()
        if bus is None:
            return orig, "no pci bus id"
        if len(bus.split(":")[0]) == 8:       # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return orig, "single NUMA node"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= orig
        if not cpus:
            return orig, "NUMA node %d has no allowed CPU" % node
        os.sched_setaffinity(0, cpus)
        return orig, "NUMA node %d (%d CPUs)" % (node, len(cpus))
    except Exception as e:  # noqa: BLE001
        return orig, "not pinned (%s)" % type(e).__name__


class Ring(object):
    """R independent env batches with resident actions and outputs + the CUDA-graph plans that step them"""

    def __init__(self, scenario, kw, n_env, dev, rank, world, requested_ring=0, max_ring=MAX_RING):
        import torch
        from multiagent_particle_envs_b200 import _lib, make_env
        self.torch, self.dev, self.n_env = torch, dev, n_env
        probe = make_env(scenario, **kw)
        sh = probe.world.native_shapes()
        self.n_agents = probe.n
        self.bytes_per_env = sh.bytes_per_env_step
        mov = [bool(a.movable) for a in probe.agents]
        self.input_bytes_per_env = input_bytes_from_shapes(sh)
        self.R = ring_size(self.input_bytes_per_env, n_env, requested_ring, max_ring)
        self.bytes_per_step = self.bytes_per_env * n_env
        self.slots = []
        for b in range(self.R):
            env = make_env(scenario, num_envs=n_env * world, device=dev, seed=1000 + b, rank=rank, world_size=world, **kw)
            env.reset()
            nw = env.world.native
            g = torch.Generator(device=dev).manual_seed(7 * b + rank)
            acts = []
            for d_act, m in zip(nw.act_dims, mov):     # 5 movement probabilities, then the utterance
                parts = []
                if m:
                    parts.append(torch.softmax(torch.randn(n_env, 5, device=dev, generator=g), 1))
                if d_act - (5 if m else 0) > 0:
                    parts.append(torch.rand(n_env, d_act - (5 if m else 0), device=dev, generator=g))
                acts.append(torch.cat(parts, 1).contiguous())
            self.slots.append((env, nw, acts, _lib.ptr_array([t.data_ptr() for t in acts]), env._flags()))
        self.unit = self.R * EPISODE
        self.stream = torch.cuda.Stream(dev)
        self.side = torch.cuda.Stream(dev)
        self.launches = 0
        self._graphs = {}
        self._flush = torch.zeros(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
        with torch.cuda.stream(self.stream):
            for i in range(self.R):      # first launches outside capture (module load, lazy init)
                self.step_slot(i)
            self.stream.synchronize()
        self.launches = 0

    def step_slot(self, i):
        env, nw, acts, ptrs, flags = self.slots[i % self.R]
        nw.step(ptrs, nw.out, flags)
        self.launches += 1

    def reset_all(self):
        for env, nw, acts, ptrs, flags in self.slots:
            nw.reset()
            self.launches += 1

    def flush_l2(self):
        """read-only sweep over 512 MB: the L2 ends up full of CLEAN lines of a buffer nobody touches again (a write
        sweep would leave 126 MB of dirty lines whose write-back competes with the timed steps)"""
        self._flush.sum()

    def warm_tlb(self):
        """touch one 4-byte word per 32 KB of every ring tensor (state, actions, outputs): address translations are
        resident as they are for a trainer that reuses its buffers every step, while the L2 stays cold (the touches
        bring in one 32-byte sector per 32 KB, ~0.1 % of the data).  MPE_BENCH_TLB_WARM=0 disables it."""
        if os.environ.get("MPE_BENCH_TLB_WARM", "1") == "0":
            return
        torch = self.torch
        acc = None
        for env, nw, acts, ptrs, flags in self.slots:
            for t in [nw.agent_pv, nw.lm_p, nw.comm, nw.out.slab] + list(acts):
                v = t.view(-1)
                if v.dtype != torch.float32:
                    v = v.view(torch.uint8)[: v.numel() // 4 * 4].view(torch.float32) if v.dtype == torch.uint8 else v.float()
                part = v[:: 8192].sum()
                acc = part if acc is None else acc + part
        self._tlb_sink = acc

    def _capture(self, first, count, two_streams, lead=0):
        """one CUDA graph stepping slots first .. first+count-1 (mod R), strictly in order on one stream, or with
        even / odd positions on two streams (fork / join) for the two-batches-in-flight extra.  The graph records an
        external timing event before its first and after its last kernel, so a region that consists of ONE graph
        launch is timed inside the graph: the device-side cost of the graph launch itself (tens of microseconds,
        dominant when K = 20) is not part of the K steps."""
        key = (first % self.R, count, two_streams, lead)
        if key in self._graphs:
            return self._graphs[key]
        torch = self.torch
        before = self.launches
        graph = torch.cuda.CUDAGraph()
        try:
            graph.ev = (torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
        except TypeError:       # older torch: no external events, fall back to events around the launch
            graph.ev = None
        with torch.cuda.graph(graph, stream=self.stream):
            for k in range(lead):            # untimed lead-in steps on the slots just before `first` (see plan())
                self.step_slot(first - lead + k)
            if graph.ev:
                graph.ev[0].record(self.stream)
            if two_streams:
                self.side.wait_stream(self.stream)
            for k in range(count):
                if two_streams and k % 2:
                    with torch.cuda.stream(self.side):
                        self.step_slot(first + k)
                else:
                    self.step_slot(first + k)
            if two_streams:
                self.stream.wait_stream(self.side)
            if graph.ev:
                graph.ev[1].record(self.stream)
        self.launches = before      # capture is not execution
        graph.last_slot = (first + count - 1) % self.R
        self._graphs[key] = graph
        return graph

    def plan(self, k, two_streams=False, lead=0):
        """graphs covering exactly k steps: whole units (R x 25 steps, then the episode resets) + one remainder.
        When the k steps fit ONE graph, `lead` untimed warm-up steps on other ring slots are captured in front of the
        graph's start event: the start-up cost of a graph launch (first kernels of a freshly launched graph run
        several microseconds late -- 0.7 us per step when K = 20) is spent before the timed K steps begin."""
        units, rem = divmod(k, self.unit)
        if units == 0 and rem + lead <= self.R:
            return (None, 0, self._capture(lead, rem, two_streams, lead), rem)
        return (self._capture(0, self.unit, two_streams) if units else None, units,
                self._capture(0, rem, two_streams) if rem else None, rem)

    def run(self, plan):
        unit_graph, units, rem_graph, rem = plan
        for _ in range(units):
            unit_graph.replay()
            self.launches += self.unit
            self.reset_all()
        if rem:
            rem_graph.replay()
            self.launches += rem

    def last_outputs(self, plan):
        """host float32 copies of what the last step of `plan` handed its caller: obs_<i> [n, obs_dim_i], rew_<i> [n],
        done_<i> [n] per agent, restricted to dump_sample's worlds"""
        unit_graph, units, rem_graph, rem = plan
        env, nw, acts, ptrs, flags = self.slots[(rem_graph if rem else unit_graph).last_slot]
        A = nw.n_agents
        arrays = {"obs_%d" % i: o for i, o in enumerate(nw.out.obs)}
        arrays.update(("rew_%d" % i, nw.out.rew[i]) for i in range(A))
        arrays.update(("done_%d" % i, nw.out.done[i]) for i in range(A))
        rows = dump_sample(self.n_env, 4 * (sum(nw.obs_dims) + 2 * A))
        if rows is not None:
            rows = self.torch.as_tensor(rows, device=self.dev)
        return {k: (t if rows is None else t.index_select(0, rows)).float().cpu().numpy() for k, t in arrays.items()}

    def timed(self, plan, spin_cycles):
        """seconds of device time for one run of `plan`, measured between two events on the launching stream; a spin
        kernel ahead of the start event absorbs the host's enqueue latency"""
        torch = self.torch
        unit_graph, units, rem_graph, rem = plan
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.stream):
            self.flush_l2()
            self.warm_tlb()
            torch.cuda._sleep(spin_cycles)
            e0.record(self.stream)
            self.run(plan)
            e1.record(self.stream)
            self.stream.synchronize()
        self.timed_by = "events around the graph launches"
        if units == 0 and rem and getattr(rem_graph, "ev", None):      # one graph launch: use the events inside it
            self.timed_by = ("external events recorded inside the single graph, after its lead-in steps "
                             "(start of timed step 1 .. end of timed step K)")
            return rem_graph.ev[0].elapsed_time(rem_graph.ev[1]) / 1e3
        return e0.elapsed_time(e1) / 1e3

    def isolated_kernel_ns(self, spin_cycles, repeats=9):
        """one fused-step launch between two events, L2 flushed by a 256 MB fill before each: median / min in ns"""
        torch = self.torch
        out = []
        with torch.cuda.stream(self.stream):
            for r in range(repeats):
                self.flush_l2()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda._sleep(spin_cycles)
                e0.record(self.stream)
                self.step_slot(r)
                e1.record(self.stream)
                self.stream.synchronize()
                out.append(e0.elapsed_time(e1) * 1e6)
        self.launches -= repeats
        out.sort()
        return {"median": out[len(out) // 2], "min": out[0], "repeats": repeats,
                "note": "event pair around ONE launch on an idle GPU with a flushed L2 (includes launch + drain)"}

    def size_matched_stream(self, lib, k, spin_cycles):
        """the same harness around a pure streaming kernel with this config's read / write byte counts per launch"""
        torch = self.torch
        rd = (self.input_bytes_per_env * self.n_env + 15) // 16 * 16
        wr = ((self.bytes_per_env - self.input_bytes_per_env) * self.n_env + 15) // 16 * 16
        src = torch.zeros(self.R * rd // 4, dtype=torch.float32, device=self.dev)
        dst = torch.empty(self.R * wr // 4, dtype=torch.float32, device=self.dev)
        threads = max(256, self.n_env)
        import ctypes

        def probe(i):
            rc = lib.mpe_probe_stream(self.dev.index, ctypes.c_void_p(src.data_ptr() + (i % self.R) * rd), rd,
                                      ctypes.c_void_p(dst.data_ptr() + (i % self.R) * wr), wr, threads,
                                      ctypes.c_void_p(self.stream.cuda_stream))
            if rc:
                raise RuntimeError("mpe_probe_stream failed: %d" % rc)

        k = max(1, min(k, self.unit))
        best = None
        with torch.cuda.stream(self.stream):
            for threads in (self.n_env, 2 * self.n_env, 4 * self.n_env, 8 * self.n_env):
                threads = max(256, threads)
                for i in range(min(self.R, 4)):
                    probe(i)
                self.stream.synchronize()
                graph = torch.cuda.CUDAGraph()
                ev = (torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
                with torch.cuda.graph(graph, stream=self.stream):
                    for i in range(5):               # lead-in, as for the timed steps
                        probe(i)
                    ev[0].record(self.stream)
                    for i in range(5, 5 + k):
                        probe(i)
                    ev[1].record(self.stream)
                graph.replay()
                self.stream.synchronize()
                self.flush_l2()
                if os.environ.get("MPE_BENCH_TLB_WARM", "1") != "0":      # same treatment as the ring (warm_tlb)
                    self._tlb_sink = src[::8192].sum() + dst[::8192].sum()
                torch.cuda._sleep(spin_cycles)
                graph.replay()
                self.stream.synchronize()
                sec = ev[0].elapsed_time(ev[1]) / 1e3 / k
                if best is None or sec < best[0]:
                    best = (sec, threads)
        sec, threads = best
        # the operation MEASURED_PEAKS.json's HBM peak was measured with (torch: b.copy_(a), read + write bytes), at THIS
        # launch's byte count instead of 2 GB: half of the step's bytes read, half written, ring-rotated, same timing
        half = (rd + wr) // 2 // 16 * 16
        csrc = torch.zeros(min(self.R, 64) * half // 4, dtype=torch.float32, device=self.dev)
        cdst = torch.empty_like(csrc)
        nslot = min(self.R, 64)
        with torch.cuda.stream(self.stream):
            graph = torch.cuda.CUDAGraph()
            ev = (torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
            w4 = half // 4
            for i in range(2):
                cdst[i * w4:(i + 1) * w4].copy_(csrc[i * w4:(i + 1) * w4])
            self.stream.synchronize()
            with torch.cuda.graph(graph, stream=self.stream):
                for i in range(min(5, k)):
                    cdst[(i % nslot) * w4:((i % nslot) + 1) * w4].copy_(csrc[(i % nslot) * w4:((i % nslot) + 1) * w4])
                ev[0].record(self.stream)
                for i in range(5, 5 + k):
                    cdst[(i % nslot) * w4:((i % nslot) + 1) * w4].copy_(csrc[(i % nslot) * w4:((i % nslot) + 1) * w4])
                ev[1].record(self.stream)
            graph.replay()
            self.stream.synchronize()
            self.flush_l2()
            if os.environ.get("MPE_BENCH_TLB_WARM", "1") != "0":
                self._tlb_sink = csrc[::8192].sum() + cdst[::8192].sum()
            torch.cuda._sleep(spin_cycles)
            graph.replay()
            self.stream.synchronize()
        copy_sec = ev[0].elapsed_time(ev[1]) / 1e3 / k
        self.copy_probe = {"ms_per_launch": 1e3 * copy_sec, "gbs": 2 * half / copy_sec / 1e9, "bytes_read_plus_written": 2 * half,
                           "launches": k,
                           "note": "torch b.copy_(a) -- the operation the HBM peak in MEASURED_PEAKS.json was measured with -- "
                                   "moving this config's bytes per launch (half read, half written) instead of 2 GB, same "
                                   "graph replay / ring rotation / L2 flush"}
        return {"ms_per_launch": 1e3 * sec, "gbs": (rd + wr) / sec / 1e9, "launches": k, "read_bytes": rd, "write_bytes": wr,
                "threads": threads,
                "note": "pure streaming kernel (float4 loads, then dependent evict-first float4 stores) with this config's "
                        "read / write byte counts per launch, best of 1 / 2 / 4 / 8 threads per world, same launch path / graph "
                        "replay / ring rotation / L2 flush: what this batch size lets ANY strictly serialized launch reach"}


def run_b200_arm(args, rank, local_rank, world):
    orig_affinity, numa = pin_to_gpu_numa(local_rank)
    import torch
    import torch.distributed as dist
    from multiagent_particle_envs_b200 import _lib
    from multiagent_particle_envs_b200.sharding import aggregate_counters

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints a "NCCL version ..." banner on stdout when its communicator is created; rank 0 must print
        # exactly ONE line on stdout, so file descriptor 1 points at stderr while the communicator comes up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    lib = _lib.load()
    N_ENV = args.num_envs
    ring = Ring(args.scenario, args.scenario_kw, N_ENV, dev, rank, world, args.ring)
    R = ring.R
    K, W = args.steps, max(args.warmup, 3)
    sm_hz = getattr(torch.cuda.get_device_properties(dev), "clock_rate", 1.9e6) * 1e3      # kHz -> Hz
    spin = int(200e-6 * sm_hz)      # ~200 us of spinning in front of every timed region

    # ---- value: exactly K strictly serialized steps, replayed from graphs captured beforehand ------------------
    plan = ring.plan(K, lead=W)
    warm_plan = ring.plan(W)
    with torch.cuda.stream(ring.stream):
        ring.run(warm_plan)                       # the W warm-up steps
        ring.run(plan if plan[1] == 0 else ring.plan(ring.unit + K % ring.unit))   # + one untimed replay of every timed graph
        ring.stream.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank).start()
    time.sleep(0.12)
    ring.launches = 0
    t0 = time.time()
    seconds = ring.timed(plan, spin)
    timed_by = ring.timed_by
    t1 = time.time()
    gpu_launches = ring.launches
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop(t0, t1)
    total_steps, max_seconds, per_rank = aggregate_counters(N_ENV * K, seconds)
    value = total_steps / max_seconds
    # copied now: the extras below step the same ring slots again
    dumped = ring.last_outputs(plan) if args.dump_outputs and rank == 0 else None

    # ---- extras on the same K steps: two batches in flight; isolated launch; size-matched streaming kernel ----
    plan2 = ring.plan(K, two_streams=True, lead=W)
    with torch.cuda.stream(ring.stream):
        ring.run(plan2 if plan2[1] == 0 else ring.plan(ring.unit + K % ring.unit, two_streams=True))
        ring.stream.synchronize()
    seconds2 = ring.timed(plan2, spin)
    total2, max2, _ = aggregate_counters(N_ENV * K, seconds2)
    kernel_ns = ring.isolated_kernel_ns(spin) if rank == 0 else None
    probe = ring.size_matched_stream(lib, K, spin) if rank == 0 else None
    if world > 1:
        dist.barrier()

    # ---- end to end through the public API with host buffers --------------------------------------------------
    env = ring.slots[0][0]
    k_e2e = max(3, min(K, args.e2e_steps))
    host_acts = [[a.cpu().pin_memory() for a in ring.slots[b % R][2]] for b in range(4)]
    h2d = sum(a.numel() * 4 for a in host_acts[0])

    def e2e_run(e, reuse):
        e.reuse_buffers = reuse
        for b in range(3):
            obs_n, rew_n, done_n, _ = e.step(host_acts[b % 4])
        nbytes = sum(o.numel() * 4 for o in obs_n) + sum(r.numel() * 4 for r in rew_n) + sum(d.numel() for d in done_n)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        chk = 0.0
        w0 = time.perf_counter()
        for b in range(k_e2e):
            obs_n, rew_n, done_n, _ = e.step(host_acts[b % 4])   # H2D + fused step + D2H + sync inside
            chk += float(rew_n[0][0])                            # the caller reads the result on the host
        torch.cuda.synchronize()
        sec = time.perf_counter() - w0
        tot, mx, _ = aggregate_counters(N_ENV * k_e2e, sec)
        return tot / mx, mx, nbytes, chk

    e2e_value, e2e_max, d2h, checksum = e2e_run(env, True)
    # the fresh-array semantics copy 15 MB per step on the host: give torch's CPU copy the threads a user process would
    # have (this script pins OMP to 1 thread for the one-world-per-process CPU arm)
    host_threads = max(1, min(16, len(os.sched_getaffinity(0)) // max(world, 1)))
    torch.set_num_threads(host_threads)
    fresh_value, fresh_max, _, _ = e2e_run(env, False)
    torch.set_num_threads(1)
    env.reuse_buffers = True

    # extra (not the headline): two env batches in flight through step_async / step_wait, so that the upload +
    # step of one overlaps the download of the other -- what a double-buffered host trainer would see
    env_b = ring.slots[1][0]
    env_b.reuse_buffers = True
    lanes = {id(env): torch.cuda.Stream(dev), id(env_b): torch.cuda.Stream(dev)}   # one stream per env batch

    def launch(e, acts):
        with torch.cuda.stream(lanes[id(e)]):
            e.step_async(acts)

    for b in range(2):
        launch(env, host_acts[b % 4]); launch(env_b, host_acts[(b + 1) % 4]); env.step_wait(); env_b.step_wait()
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    launch(env, host_acts[0])
    for b in range(k_e2e):
        cur, nxt = (env, env_b) if b % 2 == 0 else (env_b, env)
        if b + 1 < k_e2e:
            launch(nxt, host_acts[(b + 1) % 4])
        obs_n, rew_n, done_n, _ = cur.step_wait()
        checksum += float(rew_n[0][0])
    torch.cuda.synchronize()
    pipe_seconds = time.perf_counter() - w0
    pipe_total, pipe_max, _ = aggregate_counters(N_ENV * k_e2e, pipe_seconds)

    if rank == 0:
        peak, peak_src = measured_peak()
        launch_s = max_seconds / K
        achieved = ring.bytes_per_step / launch_s / 1e9
        traffic = measured_traffic(args.scenario, args.scenario_kw, N_ENV)
        headline = args.scenario == "simple_spread" and not args.scenario_kw
        cpu = None
        if world == 1 and args.cpu_seconds > 0:
            os.sched_setaffinity(0, orig_affinity)      # the CPU arm uses every host core
            w = scenario_world(args.scenario, args.scenario_kw)
            cpu = cpu_baseline_block(w.descriptor(), args.scenario, args.scenario_kw,
                                     bool(getattr(w, "collaborative", False)), args.cpu_seconds, headline)
        probe["frac"] = probe["gbs"] / peak
        copy_probe = getattr(ring, "copy_probe", None)
        if copy_probe:
            copy_probe["frac"] = copy_probe["gbs"] / peak
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * launch_s, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "timing": timed_by,
            "config": workload_config(args.scenario, args.scenario_kw, N_ENV, ring.n_agents, ring.bytes_per_env,
                                      ring.input_bytes_per_env, world, R),
            "agent_steps_per_sec": ring.n_agents * value,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": k_e2e, "ms_per_step": 1e3 * e2e_max / k_e2e,
                    "api": "MultiAgentEnv.step(pinned host tensors) with env.reuse_buffers = True: results are views of "
                           "the two flip-flopped pinned result slabs (valid until the next-but-one step)",
                    "cpu_affinity": numa},
            "e2e_fresh_arrays": {"value": fresh_value, "unit": UNIT, "ms_per_step": 1e3 * fresh_max / k_e2e,
                                 "host_copy_threads": host_threads,
                                 "api": "the same call with the default env.reuse_buffers = False: every step hands out "
                                        "freshly allocated host copies (the reference's ownership semantics)"},
            "value_two_batches_in_flight": {"value": total2 / max2, "unit": UNIT, "steps": K, "ms_per_step": 1e3 * max2 / K,
                                            "frac": ring.bytes_per_step / (max2 / K) / 1e9 / peak,
                                            "note": "extra: the same K steps with alternate ring slots on two streams "
                                                    "(fork/join CUDA graph); each batch still advances strictly in order"},
            "e2e_two_batches_in_flight": {"value": pipe_total / pipe_max, "unit": UNIT, "ms_per_step": 1e3 * pipe_max / k_e2e,
                                          "api": "step_async / step_wait alternating over two env batches"},
            "gpu_launches": gpu_launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "traffic_source": ("profiles/traffic.json (ncu --cache-control none, steady state over the ring, "
                                            "tools/traffic.py)" if traffic is not None else "not measured for this config"),
                         "frac_of_measured_traffic": (traffic / launch_s / 1e9 / peak) if traffic else None,
                         "algorithmic_bytes_per_launch": ring.bytes_per_step,
                         "kernel_ns": kernel_ns, "size_matched_stream": probe, "size_matched_copy": copy_probe,
                         "kernel": "mpe_kernel<%s program, kFusedStep>" % args.scenario},
            "per_rank": per_rank,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if dumped is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60000)
    ap.add_argument("--warmup", type=int, default=3000)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ring", type=int, default=0, help="ring batches (default: sized so that the inputs exceed 2x L2)")
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--scenario", default="simple_spread", help="other BASELINE configs: simple_tag, simple_world_comm, ...")
    ap.add_argument("--num-envs", type=int, default=65536, help="worlds per GPU")
    ap.add_argument("--num-agents", type=int, default=None, help="simple_spread only (N agents = N landmarks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (obs_<i> / rew_<i> / done_<i> "
                         "per agent, float32) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.scenario_kw = {"num_agents": args.num_agents} if args.num_agents is not None else {}
    return args


def main():
    sys.dont_write_bytecode = True      # no __pycache__ in the source tree, which may be read-only
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)     # no CUDA, no libmpe_b200.so in this process
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29400 + os.getpid() % 500), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    import __graft_entry__ as g
    g.build(quiet=True)
    run_b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
