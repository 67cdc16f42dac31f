"""NativeWorld: the batch state tensors of one World plus the libmpe_b200 handle that steps them.

PyTorch owns every buffer (device memory, pinned host memory, streams); the library borrows raw
pointers per call (include/mpe_b200.h).  Nothing in this module computes: it allocates, packs
pointers and launches.  A missing extension or a machine without a CUDA device raises.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import check


def _align(x, a=256):
    return (x + a - 1) // a * a


class ShapeHandle(object):
    """Device-less handle (mpe_create(..., device=-1)): validates the descriptor against its
    compiled program and answers the shape queries MultiAgentEnv.__init__ needs
    (environment.py:39-70).  Works on machines without a GPU."""

    def __init__(self, desc, n_env, device_index=-1):
        self.lib = _lib.load()
        self.desc = desc
        self.n_env = int(n_env)
        h = ctypes.c_void_p()
        check(self.lib.mpe_create(ctypes.byref(desc), self.n_env, device_index, ctypes.byref(h)), "mpe_create")
        self.handle = h
        lib = self.lib
        self.n_agents = lib.mpe_num_agents(h)
        self.n_landmarks = int(desc.n_landmarks)
        self.dim_c = int(desc.dim_c)
        self.custom = int(desc.scenario) == _lib.SCN_CUSTOM     # observation / reward live in the user's torch code
        self.obs_dims = [] if self.custom else [lib.mpe_obs_dim(h, i) for i in range(self.n_agents)]
        self.act_dims = [lib.mpe_act_dim(h, i) for i in range(self.n_agents)]
        self.n_speakers = lib.mpe_num_speakers(h)
        self.n_goals = lib.mpe_num_goals(h)
        self.info_dim = lib.mpe_info_dim(h)
        self.bytes_per_env_step = lib.mpe_bytes_per_env_step(h)
        self._speakers = [i for i in range(self.n_agents) if not desc.agent_silent[i]]

    def collect_supported(self, depth, hidden):
        """mpe_collect_supported: 0 if mpe_collect is built for this scenario at (depth, hidden), else
        _lib.ERR_UNSUPPORTED (ERR_BAD_ARG for a depth or width the kernel never takes)"""
        return self.lib.mpe_collect_supported(self.handle, int(depth), int(hidden))

    def speaker_slot(self, agent_index):
        """row block of agent `agent_index` in the comm tensors, or -1 if the agent is silent"""
        try:
            return self._speakers.index(agent_index)
        except ValueError:
            return -1

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.mpe_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001  (interpreter shutdown)
            pass


class Outputs(object):
    """One slab holding everything a step produces, so that a host caller gets it with a single
    DMA: obs_0 | obs_1 | ... | rew [A][N] | done [A][N] | info [A][INFO][N] (256-byte aligned parts;
    mpe_step_host coalesces the adjacent parts into one cudaMemcpyAsync)."""

    def __init__(self, nw, pinned_host=False):
        import torch
        N, A = nw.n_env, nw.n_agents
        offs, off = [], 0
        for od in nw.obs_dims:
            offs.append(off)
            off = _align(off + N * od * 4)
        rew_off = off
        off = _align(off + A * N * 4)
        done_off = off
        off = _align(off + A * N)
        info_off = off
        off = _align(off + A * nw.info_dim * N * 4)
        if pinned_host:
            self.slab = torch.empty(off, dtype=torch.uint8, pin_memory=True)
        else:
            self.slab = torch.empty(off, dtype=torch.uint8, device=nw.device)
        s = self.slab
        self.obs = [s[o:o + N * od * 4].view(torch.float32).view(N, od) for o, od in zip(offs, nw.obs_dims)]
        self.rew = s[rew_off:rew_off + A * N * 4].view(torch.float32).view(A, N)
        self.info = None
        if nw.info_dim > 0:
            self.info = s[info_off:info_off + A * nw.info_dim * N * 4].view(torch.float32).view(A, nw.info_dim, N)
        self.done = s[done_off:done_off + A * N].view(A, N)
        # per-agent views handed to the caller (built once: persistent outputs are reused every step)
        self.rew_list = [self.rew[i] for i in range(A)]
        done_b = self.done.view(torch.bool)
        self.done_list = [done_b[i] for i in range(A)]
        if pinned_host:   # NumPy views of the same pinned memory (scalar convention: no per-step tensor ops)
            self.obs_np = [o.numpy() for o in self.obs]
            self.rew_np, self.done_np = self.rew.numpy(), self.done.numpy()
            self.info_np = self.info.numpy() if self.info is not None else None
        self.obs_ptrs = _lib.ptr_array([t.data_ptr() for t in self.obs])
        self.rew_ptr = self.rew.data_ptr()
        self.done_ptr = self.done.data_ptr()
        self.info_ptr = self.info.data_ptr() if self.info is not None else None


class FreshOutputs(object):
    """Per-step device outputs for callers that keep what `step` returns (the reference hands out freshly
    allocated arrays).  Same attributes as `Outputs`, built with as few tensor operations as possible -- one
    float slab carved with as_strided, `unbind` for the per-agent views -- because at ~6 us per kernel the
    host-side cost of a step is what a GPU-resident trainer actually waits for."""

    def __init__(self, nw):
        import torch
        N, A = nw.n_env, nw.n_agents
        lay = nw._fresh_layout
        fs = torch.empty(lay["words"], dtype=torch.float32, device=nw.device)
        self.slab = fs
        self.obs = [fs.as_strided((N, od), (od, 1), off) for off, od in lay["obs"]]
        self.rew = fs.as_strided((A, N), (N, 1), lay["rew"])
        self.rew_list = self.rew.unbind(0)
        self.info = fs.as_strided((A, nw.info_dim, N), (nw.info_dim * N, N, 1), lay["info"]) if nw.info_dim > 0 else None
        done_b = torch.empty((A, N), dtype=torch.bool, device=nw.device)   # written as 0/1 bytes by the kernel
        self.done = done_b.view(torch.uint8)
        self.done_list = done_b.unbind(0)
        base = fs.data_ptr()
        self.obs_ptrs = _lib.ptr_array([base + 4 * off for off, _ in lay["obs"]])
        self.rew_ptr = base + 4 * lay["rew"]
        self.done_ptr = done_b.data_ptr()
        self.info_ptr = base + 4 * lay["info"] if nw.info_dim > 0 else None


class NativeWorld(ShapeHandle):
    def __init__(self, desc, n_env, device=None, seed=0, world_offset=0):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("multiagent_particle_envs_b200 needs a CUDA device (B200, sm_100a); "
                               "there is no CPU fallback")
        self.torch = torch
        dev = torch.device(device if device is not None else "cuda")
        if dev.type != "cuda":
            raise RuntimeError("device must be a CUDA device, got %s" % (dev,))
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        super(NativeWorld, self).__init__(desc, n_env, dev.index)
        N, A, L = self.n_env, self.n_agents, self.n_landmarks
        NC = self.n_speakers * self.dim_c
        f32 = dict(dtype=torch.float32, device=dev)
        # ---- state, struct-of-arrays over worlds (include/mpe_b200.h) ----
        self.agent_pv = torch.zeros(A, N, 4, **f32)
        self.lm_p = torch.zeros(max(L, 1), N, 2, **f32)
        self.comm = torch.zeros(max(NC, 1), N, **f32)
        self.goal = torch.zeros(max(self.n_goals, 1), N, dtype=torch.int32, device=dev)
        # ---- decoded actions for World.step() ----
        self.act_u = torch.zeros(A, N, 2, **f32)
        self.act_c = torch.zeros(max(NC, 1), N, **f32)
        self.seed = int(seed)
        self.world_offset = int(world_offset)
        self.epoch = 0
        self._epoch_dev = None
        # layout of FreshOutputs' float slab, in 4-byte words (every part 64-word = 256-byte aligned)
        off, obs_l = 0, []
        for od in self.obs_dims:
            obs_l.append((off, od))
            off = _align(off + N * od, 64)
        rew_off = off
        off = _align(off + A * N, 64)
        info_off = off
        off = _align(off + A * self.info_dim * N, 64)
        self._fresh_layout = dict(obs=obs_l, rew=rew_off, info=info_off, words=max(off, 64))
        self.out = None if self.custom else Outputs(self)   # persistent outputs (reset / step in reuse mode)
        self.cb_out = None                 # lazily created: outputs of direct scenario-callback calls (core.py)
        self._host = None                  # lazily created staging for host callers
        self._has_comm = NC > 0
        self._has_goal = self.n_goals > 0

    # ---- helpers ---------------------------------------------------------------------------
    def _stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _state_ptrs(self):
        return (self.agent_pv.data_ptr(), self.lm_p.data_ptr(),
                self.comm.data_ptr() if self._has_comm else None,
                self.goal.data_ptr() if self._has_goal else None)

    def new_outputs(self):
        return FreshOutputs(self)

    def persistent_outputs(self):
        return Outputs(self)

    # ---- reset -------------------------------------------------------------------------------
    def reset(self, mask=None):
        torch = self.torch
        mptr = None
        if mask is not None:
            mask = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if mask.numel() != self.n_env:
                raise ValueError("reset mask must have one entry per world")
            mptr = mask.data_ptr()
        pv, lm, comm, goal = self._state_ptrs()
        if self.torch.cuda.is_current_stream_capturing():
            # inside a CUDA-graph capture the epoch must live on the device, or every replay would redraw the
            # same initial conditions
            if self._epoch_dev is None:
                raise RuntimeError("call NativeWorld.enable_device_epoch() before capturing a reset in a CUDA graph")
            check(self.lib.mpe_reset_dev_epoch(self.handle, pv, lm, comm, goal, mptr, self.seed, self.world_offset,
                                               self._epoch_dev.data_ptr(), self._stream()), "mpe_reset_dev_epoch")
            return
        if self._epoch_dev is not None:
            self.epoch = int(self._epoch_dev.item())
        check(self.lib.mpe_reset(self.handle, pv, lm, comm, goal, mptr, self.seed, self.world_offset,
                                 self.epoch, self._stream()), "mpe_reset")
        self.epoch += 1
        if self._epoch_dev is not None:
            self._epoch_dev.fill_(self.epoch)

    def enable_device_epoch(self):
        """keep the reset epoch in device memory so that resets captured in CUDA graphs advance it on replay"""
        if self._epoch_dev is None:
            self._epoch_dev = self.torch.full((1,), self.epoch, dtype=self.torch.int64, device=self.device)
        return self._epoch_dev

    # ---- the hot path ------------------------------------------------------------------------
    def set_action(self, act_ptrs, flags=0):
        check(self.lib.mpe_set_action(self.handle, act_ptrs, self.act_u.data_ptr(),
                                      self.act_c.data_ptr() if self._has_comm else None,
                                      flags & ~_lib.FLAG_SHARED_REWARD, self._stream()), "mpe_set_action")

    def world_step(self):
        pv, lm, comm, _ = self._state_ptrs()
        check(self.lib.mpe_world_step(self.handle, pv, lm, comm, self.act_u.data_ptr(),
                                      self.act_c.data_ptr() if self._has_comm else None, self._stream()),
              "mpe_world_step")

    def observe(self, out=None, flags=0, with_info=True):
        out = out or self.out
        pv, lm, comm, goal = self._state_ptrs()
        check(self.lib.mpe_observe(self.handle, pv, lm, comm, goal, out.obs_ptrs, out.rew_ptr, out.done_ptr,
                                   out.info_ptr if with_info else None, flags, self._stream()), "mpe_observe")
        return out

    def step(self, act_ptrs, out=None, flags=0, with_info=False):
        """MultiAgentEnv.step fused into one launch; act_ptrs: ctypes array of device pointers.
        benchmark_data (info) is computed and written only when asked for (make_env(benchmark=True))."""
        out = out or self.out
        pv, lm, comm, goal = self._state_ptrs()
        check(self.lib.mpe_step(self.handle, pv, lm, comm, goal, act_ptrs, out.obs_ptrs, out.rew_ptr,
                                out.done_ptr, out.info_ptr if with_info else None, flags, self._stream()),
              "mpe_step")
        return out

    def rollout(self, act_seq_ptrs, n_steps, out=None, flags=0, rew_steps=None):
        """n_steps fused steps on pre-generated actions in ONE launch (mpe_rollout): the state stays in registers
        between the steps.  out.obs / out.done describe the final state, out.rew holds the summed rewards;
        rew_steps: optional float32 [n_steps, A, N] CUDA tensor receiving every step's rewards."""
        out = out or self.out
        pv, lm, comm, goal = self._state_ptrs()
        check(self.lib.mpe_rollout(self.handle, pv, lm, comm, goal, act_seq_ptrs, int(n_steps), out.obs_ptrs, out.rew_ptr,
                                   rew_steps.data_ptr() if rew_steps is not None else None, out.done_ptr, flags,
                                   self._stream()), "mpe_rollout")
        return out

    def rollout_policy(self, w1_ptrs, b1_ptrs, w2_ptrs, b2_ptrs, hidden, n_steps, out=None, flags=0, rew_steps=None,
                       act_rec_ptrs=None):
        """n_steps fused steps in ONE launch with every agent's two-layer perceptron evaluated inside the kernel
        (mpe_rollout_policy); pointer arrays hold one device pointer per agent."""
        out = out or self.out
        pv, lm, comm, goal = self._state_ptrs()
        check(self.lib.mpe_rollout_policy(self.handle, pv, lm, comm, goal, w1_ptrs, b1_ptrs, w2_ptrs, b2_ptrs, int(hidden),
                                          int(n_steps), out.obs_ptrs, out.rew_ptr,
                                          rew_steps.data_ptr() if rew_steps is not None else None, act_rec_ptrs,
                                          out.done_ptr, flags, self._stream()), "mpe_rollout_policy")
        return out

    def collect(self, depth, hidden, weight_ptrs, n_steps, out=None, flags=0, sample_seed=0, sample_step=0, rew_steps=None,
                act_rec_ptrs=None, obs_rec_ptrs=None):
        """n_steps closed-loop steps in ONE launch with one- or two-hidden-layer actors inside the kernel (mpe_collect).
        weight_ptrs: the pointer arrays (w1, b1, w2, b2, w3, b3), one device pointer per agent (w3, b3 None at depth 1).
        The exploration noise is keyed by this shard's global world indices (world_offset), so a sharded batch draws
        what the whole batch draws."""
        out = out or self.out
        pv, lm, comm, goal = self._state_ptrs()
        check(self.lib.mpe_collect(self.handle, pv, lm, comm, goal, int(depth), int(hidden), *weight_ptrs, int(n_steps),
                                   int(sample_seed), int(sample_step), self.world_offset, out.obs_ptrs, out.rew_ptr,
                                   rew_steps.data_ptr() if rew_steps is not None else None, act_rec_ptrs, obs_rec_ptrs,
                                   out.done_ptr, flags, self._stream()), "mpe_collect")
        return out

    # ---- host callers (what the reference's callers hold: NumPy arrays) -----------------------
    def host_staging(self):
        if self._host is None:
            torch = self.torch
            N = self.n_env
            host_act = [torch.zeros(N, ad, dtype=torch.float32).pin_memory() for ad in self.act_dims]
            dev_act = [torch.zeros(N, ad, dtype=torch.float32, device=self.device) for ad in self.act_dims]
            self._host = dict(
                host_act=host_act, dev_act=dev_act, host_act_np=[t.numpy() for t in host_act],
                host_act_ptrs=_lib.ptr_array([t.data_ptr() for t in host_act]),
                dev_act_ptrs=_lib.ptr_array([t.data_ptr() for t in dev_act]),
                host_out=[Outputs(self, pinned_host=True), Outputs(self, pinned_host=True)], flip=0)
        return self._host

    def step_host(self, host_act_ptrs, flags=0, dev_out=None, host_out=None, with_info=False):
        """H2D actions -> fused step -> D2H outputs, all enqueued on the current stream by
        mpe_step_host; returns the pinned host Outputs (valid after a stream synchronize)."""
        hs = self.host_staging()
        dev_out = dev_out or self.out
        if host_out is None:
            host_out = hs["host_out"][hs["flip"]]
            hs["flip"] ^= 1
        pv, lm, comm, goal = self._state_ptrs()
        check(self.lib.mpe_step_host(self.handle, pv, lm, comm, goal, host_act_ptrs, hs["dev_act_ptrs"],
                                     dev_out.obs_ptrs, dev_out.rew_ptr, dev_out.done_ptr,
                                     dev_out.info_ptr if with_info else None,
                                     host_out.obs_ptrs, host_out.rew_ptr, host_out.done_ptr,
                                     host_out.info_ptr if with_info else None,
                                     flags | _lib.FLAG_HOST_SLAB, self._stream()), "mpe_step_host")
        return host_out

    # ---- benchmark_data (e.g. simple_spread.py:47-63) -----------------------------------------
    def benchmark_data(self, i, batched, out=None):
        """scenario.benchmark_data(agent i) from the info channel, in the reference's return shape"""
        out = out or self.out
        sc = self.desc.scenario
        if out.info is None:
            return {}
        info = out.info[i]                     # [info_dim, N]
        adv = bool(self.desc.agent_adversary[i])
        L, C = self.n_landmarks, self.dim_c
        if batched:
            if sc == _lib.SCN_SPREAD:           # (rew, collisions, min_dists, occupied_landmarks)
                return (info[0], info[1], info[2], info[3])
            if sc == _lib.SCN_ADVERSARY:        # adversary: |p - goal|^2; good: (|p - lm_l|^2 ..., |p - goal|^2)
                return info[0] if adv else tuple(info[q] for q in range(L + 1))
            if sc == _lib.SCN_CRYPTO:           # (agent.state.c, goal colour)
                return (info[0:C].t(), info[C:2 * C].t())
            return info[0]
        v = (out.info_np[i, :, 0] if getattr(out, "info_np", None) is not None
             else info[:, 0].detach().to("cpu").numpy()).astype(np.float64)
        if sc == _lib.SCN_SPREAD:
            return (float(v[0]), int(v[1]), float(v[2]), int(v[3]))
        if sc == _lib.SCN_ADVERSARY:
            return float(v[0]) if adv else tuple(float(x) for x in v[:L + 1])
        if sc == _lib.SCN_CRYPTO:
            return (v[0:C].copy(), v[C:2 * C].copy())
        return int(v[0])
