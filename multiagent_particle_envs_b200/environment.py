"""MultiAgentEnv: the gym-style adapter over a (batched) World
(reference: multiagent/environment.py:12-263).

Same constructor, attributes and `step` / `reset` contract as the reference.  The per-agent
Python loops of the reference's `step` (`_set_action` -> `world.step()` -> observation / reward /
done / info callbacks -> shared-reward sum, environment.py:80-104) are ONE launch of the fused
sm_100a kernel (`mpe_step`) over all worlds of the batch.

Calling conventions
  scalar mode  (world.num_envs is None; what `make_env(name)` gives): identical to the reference --
      `action_n[i]` is a 1-D array, `obs_n[i]` a float64 ndarray, `reward_n[i]` a float,
      `done_n[i]` a bool, `info_n == {'n': [...]}`.
  batched mode (world.num_envs = N): `action_n[i]` is `[N, act_dim_i]`; CUDA tensors in ->
      CUDA tensors out (`obs_n[i]: [N, obs_dim_i]`, `reward_n[i]: [N]`, `done_n[i]: [N] bool`);
      NumPy arrays / CPU tensors in -> the step runs through pinned staging (`mpe_step_host`) and
      NumPy arrays / CPU tensors come back.
"""
import numpy as np

from . import _lib
from .multi_discrete import MultiDiscrete
from .scenario import NativeScenario
from . import spaces

try:  # pragma: no cover
    from gym import Env as _Env
except Exception:  # noqa: BLE001
    class _Env(object):
        pass


class MultiAgentEnv(_Env):
    metadata = {'render.modes': ['human', 'rgb_array']}

    def __init__(self, world, reset_callback=None, reward_callback=None,
                 observation_callback=None, info_callback=None,
                 done_callback=None, shared_viewer=True):
        self.world = world
        self.agents = self.world.policy_agents
        self.n = len(world.policy_agents)
        self.reset_callback = reset_callback
        self.reward_callback = reward_callback
        self.observation_callback = observation_callback
        self.info_callback = info_callback
        self.done_callback = done_callback
        # environment parameters (environment.py:28-36)
        self.discrete_action_space = True
        self.discrete_action_input = False
        self.force_discrete_action = world.discrete_action if hasattr(world, 'discrete_action') else False
        self.shared_reward = world.collaborative if hasattr(world, 'collaborative') else False
        self.time = 0
        #: batched mode: hand out views of the library's persistent result buffers instead of freshly allocated
        #: tensors / arrays.  CUDA callers: every step writes the same device slab (results are overwritten by the
        #: next step).  Host callers: results are views of two flip-flopped pinned slabs (valid until the
        #: next-but-one step).  Default False = the reference's ownership: every step returns fresh arrays.
        self.reuse_buffers = False

        self._custom = (getattr(world, "native_program", None) == "custom")
        if self._custom and not world.batched:
            raise NotImplementedError("user scenarios (TorchScenario) run in batched mode only: pass num_envs")
        for name, cb in (("reward_callback", reward_callback), ("observation_callback", observation_callback)):
            owner = getattr(cb, "__self__", None)
            if cb is not None and not self._custom and not isinstance(owner, NativeScenario):
                raise NotImplementedError(
                    "%s is an arbitrary Python callable; only scenarios with a compiled sm_100a program "
                    "(subclasses of NativeScenario) can be stepped, and there is no CPU fallback" % name)
        self._native_info = info_callback is not None and isinstance(getattr(info_callback, "__self__", None),
                                                                     NativeScenario)
        shapes = world.native_shapes()   # validates the descriptor; works without a GPU
        if shapes.n_agents != self.n:
            raise ValueError("native program agent count mismatch")

        # configure spaces (environment.py:39-70)
        self.action_space = []
        self.observation_space = []
        for i, agent in enumerate(self.agents):
            total_action_space = []
            if agent.movable:
                total_action_space.append(spaces.Discrete(world.dim_p * 2 + 1))
            if not agent.silent:
                total_action_space.append(spaces.Discrete(world.dim_c))
            if len(total_action_space) > 1:
                self.action_space.append(MultiDiscrete([[0, sp.n - 1] for sp in total_action_space]))
            else:
                self.action_space.append(total_action_space[0])
            if self._custom:   # as the reference does (environment.py:68): ask the callback (binds the batch: needs the GPU)
                world.bind()
                obs_dim = int(observation_callback(agent, world).shape[-1])
            else:
                obs_dim = shapes.obs_dims[i]
            self.observation_space.append(spaces.Box(low=-np.inf, high=+np.inf, shape=(obs_dim,), dtype=np.float32))
        self._act_dims = list(shapes.act_dims)
        self._sub_sizes = [([5] if a.movable else []) + ([world.dim_c] if not a.silent else []) for a in self.agents]

        # rendering (headless; attributes kept for API compatibility)
        self.shared_viewer = shared_viewer
        self.viewers = [None] if shared_viewer else [None] * self.n
        self._reset_render()

    # ------------------------------------------------------------------------------------------
    def _flags(self):
        f = 0
        if self.shared_reward:
            f |= _lib.FLAG_SHARED_REWARD
        if self.force_discrete_action:
            f |= _lib.FLAG_FORCE_DISCRETE_ACTION
        if not self.discrete_action_space:
            raise NotImplementedError("discrete_action_space=False is not supported (hard-coded True in the "
                                      "reference, environment.py:29)")
        return f

    def _index_tensors(self, action_n, nw):
        """discrete_action_input (environment.py:161-167,185-187): the kernel decodes integer sub-actions itself
        (MPE_FLAG_DISCRETE_ACTION_INPUT): action_n[i] becomes int32 [N, n_sub_i] on the device -- a no-op for a
        contiguous int32 CUDA tensor of that shape; other dtypes / host arrays are converted / uploaded here.
        Movement index 0 = none, 1 = -x, 2 = +x, 3 = -y, 4 = +y; utterance index k -> one-hot(k)."""
        import torch
        N = self.world.batch_size
        out = []
        for i, a in enumerate(action_n):
            nsub = len(self._sub_sizes[i])
            if not torch.is_tensor(a):
                a = torch.as_tensor(np.ascontiguousarray(np.asarray(a)).astype(np.int32, copy=False))
            if a.numel() != N * nsub:
                raise ValueError("action_n[%d] must hold %d x %d integer sub-actions, got shape %s"
                                 % (i, N, nsub, tuple(a.shape)))
            if a.device != nw.device or a.dtype != torch.int32:
                a = a.to(device=nw.device, dtype=torch.int32)
            out.append(a.reshape(N, nsub).contiguous())
        return out

    def _step_discrete(self, action_n, nw, flags):
        world = self.world
        on_device = all(hasattr(a, "is_cuda") and a.is_cuda for a in action_n)
        as_numpy = not any(hasattr(a, "dim") for a in action_n)
        idx = self._index_tensors(action_n, nw)
        flags |= _lib.FLAG_DISCRETE_ACTION_INPUT
        if self._custom:
            return self._step_custom(idx, nw, flags)
        out = nw.out if (self.reuse_buffers or not world.batched) else nw.new_outputs()
        nw.step(_lib.ptr_array([t.data_ptr() for t in idx]), out, flags, with_info=self._native_info)
        self._last_out = out
        world._obs_valid = False
        if not world.batched:
            return self._pack_scalar(nw, out)
        obs_n, reward_n, done_n, info_n = self._pack_batched(nw, out)
        if not on_device:     # host callers get host results back
            obs_n, reward_n, done_n = ([t.cpu() for t in x] for x in (obs_n, reward_n, done_n))
            if as_numpy:
                obs_n, reward_n, done_n = ([t.numpy() for t in x] for x in (obs_n, reward_n, done_n))
        return obs_n, reward_n, done_n, info_n

    def step(self, action_n):
        world = self.world
        nw = world.bind()
        self.agents = world.policy_agents
        if len(action_n) != self.n:
            raise ValueError("expected %d actions, got %d" % (self.n, len(action_n)))
        flags = self._flags()
        if self.discrete_action_input:
            return self._step_discrete(action_n, nw, flags)
        if self._custom:
            return self._step_custom(action_n, nw, flags)
        if not world.batched and not any(hasattr(a, "dim") for a in action_n):
            # scalar convention fast path: NumPy in, NumPy out, no tensor objects created per step
            hs = nw.host_staging()
            for i, a in enumerate(action_n):
                np.copyto(hs["host_act_np"][i][0], np.asarray(a, dtype=np.float32).reshape(-1))
            hout = nw.step_host(hs["host_act_ptrs"], flags, with_info=self._native_info)
            nw.torch.cuda.current_stream(nw.device).synchronize()
            self._last_out = hout
            world._obs_valid = False
            return self._pack_scalar(nw, hout)
        mode, payload = self._classify(action_n, nw)
        if mode == "cuda":
            out = nw.out if self.reuse_buffers else nw.new_outputs()
            nw.step(_lib.ptr_array([t.data_ptr() for t in payload]), out, flags, with_info=self._native_info)
            self._last_out = out
            world._obs_valid = False
            if not world.batched:     # scalar convention with device-side inputs (e.g. discrete_action_input)
                return self._pack_scalar(nw, out)
            return self._pack_batched(nw, out)
        # host callers: pinned staging -> mpe_step_host -> pinned outputs
        hs = nw.host_staging()
        ptrs = []
        for i, a in enumerate(payload):
            if mode == "pinned":
                ptrs.append(a.data_ptr())
            else:
                hs["host_act"][i].copy_(a if hasattr(a, "dim") else self._to_cpu_tensor(a, i))
                ptrs.append(hs["host_act"][i].data_ptr())
        hout = nw.step_host(_lib.ptr_array(ptrs), flags, with_info=self._native_info)
        nw.torch.cuda.current_stream(nw.device).synchronize()
        self._last_out = hout
        world._obs_valid = False
        if not world.batched:
            return self._pack_scalar(nw, hout)
        as_numpy = not hasattr(action_n[0], "dim")
        return self._pack_batched(nw, hout, as_numpy=as_numpy)

    # ---- K-step open-loop rollout (batch extension; SURVEY.md 8(f) rank 3) -------------------------
    def rollout(self, action_seq_n, per_step_rewards=False):
        """T consecutive `step` calls on pre-generated actions in ONE kernel launch (mpe_rollout): the loop of
        bin/interactive.py:27-39 when the actions are known in advance (recorded trajectories, CEM / MPPI candidate
        sequences).  action_seq_n[i]: float32 CUDA tensor [T, N, act_dim_i].  Returns (obs_n, reward_sum_n, done_n,
        info_n) for the state after the last step -- reward_sum_n[i] is the sum over the T steps, bit-equal to calling
        `step` T times and adding the rewards in order -- plus, with per_step_rewards=True, a fifth item: the [T, n, N]
        tensor of every step's rewards.  Batched CUDA mode only."""
        import torch
        world = self.world
        if not world.batched:
            raise ValueError("rollout needs a batched env (make_env(..., num_envs=N))")
        if self._custom:
            raise NotImplementedError("rollout is not available for user scenarios (TorchScenario)")
        if self.discrete_action_input:
            raise NotImplementedError("rollout takes action vectors, not integer actions")
        if len(action_seq_n) != self.n:
            raise ValueError("expected %d action sequences, got %d" % (self.n, len(action_seq_n)))
        nw = world.bind()
        N = nw.n_env
        T = int(action_seq_n[0].shape[0])
        seqs = []
        for i, a in enumerate(action_seq_n):
            if not (torch.is_tensor(a) and a.is_cuda and a.device == nw.device):
                raise ValueError("action_seq_n[%d] must be a CUDA tensor on %s" % (i, nw.device))
            if tuple(a.shape) != (T, N, self._act_dims[i]):
                raise ValueError("action_seq_n[%d] must have shape (%d, %d, %d), got %s"
                                 % (i, T, N, self._act_dims[i], tuple(a.shape)))
            if a.dtype != torch.float32 or not a.is_contiguous():
                a = a.to(torch.float32).contiguous()
            seqs.append(a)
        out = nw.out if self.reuse_buffers else nw.new_outputs()
        rew_steps = torch.empty((T, self.n, N), dtype=torch.float32, device=nw.device) if per_step_rewards else None
        nw.rollout(_lib.ptr_array([t.data_ptr() for t in seqs]), T, out, self._flags(), rew_steps)
        self._last_out = out
        world._obs_valid = False
        obs_n, reward_n, done_n = list(out.obs), list(out.rew_list), list(out.done_list)
        info_n = {'n': [{} for _ in range(self.n)]}
        if per_step_rewards:
            return obs_n, reward_n, done_n, info_n, rew_steps
        return obs_n, reward_n, done_n, info_n

    def rollout_policy(self, policies, n_steps, record_actions=False, per_step_rewards=False, record_observations=False,
                       explore_seed=None, explore_step=0):
        """T closed-loop steps in ONE kernel launch with the actors inside the kernel (mpe_collect).  policies[i] is agent
        i's actor with A_i = act_dim_i = action_space[i]'s width outputs, H = 32 or 64, the same depth and H for every
        agent:
          one hidden layer   logits_i = W2_i relu(W1_i obs_i + b1_i) + b2_i: a `torch.nn.Sequential(Linear(obs_dim_i,
              H), ReLU(), Linear(H, A_i))` or the tuple (W1 [H, obs_dim_i], b1 [H], W2 [A_i, H], b2 [A_i]);
          two hidden layers (the MADDPG actor) logits_i = W3_i relu(W2_i relu(W1_i obs_i + b1_i) + b2_i) + b3_i: a
              `torch.nn.Sequential(Linear(obs_dim_i, H), ReLU(), Linear(H, H), ReLU(), Linear(H, A_i))` or the tuple
              (W1, b1, W2 [H, H], b2 [H], W3 [A_i, H], b3 [A_i]);
        all in torch's Linear layout.  The logits are the heads of the agent's action space, as MADDPG splits them: 5
        movement logits if the agent moves, then dim_c communication logits if it speaks; each head gets its own
        softmax, and the comm head's probabilities are what the agent says.  explore_seed=None acts with
        softmax(logits); an int acts with MADDPG's exploration sample softmax(logits - log(-log u)) per head, u uniform in
        (0, 1) drawn from a Philox stream keyed by (explore_seed, global world index, explore_step + t, agent, logit): a
        sharded env draws what the full batch draws, and a rollout split into calls with explore_step = 0, T1, T1 + T2,
        ... draws what one call does.
        Returns (obs_n, reward_sum_n, done_n, info_n, extras) for the state after the last step; extras["actions"]
        (record_actions) is a list of [T, N, A_i] tensors with the actions taken, extras["rewards"] (per_step_rewards) a
        [T, n, N] tensor, extras["observations"] (record_observations) a list of [T, N, obs_dim_i] tensors whose row t is
        the observation agent i acted on at step t -- with the final obs_n, the (obs, act, rew, next obs) of every step.
        World state lives in registers for all T steps.  Batched CUDA mode; scenarios whose program was built with the
        policy kernel (simple, simple_spread N=3, simple_tag 3+1, simple_adversary 1+2, simple_push,
        simple_speaker_listener, simple_reference, simple_crypto) -- anything else raises MpeError."""
        import torch
        world = self.world
        if not world.batched:
            raise ValueError("rollout_policy needs a batched env (make_env(..., num_envs=N))")
        if self._custom or self.discrete_action_input or self.force_discrete_action:
            raise NotImplementedError("rollout_policy: compiled scenarios with plain action vectors only")
        if len(policies) != self.n:
            raise ValueError("expected %d policies, got %d" % (self.n, len(policies)))
        nw = world.bind()
        N, T = nw.n_env, int(n_steps)
        flags = self._flags()
        if explore_seed is not None:
            explore_seed, explore_step = int(explore_seed), int(explore_step)
            if not 0 <= explore_seed < 2 ** 64:
                raise ValueError("explore_seed must be in [0, 2**64), got %d" % explore_seed)
            if explore_step < 0 or explore_step + T >= 2 ** 32:
                raise ValueError("explore_step + n_steps must stay below 2**32 (the step counter of the noise stream)")
            flags |= _lib.FLAG_SAMPLE_ACTIONS
        # a scenario without the kernel is refused before the actors are looked at: their shapes mean nothing there
        if all(nw.collect_supported(d, h) != 0 for d in (1, 2) for h in (32, 64)):
            _lib.check(_lib.ERR_UNSUPPORTED, "rollout_policy (mpe_collect_supported)")
        depth, hidden, params = actor_parameters(policies, nw.obs_dims, nw.act_dims)
        keep = []
        for W in params:
            W = [t.detach().to(device=nw.device, dtype=torch.float32) for t in W]
            W[0] = W[0].t()                      # W1 input-major for the kernel
            keep.append([t.contiguous() for t in W])
        ptrs = [_lib.ptr_array([W[k].data_ptr() for W in keep]) if k < len(keep[0]) else None for k in range(6)]
        out = nw.out if self.reuse_buffers else nw.new_outputs()
        rew_steps = torch.empty((T, self.n, N), dtype=torch.float32, device=nw.device) if per_step_rewards else None
        actions = [torch.empty((T, N, ad), dtype=torch.float32, device=nw.device)
                   for ad in nw.act_dims] if record_actions else None
        observations = [torch.empty((T, N, od), dtype=torch.float32, device=nw.device)
                        for od in nw.obs_dims] if record_observations else None
        nw.collect(depth, hidden, ptrs, T, out, flags, explore_seed or 0, explore_step if explore_seed is not None else 0,
                   rew_steps, _lib.ptr_array([a.data_ptr() for a in actions]) if actions is not None else None,
                   _lib.ptr_array([o.data_ptr() for o in observations]) if observations is not None else None)
        self._last_out = out
        world._obs_valid = False
        info_n = {'n': [{} for _ in range(self.n)]}
        return list(out.obs), list(out.rew_list), list(out.done_list), info_n, \
            {"actions": actions, "rewards": rew_steps, "observations": observations}

    # ---- user scenarios: native _set_action + World.step, callbacks in the user's torch code -------
    def _step_custom(self, action_n, nw, flags):
        import torch
        world = self.world
        acts = []
        for i, a in enumerate(action_n):
            if flags & _lib.FLAG_DISCRETE_ACTION_INPUT:      # already int32 [N, n_sub] on the device (_index_tensors)
                acts.append(a)
                continue
            t = a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, dtype=np.float32))
            t = t.to(device=nw.device, dtype=torch.float32).reshape(nw.n_env, self._act_dims[i]).contiguous()
            acts.append(t)
        nw.set_action(_lib.ptr_array([t.data_ptr() for t in acts]), flags)      # environment.py:87-88
        world.step()                                                            # :90
        obs_n = [self._get_obs(agent) for agent in self.agents]                 # :92-97
        reward_n = [torch.as_tensor(self._get_reward(agent), device=nw.device, dtype=torch.float32).expand(nw.n_env)
                    for agent in self.agents]
        if self.done_callback is None:
            done_n = [torch.zeros(nw.n_env, dtype=torch.bool, device=nw.device) for _ in self.agents]
        else:
            done_n = [self.done_callback(agent, world) for agent in self.agents]
        info_n = {'n': [self._get_info(agent) for agent in self.agents]}
        if self.shared_reward:                                                  # :100-102
            total = torch.stack(reward_n).sum(0)
            reward_n = [total] * self.n
        return obs_n, reward_n, done_n, info_n

    # ---- asynchronous stepping for host callers (batch extension) ------------------------------
    def step_async(self, action_n):
        """Enqueue H2D(actions) -> fused step -> D2H(outputs) on the current CUDA stream and return
        immediately; the caller overlaps its own host work (or another env's step) with the transfers and
        collects the results with `step_wait()`.  Host inputs only (NumPy / CPU tensors), batched mode."""
        world = self.world
        if not world.batched:
            raise ValueError("step_async needs a batched env (make_env(..., num_envs=N))")
        if getattr(self, "_pending", None) is not None:
            raise RuntimeError("step_async called twice without step_wait")
        if self._custom:
            raise NotImplementedError("step_async is not available for user scenarios (TorchScenario): their "
                                      "observation / reward callbacks run as torch ops after the native step")
        if self.discrete_action_input:
            raise NotImplementedError("step_async takes action vectors; integer actions go through step()")
        if len(action_n) != self.n:
            raise ValueError("expected %d actions, got %d" % (self.n, len(action_n)))
        nw = world.bind()
        self.agents = world.policy_agents
        mode, payload = self._classify(action_n, nw)
        if mode == "cuda":
            raise ValueError("step_async is for host buffers; CUDA-tensor steps are already asynchronous")
        hs = nw.host_staging()
        ptrs = []
        for i, a in enumerate(payload):
            if mode == "pinned":
                ptrs.append(a.data_ptr())
            else:
                hs["host_act"][i].copy_(a)
                ptrs.append(hs["host_act"][i].data_ptr())
        hout = nw.step_host(_lib.ptr_array(ptrs), self._flags(), with_info=self._native_info)
        ev = nw.torch.cuda.Event()
        ev.record(nw.torch.cuda.current_stream(nw.device))
        self._pending = (hout, ev, payload, not hasattr(action_n[0], "dim"))
        world._obs_valid = False

    def step_wait(self):
        """Block until the step enqueued by `step_async` has landed in host memory; returns what `step` returns."""
        if getattr(self, "_pending", None) is None:
            raise RuntimeError("step_wait without step_async")
        hout, ev, _keepalive, as_numpy = self._pending
        self._pending = None
        ev.synchronize()
        self._last_out = hout
        return self._pack_batched(self.world.bind(), hout, as_numpy=as_numpy)

    # ---- input classification ---------------------------------------------------------------
    def _to_cpu_tensor(self, a, i):
        import torch
        t = torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float32)))
        return t.reshape(self.world.batch_size, self._act_dims[i])

    def _classify(self, action_n, nw):
        import torch
        N = self.world.batch_size
        if all(torch.is_tensor(a) and a.is_cuda for a in action_n):
            payload = []
            for i, a in enumerate(action_n):
                if a.device != nw.device:
                    raise ValueError("action_n[%d] lives on %s but this env's worlds live on %s" % (i, a.device, nw.device))
                if a.shape != (N, self._act_dims[i]):
                    raise ValueError("action_n[%d] must have shape (%d, %d), got %s" %
                                     (i, N, self._act_dims[i], tuple(a.shape)))
                if a.dtype != torch.float32 or not a.is_contiguous() or a.data_ptr() % 16:
                    a = a.to(torch.float32).contiguous().clone()
                payload.append(a)
            return "cuda", payload
        payload = []
        pinned = True
        for i, a in enumerate(action_n):
            if torch.is_tensor(a):
                a = a.detach()
                if a.is_cuda:
                    a = a.cpu()
                a = a.reshape(N, -1)
                ok = a.dtype == torch.float32 and a.is_contiguous() and a.is_pinned()
                if not ok:
                    a = a.to(torch.float32).contiguous()
                pinned = pinned and ok
            else:
                a = self._to_cpu_tensor(a, i)
                pinned = False
            if a.shape != (N, self._act_dims[i]):
                raise ValueError("action_n[%d] must have %d x %d elements, got shape %s" %
                                 (i, N, self._act_dims[i], tuple(a.shape)))
            payload.append(a)
        return ("pinned" if pinned else "host"), payload

    # ---- output packing -----------------------------------------------------------------------
    def _info_list(self, nw, out, batched):
        if self.info_callback is None:
            return [{} for _ in range(self.n)]
        if self._native_info:
            return [nw.benchmark_data(i, batched, out) for i in range(self.n)]
        return [self.info_callback(agent, self.world) for agent in self.agents]

    def _pack_batched(self, nw, out, as_numpy=False):
        obs_n = list(out.obs)
        reward_n = list(out.rew_list)
        done_n = list(out.done_list)
        if self.done_callback is not None:
            done_n = [self.done_callback(agent, self.world) for agent in self.agents]
        info_n = {'n': self._info_list(nw, out, True)}
        if out.slab.device.type == "cpu" and not self.reuse_buffers:
            # pinned staging slabs are reused every other step: the caller gets its own copies (the reference
            # returns freshly allocated arrays, and trainers keep them in replay buffers by reference)
            own = lambda t: t.clone() if hasattr(t, "clone") else t
            obs_n, reward_n, done_n = [own(o) for o in obs_n], [own(r) for r in reward_n], [own(d) for d in done_n]
            info_n = {'n': [tuple(own(x) for x in e) if isinstance(e, tuple) else own(e) for e in info_n['n']]}
        if as_numpy:
            obs_n = [o.numpy() for o in obs_n]
            reward_n = [r.numpy() for r in reward_n]
            done_n = [d.numpy() if hasattr(d, "numpy") else d for d in done_n]
        return obs_n, reward_n, done_n, info_n

    def _pack_scalar(self, nw, hout):
        if getattr(hout, "obs_np", None) is not None:       # pinned host outputs: plain NumPy views
            obs_n = [o[0].astype(np.float64) for o in hout.obs_np]
            rew = hout.rew_np[:, 0].astype(np.float64)
            done_n = [bool(d) for d in hout.done_np[:, 0]]
        else:
            obs_n = [o[0].detach().to("cpu").numpy().astype(np.float64) for o in hout.obs]
            rew = hout.rew[:, 0].detach().to("cpu").numpy().astype(np.float64)
            done_n = [bool(d) for d in hout.done[:, 0].detach().to("cpu")]
        reward_n = [rew[i] for i in range(self.n)]
        if self.done_callback is not None:
            done_n = [self.done_callback(agent, self.world) for agent in self.agents]
        info_n = {'n': self._info_list(nw, hout, False)}
        return obs_n, reward_n, done_n, info_n

    # ------------------------------------------------------------------------------------------
    def reset(self, mask=None, seed=None):
        """environment.py:106-116.  `mask` ([N] bool) resets a subset of the worlds (batched
        extension); observations are returned for every world."""
        world = self.world
        nw = world.bind()
        if mask is None and seed is None:
            self.reset_callback(world)
        else:
            self.reset_callback(world, mask=mask, seed=seed)
        self._reset_render()
        self.agents = world.policy_agents
        if self._custom:
            return [self._get_obs(agent) for agent in self.agents]
        out = nw.out if (self.reuse_buffers or not world.batched) else nw.new_outputs()
        nw.observe(out, 0, with_info=False)
        world._obs_valid = False
        if world.batched:
            return list(out.obs)
        return [o[0].detach().to("cpu").numpy().astype(np.float64) for o in out.obs]

    # ---- per-agent accessors kept for API compatibility (environment.py:119-141) --------------
    def _get_info(self, agent):
        if self.info_callback is None:
            return {}
        return self.info_callback(agent, self.world)

    def _get_obs(self, agent):
        if self.observation_callback is None:
            return np.zeros(0)
        return self.observation_callback(agent, self.world)

    def _get_done(self, agent):
        if self.done_callback is None:
            return False
        return self.done_callback(agent, self.world)

    def _get_reward(self, agent):
        if self.reward_callback is None:
            return 0.0
        return self.reward_callback(agent, self.world)

    def _set_action(self, action, agent, action_space, time=None):
        """environment.py:144-192 for ONE agent: decodes into agent.action.u / .c via the native
        set_action kernel (all agents are decoded; the other agents' inputs are zero)."""
        import torch
        nw = self.world.bind()
        idx = self.world._agent_index(agent)
        acts = [torch.zeros(nw.n_env, ad, device=nw.device) for ad in self._act_dims]
        acts[idx] = torch.as_tensor(np.asarray(action, dtype=np.float32) if not torch.is_tensor(action) else action,
                                    dtype=torch.float32, device=nw.device).reshape(nw.n_env, -1).contiguous()
        keep_u, keep_c = nw.act_u.clone(), nw.act_c.clone()
        nw.set_action(_lib.ptr_array([t.data_ptr() for t in acts]), self._flags())
        s = nw.speaker_slot(idx)
        new_u = nw.act_u[idx].clone()
        new_c = nw.act_c[s * nw.dim_c:(s + 1) * nw.dim_c].clone() if s >= 0 else None
        nw.act_u.copy_(keep_u)
        nw.act_c.copy_(keep_c)
        nw.act_u[idx] = new_u
        if new_c is not None:
            nw.act_c[s * nw.dim_c:(s + 1) * nw.dim_c] = new_c

    # ---- rendering: a headless rasteriser stands in for the pyglet viewer (SURVEY.md 8(f) rank 4) ---
    def _reset_render(self):
        self.render_geoms = None
        self.render_geoms_xform = None

    def render(self, mode='human', world_index=0):
        """environment.py:200-263 without a window: returns one uint8 [700, 700, 3] image per viewer
        (one shared viewer, or one per agent when shared_viewer=False) of world `world_index`;
        mode 'human' additionally prints the communication line the reference prints (:201-213)."""
        from .raster import draw_world
        world = self.world
        nw = world.bind()
        pv = nw.agent_pv[:, world_index].detach().to("cpu").numpy().astype(np.float64)
        lm = nw.lm_p[:, world_index].detach().to("cpu").numpy().astype(np.float64)[:len(world.landmarks)]
        if mode == 'human':
            alphabet = 'ABCDEFGHIJKLMNOPQRSTUVWXYZ'
            message = ''
            for agent in world.agents:
                for i, other in enumerate(world.agents):
                    if other is agent:
                        continue
                    s = nw.speaker_slot(i)
                    c = np.zeros(0) if s < 0 else nw.comm[s * nw.dim_c:(s + 1) * nw.dim_c, world_index].detach().to("cpu").numpy()
                    word = '_' if (c.size == 0 or np.all(c == 0)) else alphabet[int(np.argmax(c))]
                    message += (other.name + ' to ' + agent.name + ': ' + word + '   ')
            print(message)
        ents = world.entities
        pos = np.concatenate([pv[:, 0:2], lm], axis=0) if len(lm) else pv[:, 0:2]
        sizes = [e.size for e in ents]
        colors = [e.color for e in ents]
        alphas = [0.5 if 'agent' in e.name else 1.0 for e in ents]
        results = []
        for i in range(len(self.viewers)):
            center = (0.0, 0.0) if self.shared_viewer else tuple(pv[i, 0:2])
            results.append(draw_world(pos, sizes, colors, alphas, center=center))
        return results


def actor_parameters(policies, obs_dims, act_dims=None):
    """(depth, H, [per-agent weight tuples in torch's Linear layout]) of the actors MultiAgentEnv.rollout_policy runs:
    depth 1 -- a module holding exactly two Linear layers (Linear -> ReLU -> Linear) or (W1, b1, W2, b2); depth 2 -- a
    `Sequential(Linear, ReLU, Linear, ReLU, Linear)` or (W1, b1, W2, b2, W3, b3).  Every agent must have the same depth
    and H, and the shapes must fit its observation and its action width act_dims[i] (None: 5 for every agent, the
    movement head alone); anything else raises ValueError.  Works on tensors of any device."""
    import torch
    if act_dims is None:
        act_dims = [5] * len(policies)
    depth = hidden = None
    params = []
    for i, pol in enumerate(policies):
        if isinstance(pol, torch.nn.Module):
            lin = [m for m in pol.modules() if isinstance(m, torch.nn.Linear)]
            if len(lin) == 2:
                pol = (lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias)
            elif len(lin) == 3:
                kinds = [type(m) for m in pol.children()] if isinstance(pol, torch.nn.Sequential) else []
                if kinds != [torch.nn.Linear, torch.nn.ReLU, torch.nn.Linear, torch.nn.ReLU, torch.nn.Linear]:
                    raise ValueError("policy %d must be Linear -> ReLU -> Linear -> ReLU -> Linear" % i)
                pol = tuple(t for m in lin for t in (m.weight, m.bias))
            else:
                raise ValueError("policy %d must be Linear -> ReLU -> Linear" % i)
        pol = tuple(pol)
        if len(pol) not in (4, 6):
            raise ValueError("policy %d: expected (W1, b1, W2, b2) or (W1, b1, W2, b2, W3, b3), got %d tensors" % (i, len(pol)))
        d, H = len(pol) // 2 - 1, int(pol[0].shape[0])
        if depth is None:
            depth, hidden = d, H
        if d != depth:
            raise ValueError("policy %d has %d hidden layers, policy 0 has %d: all actors must have the same depth" % (i, d, depth))
        ad = int(act_dims[i])
        want = [(hidden, obs_dims[i]), (hidden,)] + ([(ad, hidden), (ad,)] if depth == 1 else
                                                      [(hidden, hidden), (hidden,), (ad, hidden), (ad,)])
        if [tuple(t.shape) for t in pol] != want:
            raise ValueError("policy %d: expected shapes %s, got %s" % (i, want, [tuple(t.shape) for t in pol]))
        params.append(pol)
    return depth, hidden, params
