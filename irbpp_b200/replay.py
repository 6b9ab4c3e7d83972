"""Prioritized n-step replay for N bins on the device: the reference's learner memory at N = 4096 (SURVEY.md 8(f)2).

``main.py:61-63`` builds one ``ReplayMemory`` (``memory.py:95-208``) per bin, ``trainer.py:184-186`` appends to them in
a Python loop and ``agent.py:69`` samples ``int(batch_size / len(memory))`` transitions from each, which is 0 once there
are more bins than batch entries.  ``PrioritizedReplayBank`` holds the N memories as N banks of one device allocation;
bank ``b`` behaves exactly like ``ReplayMemory(args, capacity, obs_len)`` (sum tree, write index, ``full``, running max
priority, episode timestep) and every operation is one batched CUDA launch (``csrc/irbpp_replay.cuh``):

* ``append_from_env`` / ``append_batch`` -- ``self.mem[i].append(...)`` for every bin whose ``infos[i]['Valid']`` is set;
* ``sample(batch_size)`` -- what ``Agent.learn`` concatenates from the memories (``agent.py:68-82``).  N <= batch: every
  bank gives ``batch // N`` stratified draws, as in the reference.  N > batch (where the reference draws nothing):
  ``batch`` banks chosen uniformly without replacement on the device, one draw each; the reference's weight formula
  normalises a single draw by itself, so every weight is 1;
* ``update_priorities(tree_idxs, losses)`` -- ``np.power(loss, omega)`` on the host as in ``memory.py:207``, then the
  leaf writes in batch order on the device;
* ``as_agent_memory()`` -- ``[self]``: the unmodified ``Agent.learn(memory)`` then sees one memory, samples
  ``batch_size`` from it and hands the CPU loss to ``memory[0].update_priorities``.

Draws come from a counter-based stream (seed, call counter); a row that is rejected ``max_attempts`` times (the
reference would retry forever, e.g. on an empty bank) raises ``RuntimeError``.
"""
import ctypes

import numpy as np

from . import _lib
from .learner_glue import segment_size


class PrioritizedReplayBank(object):
    def __init__(self, num_envs, capacity_per_env, obs_len, device, discount=0.99, multi_step=3, priority_weight=1.0,
                 priority_exponent=0.5, seed=0, max_attempts=4096):
        import torch
        self._torch = torch
        self._lib = _lib.load()
        if not 0 <= int(multi_step) <= _lib.REPLAY_MAX_STEPS:
            raise ValueError("multi_step must be in [0, %d]" % _lib.REPLAY_MAX_STEPS)
        self.num_envs, self.capacity, self.obs_len = int(num_envs), int(capacity_per_env), int(obs_len)
        self.device = torch.device(device)
        self.discount, self.n = discount, int(multi_step)
        self.priority_weight = priority_weight          # beta; annealed by the caller (trainer.py:196-197)
        self.priority_exponent = priority_exponent
        self.seed, self.max_attempts, self.calls = int(seed), int(max_attempts), 0
        N, C, dev = self.num_envs, self.capacity, self.device
        self.row_stride = (self.obs_len + 3) // 4 * 4
        self.tree = torch.zeros((N, 2 * C - 1), dtype=torch.float32, device=dev)
        self.states = torch.zeros((N, C, self.row_stride), dtype=torch.float32, device=dev)
        self.actions = torch.zeros((N, C), dtype=torch.int64, device=dev)
        self.rewards = torch.zeros((N, C), dtype=torch.float32, device=dev)
        self.nonterminals = torch.zeros((N, C), dtype=torch.uint8, device=dev)
        self.index = torch.zeros(N, dtype=torch.int32, device=dev)
        self.full = torch.zeros(N, dtype=torch.uint8, device=dev)
        self.max_priority = torch.ones(N, dtype=torch.float32, device=dev)      # memory.py:27
        self.timestep = torch.zeros(N, dtype=torch.int32, device=dev)
        self._banks = _lib.IrbppReplayBanks(N, C, self.obs_len, self.row_stride, *[t.data_ptr() for t in (
            self.tree, self.states, self.actions, self.rewards, self.nonterminals, self.index, self.full,
            self.max_priority, self.timestep)])
        self._scaling = [float(np.float32(discount ** i)) for i in range(self.n)]   # memory.py:107 as float32

    def _stream(self):
        return self._torch.cuda.current_stream(self.device).cuda_stream

    def _check(self, rc):
        _lib.check(self._lib, None, rc)

    def _append(self, state, action, reward, done, valid, reward_clip):
        if state.dim() != 2 or state.shape[0] != self.num_envs or state.shape[1] < self.obs_len or state.stride(1) != 1 \
                or state.dtype != self._torch.float32 or state.device != self.device:
            raise ValueError("state must be a float32 [N, >= obs_len] tensor with unit column stride on %s" % self.device)
        self._check(self._lib.irbpp_replay_append(
            ctypes.byref(self._banks), state.data_ptr(), state.stride(0), action.data_ptr(), reward.data_ptr(),
            done.data_ptr(), valid.data_ptr() if valid is not None else None, float(reward_clip), self._stream()))

    def _dev(self, x, dtype):
        torch = self._torch
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))
        t = t.reshape(-1).to(device=self.device, dtype=dtype)
        if t.numel() != self.num_envs:
            raise ValueError("expected %d entries, got %d" % (self.num_envs, t.numel()))
        return t.contiguous()

    def append_from_env(self, env, state, action, reward_clip=0.0):
        """``trainer.py:181-186`` for every bin: ``state`` / ``action`` as the actor loop holds them (device), the step's
        reward / done / valid read from the environment's device result arrays (``GpuVecEnv.last_step_device``).  One
        launch, no host round trip (it can be captured in a CUDA graph)."""
        dv = env.last_step_device()
        torch = self._torch
        action = action.reshape(-1)
        if action.dtype != torch.int64 or not action.is_contiguous():
            action = action.to(torch.int64).contiguous()
        self._append(state, action, dv["reward"], dv["done"], dv["valid"], reward_clip)

    def append_batch(self, state, action, reward, done, valid=None):
        """``self.mem[i].append(state[i], action[i], reward[i], done[i])`` for every i with ``valid[i]`` (all when
        ``valid`` is None); ``reward`` is used as given (clip it first, as ``trainer.py:181-182`` does).  ``action`` /
        ``reward`` / ``done`` / ``valid`` may be host arrays."""
        torch = self._torch
        self._append(state, self._dev(action, torch.int64), self._dev(reward, torch.float32),
                     self._dev(done, torch.uint8), None if valid is None else self._dev(valid, torch.uint8), 0.0)

    def sample(self, batch_size, u_table=None):
        """``(tree_idxs, states, actions, returns, next_states, nonterminals, weights)`` shaped as ``Agent.learn`` builds
        them (``agent.py:77-82``), all on the device; ``tree_idxs`` int64 [B] = bank * (2C-1) + tree node.
        ``u_table`` (float64 [B, A]) replaces the random stream: draw ``a`` of row ``r`` uses ``u_table[r, a]``."""
        torch = self._torch
        m, per = segment_size(batch_size, self.num_envs)
        rows, dev = m * per, self.device
        a = _lib.IrbppReplaySampleArgs()
        a.batch, a.multi_step = int(batch_size), self.n
        for k, s in enumerate(self._scaling):
            a.n_step_scaling[k] = s
        a.priority_weight = float(self.priority_weight)
        a.seed, a.counter = self.seed & 0xFFFFFFFFFFFFFFFF, self.calls
        self.calls += 1
        if u_table is not None:
            table = torch.as_tensor(np.ascontiguousarray(u_table, dtype=np.float64)).to(dev)
            if table.dim() != 2 or table.shape[0] < rows:
                raise ValueError("u_table must be [>= %d, attempts]" % rows)
            a.u_table, a.max_attempts = table.data_ptr(), table.shape[1]
        else:
            table, a.u_table, a.max_attempts = None, None, self.max_attempts
        self.last_banks = torch.empty(m, dtype=torch.int32, device=dev)
        out = (torch.empty(rows, dtype=torch.int64, device=dev), torch.empty((rows, self.obs_len), dtype=torch.float32, device=dev),
               torch.empty(rows, dtype=torch.int64, device=dev), torch.empty(rows, dtype=torch.float32, device=dev),
               torch.empty((rows, self.obs_len), dtype=torch.float32, device=dev), torch.empty(rows, dtype=torch.float32, device=dev),
               torch.empty(rows, dtype=torch.float32, device=dev))
        err = torch.empty(rows, dtype=torch.int32, device=dev)
        a.banks = self.last_banks.data_ptr()
        a.tree_index, a.states, a.actions, a.returns, a.next_states, a.nonterminals, a.weights = [t.data_ptr() for t in out]
        a.error = err.data_ptr()
        self._check(self._lib.irbpp_replay_sample(ctypes.byref(self._banks), ctypes.byref(a), self._stream()))
        if bool(err.any()):
            raise RuntimeError("replay sample: %d of %d draws still rejected after %d attempts (empty bank?)"
                               % (int(err.sum()), rows, a.max_attempts))
        return out

    def update_priorities(self, idxs, priorities):
        """``memory.py:206-208``: ``priorities`` (the CPU loss ``agent.py:124`` passes) raised to ``priority_exponent``
        with ``np.power`` on the host, then written to the leaves ``idxs`` (from ``sample``) in order on the device."""
        torch = self._torch
        if isinstance(priorities, torch.Tensor):
            priorities = priorities.detach().cpu()
        powered = np.power(priorities, self.priority_exponent)
        pr = torch.as_tensor(np.asarray(powered, dtype=np.float32)).reshape(-1).to(self.device)
        idx = torch.as_tensor(idxs, dtype=torch.int64).reshape(-1).to(self.device).contiguous()
        if idx.numel() != pr.numel():
            raise ValueError("%d indices for %d priorities" % (idx.numel(), pr.numel()))
        self._check(self._lib.irbpp_replay_update_priorities(ctypes.byref(self._banks), idx.data_ptr(), pr.data_ptr(),
                                                             int(idx.numel()), self._stream()))

    def as_agent_memory(self):
        """The ``memory`` argument of the unmodified ``Agent.learn`` (``agent.py:68``)."""
        return [self]

    def snapshot(self):
        """Host copies of the bookkeeping: ``tree`` [N, 2C-1], ``index``, ``full``, ``max`` and ``t`` [N]."""
        return {"tree": self.tree.cpu().numpy(), "index": self.index.cpu().numpy(), "full": self.full.cpu().numpy().astype(bool),
                "max": self.max_priority.cpu().numpy(), "t": self.timestep.cpu().numpy()}
