"""Glue between ``GpuVecEnv`` and the reference's learner for large N (SURVEY.md 8(f)2).

The reference's actor loop (``trainer.py:157-186``) is written for a handful of environments: per step it walks
``infos`` in Python (``:167-178``), appends to one ``ReplayMemory`` per environment in Python (``:183-185``) and
``Agent.learn`` samples ``int(batch_size / len(memory))`` transitions from EVERY memory (``agent.py:69``), which is
0 once there are more environments than batch entries.  At 4096 bins those loops, not the environment, set the
iteration rate.  This module keeps the loop's shape and removes the per-environment Python work:

* ``get_mask_from_state``  -- ``tools.get_mask_from_state`` (``tools.py:283-300``, selectedAction branch) as a view
  of the device observation;
* ``EpisodeStats``         -- the ``episode_rewards / episode_ratio / episode_counter`` deques of
  ``trainer.py:145-147,167-178`` fed from the step's result arrays (``LazyInfos.finished()``), no loop over bins;
* ``ReplayBank``           -- the N per-environment ring buffers of ``main.py:61-63`` as ONE device-resident bank
  ``[capacity, N, obs_len]``; ``append_batch`` replaces the loop of ``trainer.py:183-185``; ``sample`` draws a batch
  with the reference's segment rule made safe for N > batch_size (``segment_size``);
* ``segment_size``         -- the shim for ``agent.py:69``.

``ReplayBank`` samples uniformly, without priorities or n-step returns; it exists so that the actor loop can be run end
to end at N = 4096 and timed (``tools/actor_loop.py``).  The reference's learner memory (prioritized n-step replay,
``memory.py``) at N = 4096 is ``irbpp_b200.replay.PrioritizedReplayBank``, which also uses ``segment_size``.
"""
from collections import deque

import numpy as np


def get_mask_from_state(state, selected_action):
    """Action mask = column 4 of the candidate rows (reference ``tools.py:298-299``); ``state`` is the
    ``[N, obs_len]`` observation (device tensor or NumPy array), the result a view ``[N, selected_action]``."""
    n = state.shape[0]
    return state[:, :selected_action * 5].reshape(n, selected_action, 5)[:, :, 4]


def segment_size(batch_size, num_memories):
    """``agent.py:69`` computes ``int(batch_size / len(memory))`` transitions per memory, 0 for more memories than
    batch entries.  Returns ``(memories_to_sample, per_memory)``: every memory when they fit, else ``batch_size``
    randomly chosen memories with one transition each."""
    per = batch_size // num_memories
    if per >= 1:
        return num_memories, per
    return batch_size, 1


class EpisodeStats(object):
    """The three ``deque(maxlen=10)`` of ``trainer.py:145-147`` updated from a step's ``(done, infos)`` without a
    Python loop over the bins that did not finish (``trainer.py:167-178`` touches every bin)."""

    def __init__(self, maxlen=10):
        self.episode_rewards = deque(maxlen=maxlen)
        self.episode_ratio = deque(maxlen=maxlen)
        self.episode_counter = deque(maxlen=maxlen)
        self.episodes = 0

    def update(self, done, infos):
        idx, ep_r, ratio, counter, valid = infos.finished()
        if len(idx):                                   # finished episodes of this step only (in bin order, as the reference)
            keep = valid.astype(bool)
            tail = slice(-self.episode_rewards.maxlen, None)      # only the last maxlen can survive in the deques
            self.episode_rewards.extend(ep_r[keep][tail].tolist())
            self.episode_ratio.extend(ratio[keep][tail].tolist())
            self.episode_counter.extend(counter[keep][tail].tolist())
        self.episodes += int(len(idx))
        return infos.valid_array()


class ReplayBank(object):
    """One ring buffer for all N environments on the device: slot ``t mod capacity`` holds the transition every
    environment made at its step ``t`` (the reference keeps ``N`` ``ReplayMemory`` objects of capacity
    ``memory_capacity / N`` each, ``main.py:61-63``).  Invalid samples (``infos[i]['Valid'] == False``,
    ``trainer.py:183-185``) are stored with weight 0 and never sampled."""

    def __init__(self, num_envs, capacity_per_env, obs_len, device, state_dtype=None):
        import torch
        self._torch = torch
        self.n, self.cap, self.device = int(num_envs), int(capacity_per_env), torch.device(device)
        self.states = torch.empty((self.cap, self.n, obs_len), dtype=state_dtype or torch.float32, device=self.device)
        self.actions = torch.zeros((self.cap, self.n), dtype=torch.int64, device=self.device)
        self.rewards = torch.zeros((self.cap, self.n), dtype=torch.float32, device=self.device)
        self.nonterminal = torch.zeros((self.cap, self.n), dtype=torch.bool, device=self.device)
        self.valid = torch.zeros((self.cap, self.n), dtype=torch.bool, device=self.device)
        self.t = 0

    def __len__(self):
        return min(self.t, self.cap)

    def append_from_env(self, env, state, action, reward_clip=0.0):
        """The same append with the step's reward / done / valid taken from the environment's DEVICE result arrays
        (``GpuVecEnv.last_step_device``): no host round trip, five device-to-device copies."""
        torch = self._torch
        dv = env.last_step_device()
        s = self.t % self.cap
        self.states[s].copy_(state)
        self.actions[s].copy_(action.reshape(-1))
        if reward_clip > 0:
            torch.clamp(dv["reward"], -reward_clip, reward_clip, out=self.rewards[s])       # trainer.py:180-181
        else:
            self.rewards[s].copy_(dv["reward"])
        torch.eq(dv["done"], 0, out=self.nonterminal[s])
        torch.ne(dv["valid"], 0, out=self.valid[s])
        self.t += 1

    def append_batch(self, state, action, reward, done, valid=None):
        """``self.mem[i].append(state[i], action[i], reward[i], done[i])`` for every i (``trainer.py:183-185``) as
        five batched copies.  ``reward`` / ``done`` / ``valid`` may be host arrays (what ``envs.step`` returns)."""
        torch = self._torch
        s = self.t % self.cap
        self.states[s].copy_(state)
        self.actions[s].copy_(torch.as_tensor(action).reshape(-1).to(self.device, non_blocking=True))
        self.rewards[s].copy_(torch.as_tensor(reward).reshape(-1).to(self.device, non_blocking=True))
        self.nonterminal[s].copy_(~torch.as_tensor(np.asarray(done)).to(self.device, non_blocking=True))
        if valid is None:
            self.valid[s].fill_(True)
        else:
            self.valid[s].copy_(torch.as_tensor(np.asarray(valid)).to(self.device, non_blocking=True))
        self.t += 1

    def sample(self, batch_size, generator=None):
        """A batch drawn with the reference's segment rule (``agent.py:69-75``): ``per`` transitions from each of
        ``m`` memories (all of them when ``N <= batch_size``, else ``batch_size`` random ones).  Returns
        ``(env_idx, slot_idx, states, actions, rewards, next_states, nonterminals)``; next states are the
        following slot of the same environment (the newest slot is never drawn)."""
        torch = self._torch
        filled = len(self)
        if filled < 2:
            raise RuntimeError("not enough transitions")
        m, per = segment_size(batch_size, self.n)
        if m == self.n:
            envs = torch.arange(self.n, device=self.device).repeat_interleave(per)
        else:
            envs = torch.randperm(self.n, device=self.device, generator=generator)[:m]
        newest = (self.t - 1) % self.cap
        off = torch.randint(1, filled, (envs.numel(),), device=self.device, generator=generator)      # 1 .. filled-1 steps back
        slots = (newest - off) % self.cap
        nxt = (slots + 1) % self.cap
        return (envs, slots, self.states[slots, envs], self.actions[slots, envs], self.rewards[slots, envs],
                self.states[nxt, envs], self.nonterminal[slots, envs])
