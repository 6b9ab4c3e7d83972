"""NumPy restatement of the reference's prioritized replay memory (memory.py:15-208) for N banks at once.

TEST INFRASTRUCTURE ONLY: the checker of ``irbpp_b200.replay.PrioritizedReplayBank`` on machines without the reference
tree.  Bank ``b`` is one ``ReplayMemory(args, capacity, obs_len)``; the arithmetic follows what the reference computes
(measured on it, see csrc/irbpp_replay.cuh):

* ``SegmentTree``: ``2C-1`` float32 nodes, leaves ``C-1 .. 2C-2`` (``memory.py:29``); ``update`` sets the leaf and
  re-adds its ancestors in float32 (``:45-56``); ``append`` stores the transition, writes the leaf with the current
  max and advances ``index`` / ``full`` (``:58-69``); the stored action, reward and nonterminal are float32 (``:30-34``);
* ``ReplayMemory.append``: nonterminal = ``not terminal``, ``t`` restarts at 0 after a terminal (``:110-113``);
* ``_get_sample_from_segment``: ``segment = total / batch`` and ``i * segment`` in float32, the draw
  ``lo + (hi - lo) * u`` in float64 (NumPy's uniform), the descent on the float32 rounding of the draw with float32
  subtractions (``:72-79``), the rejection rule of ``:169`` and the n-step window of ``_get_transition_new``
  (``:115-130``: position t is real while position t-1 was nonterminal, else blank);
* ``sample``: IS weights ``(capacity * p / total) ** -beta`` in float32 normalised by the maximum of the bank's draws
  (``:199-202``); ``ndarray / p_total`` is ``Tensor.__rtruediv__``, which torch computes as ``p * (1 / total)``;
* ``update_priorities``: writes in order, ``max`` over every written value (``:206-208``); the caller passes the
  already powered priorities (``np.power`` stays with the caller, as on the device path).

``u[row, attempt]`` replaces ``np.random.uniform``'s stream.  Returns are summed in float32 in index order (the
reference's ``torch.matmul`` may associate differently: compare them with a tolerance).
"""
import numpy as np


class ReplayPort(object):
    def __init__(self, num_banks, capacity, obs_len, discount=0.99, multi_step=3, priority_weight=1.0):
        N, C = int(num_banks), int(capacity)
        self.N, self.C, self.L, self.n = N, C, int(obs_len), int(multi_step)
        self.priority_weight = priority_weight
        self.scale = np.array([discount ** i for i in range(self.n)], dtype=np.float32)      # memory.py:107
        self.tree = np.zeros((N, 2 * C - 1), np.float32)
        self.states = np.zeros((N, C, self.L), np.float32)
        self.actions = np.zeros((N, C), np.float32)
        self.rewards = np.zeros((N, C), np.float32)
        self.nonterminals = np.zeros((N, C), np.float32)
        self.index = np.zeros(N, np.int64)
        self.full = np.zeros(N, bool)
        self.max = np.ones(N, np.float32)
        self.t = np.zeros(N, np.int64)

    def _propagate(self, banks, nodes):
        nodes = nodes.copy()
        while True:
            live = nodes > 0
            if not live.any():
                return
            b, nd = banks[live], (nodes[live] - 1) // 2
            self.tree[b, nd] = self.tree[b, 2 * nd + 1] + self.tree[b, 2 * nd + 2]
            nodes[live] = nd

    def append(self, state, action, reward, done, valid=None):
        """``mem[i].append(state[i], action[i], reward[i], done[i])`` for every i with ``valid[i]``."""
        state = np.asarray(state, np.float32)
        done = np.asarray(done, bool).reshape(-1)
        valid = np.ones(self.N, bool) if valid is None else np.asarray(valid, bool).reshape(-1)
        b = np.nonzero(valid)[0]
        slot = self.index[b]
        self.states[b, slot] = state[b, :self.L]
        self.actions[b, slot] = np.asarray(action).reshape(-1)[b].astype(np.float32)
        self.rewards[b, slot] = np.asarray(reward, np.float32).reshape(-1)[b]
        self.nonterminals[b, slot] = (~done[b]).astype(np.float32)
        leaf = slot + self.C - 1
        self.tree[b, leaf] = self.max[b]
        self._propagate(b, leaf)
        self.index[b] = (slot + 1) % self.C
        self.full[b] |= self.index[b] == 0
        self.t[b] = np.where(done[b], 0, self.t[b] + 1)

    def _draw(self, b, i, per, u_row):
        tree, C = self.tree[b], self.C
        total = tree[0]
        segment = np.float32(total / np.float32(per))
        lo, hi = np.float32(np.float32(i) * segment), np.float32(np.float32(i + 1) * segment)
        for u in u_row:
            v = float(lo) + (float(hi) - float(lo)) * float(u)
            x, node = np.float32(v), 0
            while 2 * node + 1 < 2 * C - 1:
                left = 2 * node + 1
                if x <= tree[left]:
                    node = left
                else:
                    x, node = np.float32(x - tree[left]), left + 1
            idx, w = node - C + 1, int(self.index[b])
            if (w - idx) % C > self.n and (idx - w) % C >= 1 and tree[node] != 0:
                return node
        raise RuntimeError("bank %d row %d: no valid draw in %d attempts" % (b, i, len(u_row)))

    def sample(self, batch_size, u, banks=None):
        """``per`` draws from each bank (``agent.py:69``) or, for N > batch, one draw from each of ``banks``; row ``r``
        uses ``u[r, :]``.  Returns ``(tree_idx, states, actions, returns, next_states, nonterminals, weights)`` with
        ``tree_idx = bank * (2C-1) + node``."""
        per = batch_size // self.N
        if per >= 1:
            banks = np.arange(self.N)
        else:
            per, banks = 1, np.asarray(banks)
        C, L, n = self.C, self.L, self.n
        rows = len(banks) * per
        out_idx = np.zeros(rows, np.int64)
        st, nx = np.zeros((rows, L), np.float32), np.zeros((rows, L), np.float32)
        act, ret = np.zeros(rows, np.int64), np.zeros(rows, np.float32)
        nt, wt = np.zeros(rows, np.float32), np.zeros(rows, np.float32)
        r = 0
        for b in banks:
            total = self.tree[b, 0]
            cap = C if self.full[b] else int(self.index[b])
            w0 = r
            for i in range(per):
                node = self._draw(b, i, per, u[r])
                idx = node - C + 1
                live, R = True, np.float32(0)
                for t in range(n):
                    if t > 0:
                        live = live and self.nonterminals[b, (idx + t - 1) % C] != 0
                    rew = self.rewards[b, (idx + t) % C] if live else np.float32(0)
                    R = np.float32(R + np.float32(rew * self.scale[t]))
                if n > 0:
                    live = live and self.nonterminals[b, (idx + n - 1) % C] != 0
                out_idx[r] = b * (2 * C - 1) + node
                st[r] = self.states[b, idx]
                act[r] = int(self.actions[b, idx])
                ret[r] = R
                if live:
                    nx[r] = self.states[b, (idx + n) % C]
                    nt[r] = self.nonterminals[b, (idx + n) % C]
                x = np.float32(np.float32(cap) * np.float32(self.tree[b, node] * np.float32(np.float32(1) / total)))
                wt[r] = np.float32(1) / x if self.priority_weight == 1 else np.power(x, np.float32(-self.priority_weight))
                r += 1
            wt[w0:r] = wt[w0:r] / wt[w0:r].max()
        return out_idx, st, act, ret, nx, nt, wt

    def update_priorities(self, tree_idx, priorities):
        T = 2 * self.C - 1
        for g, p in zip(np.asarray(tree_idx).reshape(-1), np.asarray(priorities, np.float32).reshape(-1)):
            b, node = int(g) // T, int(g) % T
            self.tree[b, node] = p
            self._propagate(np.array([b]), np.array([node]))
            self.max[b] = p if p > self.max[b] else self.max[b]
