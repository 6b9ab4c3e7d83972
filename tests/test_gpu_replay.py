"""PrioritizedReplayBank (irbpp_b200/replay.py, csrc/irbpp_replay.cuh) on the B200: the golden traces of the unmodified
memory.py, a 4096-bin trace driven by GpuVecEnv against the oracle port, the rule for more bins than batch entries, the
call shape of Agent.learn, and an append captured in a CUDA graph.  Tolerances as stated in test_replay_port."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from test_replay_port import GOLDENS, run_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _bank(N, C, L, **kw):
    from irbpp_b200.replay import PrioritizedReplayBank
    return PrioritizedReplayBank(N, C, L, DEV, **kw)


class GpuImpl(object):
    def __init__(self, bank):
        self.bank = bank

    def append(self, state, action, reward, done, valid):
        self.bank.append_batch(torch.from_numpy(np.ascontiguousarray(state)).to(DEV), action, reward, done, valid)

    def sample(self, batch, u, beta):
        self.bank.priority_weight = beta
        return [t.cpu().numpy() for t in self.bank.sample(batch, u_table=u)]

    def update(self, idx, loss, exponent):
        assert exponent == self.bank.priority_exponent
        self.bank.update_priorities(torch.from_numpy(idx).to(DEV), torch.from_numpy(np.asarray(loss, np.float32)))

    def snapshot(self):
        return self.bank.snapshot()


@pytest.mark.parametrize("name", GOLDENS)
def test_gpu_replay_reproduces_reference_golden(name):
    d = load_golden(name)
    bank = _bank(int(d["N"]), int(d["C"]), int(d["L"]), discount=float(d["discount"]), multi_step=int(d["n"]),
                 priority_exponent=float(d["priority_exponent"]))
    assert run_golden(d, GpuImpl(bank)) == len(d["round_step"])


def _valid_actions(state, sel, gen):
    from irbpp_b200.learner_glue import get_mask_from_state
    q = torch.rand((state.shape[0], sel), device=state.device, generator=gen)
    q[get_mask_from_state(state, sel) == 0] = -1.0
    return q.argmax(1)


def test_gpu_replay_env_trace_4096_bins_matches_port():
    """N = 4096, C = 24 (1e5 / 4096), L = 3533: 200 steps of GpuVecEnv with episode ends, append_from_env with the
    reward clip of trainer.py:181-182, sample / update every 4th step from step 40 (N > batch: device-chosen banks),
    every tree, index, full, max and t against oracle/replay_port.py."""
    from irbpp_b200 import shapes
    from irbpp_b200.vec_env import GpuVecEnv
    from oracle.replay_port import ReplayPort
    N, C, sel, batch, clip = 4096, 24, 500, 64, 10.0
    env = GpuVecEnv(shapes.make_blockout_library(32, seed=1), None, num_envs=N, device=DEV, item_seed=3)
    L = env.obs_len
    assert L == 3533
    bank = _bank(N, C, L, priority_weight=0.4)
    port = ReplayPort(N, C, L, 0.99, 3)
    gen = torch.Generator(device=DEV); gen.manual_seed(0)
    rng = np.random.default_rng(0)
    state = env.reset()
    clip_t = torch.ones((N, 1)) * clip
    episodes = rounds = 0
    for T in range(1, 201):
        action = _valid_actions(state, sel, gen)
        next_state, reward, done, infos = env.step(action.cpu().numpy())
        bank.append_from_env(env, state, action, reward_clip=clip)
        r = torch.maximum(torch.minimum(reward, clip_t), -clip_t)
        port.append(state.cpu().numpy(), action.cpu().numpy(), r.numpy()[:, 0], done, infos.valid_array())
        episodes += int(np.sum(done))
        s = bank.snapshot()
        assert np.array_equal(s["tree"], port.tree), T
        assert np.array_equal(s["index"], port.index) and np.array_equal(s["full"], port.full), T
        assert np.array_equal(s["max"], port.max) and np.array_equal(s["t"], port.t), T
        if T >= 40 and T % 4 == 0:
            bank.priority_weight = port.priority_weight = min(0.4 + 0.01 * T, 1.0)
            u = rng.random((batch, 64))
            got = [t.cpu().numpy() for t in bank.sample(batch, u_table=u)]
            want = port.sample(batch, u, banks=bank.last_banks.cpu().numpy())
            for j in (0, 1, 2, 4, 5):
                assert np.array_equal(got[j], want[j]), (T, j)
            assert np.all(np.abs(got[3] - want[3]) <= 1e-6 * (1 + np.abs(want[3]))), T
            assert np.array_equal(got[6], np.ones(batch, np.float32))           # one draw per bank: weight 1
            loss = torch.from_numpy(rng.uniform(0.01, 4, batch).astype(np.float32))
            bank.update_priorities(torch.from_numpy(got[0]).to(DEV), loss)
            port.update_priorities(got[0], np.power(loss.numpy(), 0.5))
            assert np.array_equal(bank.tree.cpu().numpy(), port.tree) and np.array_equal(bank.max_priority.cpu().numpy(), port.max), T
            rounds += 1
        state = next_state
    env.close()
    assert episodes > 100 and rounds == 41


def test_gpu_replay_more_banks_than_batch_rule():
    """N > batch with the production stream: `batch` distinct banks, every draw passes the rejection rule of
    memory.py:169 with its state gathered from its slot, every weight is 1, and the banks are chosen uniformly."""
    N, C, L, batch, n = 4096, 24, 40, 64, 3
    bank = _bank(N, C, L, seed=9)
    g = torch.Generator(device=DEV); g.manual_seed(1)
    for t in range(30):
        bank.append_batch(torch.randn((N, L), device=DEV, generator=g), torch.randint(0, 500, (N,)),
                          torch.rand(N), torch.rand(N) < 0.1, torch.rand(N) < 0.9)
    idx, st, act, ret, nx, nt, wt = bank.sample(batch)
    T = 2 * C - 1
    banks = bank.last_banks.cpu().numpy()
    gi = idx.cpu().numpy()
    assert len(set(banks.tolist())) == batch and np.array_equal(gi // T, banks)
    node = gi % T
    slot = node - (C - 1)
    assert np.all(slot >= 0)
    w = bank.index.cpu().numpy()[banks]
    assert np.all((w - slot) % C > n) and np.all((slot - w) % C >= 1)
    assert np.all(bank.tree.cpu().numpy()[banks, node] != 0)
    assert torch.equal(st, bank.states[torch.from_numpy(banks).long().to(DEV), torch.from_numpy(slot).to(DEV), :L])
    assert torch.equal(wt, torch.ones(batch, device=DEV))
    small = _bank(8, C, L, seed=2)                              # uniformity: 8 banks, 4 per call
    for t in range(30):
        small.append_batch(torch.randn((8, L), device=DEV, generator=g), np.zeros(8), np.ones(8), np.zeros(8, bool))
    counts = np.zeros(8)
    for _ in range(2000):
        small.sample(4)
        counts += np.bincount(small.last_banks.cpu().numpy(), minlength=8)
    assert np.all(np.abs(counts - 1000) < 120), counts
    empty = _bank(4, C, L, max_attempts=64)
    with pytest.raises(RuntimeError, match="rejected"):
        empty.sample(4)


@pytest.mark.parametrize("N,L", [(4096, 3533), (4096, 10 + 1024), (16, 3533)])
def test_gpu_replay_runs_unmodified_agent_learn_call_shape(N, L):
    """agent.py:68-124 verbatim in call shape, with a linear stand-in for the network: len(memory) == 1, so one
    sample(batch_size); the CPU loss goes back through memory[0].update_priorities.  Location (L = 3533) and order
    (k + 1024) observations of the hierarchical trainer."""
    C, batch_size = 24, 64
    bank = _bank(N, C, L, priority_weight=0.4)
    g = torch.Generator(device=DEV); g.manual_seed(5)
    for t in range(30):
        bank.append_batch(torch.randn((N, L), device=DEV, generator=g), torch.randint(0, 10, (N,)),
                          torch.rand(N), torch.rand(N) < 0.05)
    W = torch.randn((L, 10), device=DEV, generator=g) * 0.01
    memory = bank.as_agent_memory()
    for it in range(3):
        segment_size = int(batch_size / len(memory))
        idxs, states, actions, returns, next_states, nonterminals, weights = [], [], [], [], [], [], []
        for mem in memory:
            idx, state, action, ret, next_state, nonterminal, weight = mem.sample(segment_size)
            idxs.append(idx), states.append(state), actions.append(action), returns.append(ret)
            next_states.append(next_state), nonterminals.append(nonterminal), weights.append(weight)
        states = torch.cat(states, 0)
        actions = torch.cat(actions, 0)
        returns = torch.cat(returns, 0)
        next_states = torch.cat(next_states, 0)
        nonterminals = torch.cat(nonterminals, 0).reshape(batch_size, 1)
        weights = torch.cat(weights, 0)
        q = states @ W
        target = returns.unsqueeze(1) + nonterminals * 0.99 ** 3 * (next_states @ W).max(1, keepdim=True)[0]
        loss = (q[range(batch_size), actions] - target[:, 0]).abs() + 1e-3
        assert torch.isfinite((weights * loss).mean())          # the weighted loss agent.py:119 backpropagates
        for i in range(len(memory)):
            memory[i].update_priorities(idxs[i], loss[i * segment_size:(i + 1) * segment_size].detach().cpu())
        leaves = bank.tree.reshape(-1)[idxs[0]].cpu().numpy()
        last = {int(k): j for j, k in enumerate(idxs[0].cpu().numpy())}          # a later duplicate wins
        want = np.power(loss.detach().cpu().numpy(), 0.5).astype(np.float32)
        assert all(leaves[j] == want[last[int(k)]] for j, k in enumerate(idxs[0].cpu().numpy()))
        assert states.shape == (batch_size, L) and weights.shape == (batch_size,) and actions.dtype == torch.int64
        bank.priority_weight = min(bank.priority_weight + 0.1, 1)


def test_gpu_replay_append_from_env_in_cuda_graph():
    """append_from_env reads the step's results on the device and never synchronises: it can be captured in a CUDA
    graph, and the replayed graph appends exactly what the eager call appends."""
    from irbpp_b200 import shapes
    from irbpp_b200.vec_env import GpuVecEnv
    N, C = 256, 24
    env = GpuVecEnv(shapes.make_blockout_library(16, seed=2), None, num_envs=N, device=DEV, item_seed=4)
    L = env.obs_len
    eager, graphed = _bank(N, C, L), _bank(N, C, L)
    gen = torch.Generator(device=DEV); gen.manual_seed(2)
    state = env.reset()
    static_state, static_action = torch.zeros_like(state), torch.zeros(N, dtype=torch.int64, device=DEV)
    action = _valid_actions(state, 500, gen)
    env.step(action.cpu().numpy())
    static_state.copy_(state); static_action.copy_(action)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        graphed.append_from_env(env, static_state, static_action, reward_clip=10.0)       # warm-up (not captured)
    torch.cuda.current_stream().wait_stream(s)
    eager.append_from_env(env, state, action, reward_clip=10.0)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.append_from_env(env, static_state, static_action, reward_clip=10.0)
    for t in range(25):
        action = _valid_actions(state, 500, gen)
        next_state = env.step(action.cpu().numpy())[0]
        static_state.copy_(state); static_action.copy_(action)
        graph.replay()
        eager.append_from_env(env, state, action, reward_clip=10.0)
        state = next_state
    torch.cuda.synchronize()
    a, b = eager.snapshot(), graphed.snapshot()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    for name in ("states", "actions", "rewards", "nonterminals"):
        assert torch.equal(getattr(eager, name), getattr(graphed, name)), name
    env.close()
