"""The replay kernels of csrc/irbpp_replay.cuh run on host threads (tests/host_harness/cuda_emu.h, built by
test_kernels_emulated.build_emulated) through the C ABI against the golden traces of the unmodified memory.py, with the
tolerances of test_replay_port.  The same checks on the B200 are in test_gpu_replay.py."""
import ctypes

import numpy as np
import pytest

from conftest import load_golden
from test_kernels_emulated import build_emulated
from test_replay_port import GOLDENS, powered, run_golden

pytestmark = pytest.mark.timeout(900)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    return build_emulated(str(tmp_path_factory.mktemp("emu_replay")))


def _P(a):
    return ctypes.c_void_p(a.ctypes.data)


class EmuReplay(object):
    """irbpp_replay_* of the emulated library on NumPy buffers (device == host under the emulation)."""

    def __init__(self, lib, N, C, L, n, discount):
        from irbpp_b200 import _lib
        self.lib, self._lib, self.N, self.C, self.L, self.n = lib, _lib, N, C, L, n
        stride = (L + 3) // 4 * 4
        self.tree = np.zeros((N, 2 * C - 1), np.float32)
        self.states = np.zeros((N, C, stride), np.float32)
        self.actions = np.zeros((N, C), np.int64)
        self.rewards = np.zeros((N, C), np.float32)
        self.nonterminals = np.zeros((N, C), np.uint8)
        self.index = np.zeros(N, np.int32)
        self.full = np.zeros(N, np.uint8)
        self.max = np.ones(N, np.float32)
        self.t = np.zeros(N, np.int32)
        self.banks = _lib.IrbppReplayBanks(N, C, L, stride, *[a.ctypes.data for a in (
            self.tree, self.states, self.actions, self.rewards, self.nonterminals, self.index, self.full, self.max, self.t)])
        self.scaling = [float(np.float32(discount ** i)) for i in range(n)]

    def append(self, state, action, reward, done, valid):
        state = np.ascontiguousarray(state, np.float32)
        action = np.ascontiguousarray(action, np.int64)
        reward = np.ascontiguousarray(reward, np.float32)
        done = np.ascontiguousarray(done, np.uint8)
        valid = np.ascontiguousarray(valid, np.uint8)
        assert self.lib.emu_irbpp_replay_append(ctypes.byref(self.banks), _P(state), ctypes.c_int64(state.shape[1]), _P(action),
                                                _P(reward), _P(done), _P(valid), ctypes.c_float(0.0), None) == 0

    def sample(self, batch, u, beta):
        from irbpp_b200.learner_glue import segment_size
        m, per = segment_size(batch, self.N)
        rows = m * per
        u = np.ascontiguousarray(u, np.float64)
        outs = (np.zeros(rows, np.int64), np.zeros((rows, self.L), np.float32), np.zeros(rows, np.int64),
                np.zeros(rows, np.float32), np.zeros((rows, self.L), np.float32), np.zeros(rows, np.float32),
                np.zeros(rows, np.float32))
        banks, err = np.zeros(m, np.int32), np.zeros(rows, np.int32)
        a = self._lib.IrbppReplaySampleArgs()
        a.batch, a.multi_step, a.priority_weight = batch, self.n, beta
        for k, s in enumerate(self.scaling):
            a.n_step_scaling[k] = s
        a.u_table, a.max_attempts, a.banks = u.ctypes.data, u.shape[1], banks.ctypes.data
        a.tree_index, a.states, a.actions, a.returns, a.next_states, a.nonterminals, a.weights = [o.ctypes.data for o in outs]
        a.error = err.ctypes.data
        assert self.lib.emu_irbpp_replay_sample(ctypes.byref(self.banks), ctypes.byref(a), None) == 0
        assert not err.any()
        assert np.array_equal(banks, np.arange(m))
        return outs

    def update(self, idx, loss, exponent=None):
        idx = np.ascontiguousarray(idx, np.int64)
        pr = np.ascontiguousarray(loss if exponent is None else powered(loss, exponent), np.float32)
        assert self.lib.emu_irbpp_replay_update_priorities(ctypes.byref(self.banks), _P(idx), _P(pr), len(idx), None) == 0

    def snapshot(self):
        return {"tree": self.tree, "index": self.index, "full": self.full.astype(bool), "max": self.max, "t": self.t}


@pytest.mark.parametrize("name", GOLDENS)
def test_emulated_replay_kernels_reproduce_reference_golden(emu, name):
    d = load_golden(name)
    impl = EmuReplay(emu, int(d["N"]), int(d["C"]), int(d["L"]), int(d["n"]), float(d["discount"]))
    assert run_golden(d, impl) == len(d["round_step"])


def test_emulated_replay_more_banks_than_batch(emu):
    """N > batch: `batch` distinct banks, one draw each, every weight 1; the draw follows the port's rule for the
    chosen banks; duplicate leaves in one update: the later write wins."""
    from oracle.replay_port import ReplayPort
    N, C, L, n, batch = 9, 24, 6, 3, 4
    rng = np.random.default_rng(4)
    impl, port = EmuReplay(emu, N, C, L, n, 0.99), ReplayPort(N, C, L, 0.99, n)
    for t in range(40):
        args = (rng.normal(size=(N, L)).astype(np.float32), rng.integers(0, 500, N), rng.uniform(-1, 5, N).astype(np.float32),
                rng.random(N) < 0.1, rng.random(N) < 0.9)
        impl.append(*args)
        port.append(*args)
    from irbpp_b200 import _lib
    for rnd in range(3):
        u = rng.random((batch, 16))
        outs = (np.zeros(batch, np.int64), np.zeros((batch, L), np.float32), np.zeros(batch, np.int64), np.zeros(batch, np.float32),
                np.zeros((batch, L), np.float32), np.zeros(batch, np.float32), np.zeros(batch, np.float32))
        banks, err = np.zeros(batch, np.int32), np.zeros(batch, np.int32)
        a = _lib.IrbppReplaySampleArgs()
        a.batch, a.multi_step, a.priority_weight, a.seed, a.counter = batch, n, 0.6, 5, rnd
        for k in range(n):
            a.n_step_scaling[k] = float(np.float32(0.99 ** k))
        a.u_table, a.max_attempts, a.banks = u.ctypes.data, u.shape[1], banks.ctypes.data
        a.tree_index, a.states, a.actions, a.returns, a.next_states, a.nonterminals, a.weights = [o.ctypes.data for o in outs]
        a.error = err.ctypes.data
        assert emu.emu_irbpp_replay_sample(ctypes.byref(impl.banks), ctypes.byref(a), None) == 0
        assert not err.any() and len(set(banks.tolist())) == batch and banks.min() >= 0 and banks.max() < N
        assert np.array_equal(outs[6], np.ones(batch, np.float32))
        port.priority_weight = 0.6
        want = port.sample(batch, u, banks=banks)
        for j in (0, 1, 2, 4, 5):                   # tree index, state, action, next state, nonterminal
            assert np.array_equal(outs[j], want[j]), j
        assert np.all(np.abs(outs[3] - want[3]) <= 1e-6 * (1 + np.abs(want[3])))
        idx = np.concatenate([outs[0], outs[0][:1]])
        pr = rng.uniform(0.1, 3, len(idx)).astype(np.float32)
        impl.update(idx, pr)
        port.update_priorities(idx, pr)
        assert np.array_equal(impl.tree, port.tree) and np.array_equal(impl.max, port.max)
