"""The oracle's restatement of the reference's prioritized replay (oracle/replay_port.py) against the golden traces of
the unmodified memory.py (tests/golden/make_replay_golden.py), and against memory.py itself on fresh random traces where
the reference tree is mounted.  ``run_golden`` drives any implementation through a trace; the emulated-kernel and GPU
tests reuse it.

Exact (==): sum trees after every append and update, index / full / max / t, sampled tree indices, states, actions,
next states, nonterminals, and the weights at beta = 1.  Within a tolerance: returns (|d| <= 1e-6 * (1 + |R|): the
reference's torch.matmul may associate the n-term dot product differently) and weights at beta != 1
(|d| <= 4e-7 * w: a float32 pow of another library may round the last bit differently)."""
import importlib.util
import os
import warnings

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden

GOLDENS = ("replay_c24", "replay_c16")


def powered(loss, exponent):
    """memory.py:207 on the CPU loss agent.py:124 passes."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)          # NumPy 2 on torch's __array_wrap__
        return np.asarray(np.power(torch.from_numpy(np.asarray(loss, np.float32)), exponent), np.float32)


def check_sample(got, d, k):
    idx, st, act, ret, nx, nt, wt = [np.asarray(x) for x in got]
    assert np.array_equal(idx, d["s_idx"][k]), k
    assert np.array_equal(st, d["s_states"][k]) and np.array_equal(nx, d["s_next"][k]), k
    assert np.array_equal(act, d["s_actions"][k]) and np.array_equal(nt, d["s_nonterm"][k]), k
    want_r = d["s_returns"][k]
    assert np.all(np.abs(ret - want_r) <= 1e-6 * (1 + np.abs(want_r))), (k, ret, want_r)
    if float(d["beta"][k]) == 1.0:
        assert np.array_equal(wt, d["s_weights"][k]), k
    else:
        assert np.all(np.abs(wt - d["s_weights"][k]) <= 4e-7 * d["s_weights"][k]), (k, wt, d["s_weights"][k])


def run_golden(d, impl, rounds_limit=None):
    """``impl``: append(state, action, reward, done, valid), sample(batch, u, beta) -> 7 arrays,
    update(tree_idx, cpu_loss, priority_exponent), snapshot() -> dict(tree, index, full, max, t)."""
    rounds = {int(s): k for k, s in enumerate(d["round_step"])}
    batch, done_rounds = int(d["batch"]), 0
    for t in range(len(d["state"])):
        impl.append(d["state"][t], d["action"][t], d["reward"][t], d["done"][t], d["valid"][t])
        s = impl.snapshot()
        assert np.array_equal(s["tree"], d["tree"][t]), t
        for key in ("index", "full", "max", "t"):
            assert np.array_equal(np.asarray(s[key]).astype(d[key].dtype), d[key][t]), (t, key)
        k = rounds.get(t + 1)
        if k is None:
            continue
        got = impl.sample(batch, d["u"][k], float(d["beta"][k]))
        check_sample(got, d, k)
        impl.update(got[0], d["loss"][k], float(d["priority_exponent"]))
        s = impl.snapshot()
        assert np.array_equal(s["tree"], d["u_tree"][k]) and np.array_equal(s["max"], d["u_max"][k]), k
        done_rounds += 1
        if rounds_limit is not None and done_rounds >= rounds_limit:
            break
    return done_rounds


class PortImpl(object):
    def __init__(self, d):
        from oracle.replay_port import ReplayPort
        self.p = ReplayPort(int(d["N"]), int(d["C"]), int(d["L"]), float(d["discount"]), int(d["n"]))

    def append(self, *a):
        self.p.append(*a)

    def sample(self, batch, u, beta):
        self.p.priority_weight = beta
        return self.p.sample(batch, u)

    def update(self, idx, loss, exponent):
        self.p.update_priorities(idx, powered(loss, exponent))

    def snapshot(self):
        return {"tree": self.p.tree, "index": self.p.index, "full": self.p.full, "max": self.p.max, "t": self.p.t}


@pytest.mark.parametrize("name", GOLDENS)
def test_port_reproduces_reference_golden(name):
    d = load_golden(name)
    assert run_golden(d, PortImpl(d)) == len(d["round_step"])


def _generator():
    spec = importlib.util.spec_from_file_location("make_replay_golden", os.path.join(GOLDEN, "make_replay_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("cfg", [
    dict(N=5, C=20, L=6, n=3, batch=10, steps=160, learn_start=25, freq=2, beta0=0.5, beta_inc=0.01, seed=11),
    dict(N=2, C=24, L=4, n=1, batch=4, steps=120, learn_start=30, freq=3, beta0=1.0, beta_inc=0.0, seed=12),
    dict(N=3, C=13, L=5, n=2, batch=3, steps=140, learn_start=20, freq=2, beta0=1.0, beta_inc=0.0, seed=13)])
def test_port_matches_verbatim_memory_py(cfg):
    from oracle import ref_loader
    if not os.path.isfile(os.path.join(ref_loader.REFERENCE_ROOT, "memory.py")):
        pytest.skip("reference tree not mounted")
    gen = _generator()
    d = gen.record(cfg)
    d["discount"], d["priority_exponent"] = np.float64(0.99), np.float64(0.5)
    assert run_golden(d, PortImpl(d)) > 10
