"""Golden traces of the reference's prioritized replay memory: tests/golden/replay_*.npz.

Runs the UNMODIFIED ``memory.py`` of the reference (loaded from where it lies through ``oracle/ref_loader.py``; needs
the reference tree, numpy and torch) with N ``ReplayMemory`` objects driven the way ``trainer.py:184-186`` appends
(only bins whose ``Valid`` is set) and ``agent.py:68-124`` samples and updates (``batch // N`` draws per memory, the
CPU loss to ``update_priorities``).  ``np.random.uniform`` is routed to a recorded table ``u[row, attempt]`` so that the
device kernels can be compared exactly.  Recorded after every append and every update: the sum trees, index, full,
max and t of every memory; per learning round: the table, beta, the sample outputs and the losses.

    python tests/golden/make_replay_golden.py
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

# name: (N, C, obs_len, n, batch, steps, learn_start, replay_frequency, beta0, beta_increase, seed)
CONFIGS = {
    "replay_c24": dict(N=4, C=24, L=7, n=3, batch=8, steps=300, learn_start=20, freq=4, beta0=1.0, beta_inc=0.0, seed=1),
    "replay_c16": dict(N=3, C=16, L=9, n=3, batch=6, steps=260, learn_start=30, freq=3, beta0=0.4, beta_inc=0.004, seed=2),
}
ATTEMPTS = 64


def load_memory_module():
    from oracle import ref_loader
    if not os.path.isfile(os.path.join(ref_loader.REFERENCE_ROOT, "memory.py")):
        raise RuntimeError("reference memory.py not found under %s" % ref_loader.REFERENCE_ROOT)
    return ref_loader._load("irbpp_ref_memory", "memory.py")


class _TableUniform(object):
    """Stand-in for ``np.random.uniform(low, high)``: NumPy's ``low + (high - low) * u`` in float64 with ``u`` taken
    from ``table[row, attempt]``; ``row`` is set per draw by the wrapped ``_get_sample_from_segment``."""

    def __init__(self):
        self.table, self.row, self.attempt, self.max_attempt = None, 0, 0, 0

    def __call__(self, low, high):
        lo, hi = float(low), float(high)
        u = float(self.table[self.row, self.attempt])
        self.attempt += 1
        self.max_attempt = max(self.max_attempt, self.attempt)
        return lo + (hi - lo) * u


def record(cfg, memory_module=None):
    """Run one trace through the verbatim memory.py; returns the arrays of the golden file."""
    mm = memory_module or load_memory_module()
    N, C, L, n, batch = cfg["N"], cfg["C"], cfg["L"], cfg["n"], cfg["batch"]
    per = batch // N
    args = SimpleNamespace(distributed=False, device="cpu", discount=0.99, multi_step=n, priority_weight=cfg["beta0"],
                           priority_exponent=0.5)
    mems = [mm.ReplayMemory(args, C, L) for _ in range(N)]
    uni = _TableUniform()
    for i, m in enumerate(mems):
        orig = m._get_sample_from_segment

        def wrapped(segment, j, _orig=orig, _i=i):
            uni.row, uni.attempt = _i * per + j, 0
            return _orig(segment, j)
        m._get_sample_from_segment = wrapped
    rng = np.random.default_rng(cfg["seed"])
    rec = {k: [] for k in ("state", "action", "reward", "done", "valid", "tree", "index", "full", "max", "t",
                           "round_step", "u", "beta", "s_idx", "s_states", "s_actions", "s_returns", "s_next", "s_nonterm",
                           "s_weights", "loss", "u_tree", "u_max")}

    def bookkeeping():
        return (np.stack([m.transitions.sum_tree.numpy().copy() for m in mems]),
                np.array([m.transitions.index.value for m in mems], np.int64),
                np.array([bool(m.transitions.full.value) for m in mems]),
                np.array([float(m.transitions.max) for m in mems], np.float32),
                np.array([m.t for m in mems], np.int64))
    real_uniform = np.random.uniform
    np.random.uniform = uni
    try:
        for T in range(1, cfg["steps"] + 1):
            state = torch.from_numpy(rng.normal(size=(N, L)).astype(np.float32))
            action = torch.from_numpy(rng.integers(0, 500, size=N).astype(np.int64))
            reward = torch.from_numpy(rng.uniform(-2, 12, size=(N, 1)).astype(np.float32))
            done = rng.random(N) < 0.15
            valid = rng.random(N) < 0.9
            for i in range(N):                                                  # trainer.py:184-186
                if valid[i]:
                    mems[i].append(state[i], action[i], reward[i], done[i])
            for k, v in (("state", state.numpy()), ("action", action.numpy()), ("reward", reward.numpy()[:, 0]),
                         ("done", done), ("valid", valid)):
                rec[k].append(v)
            for k, v in zip(("tree", "index", "full", "max", "t"), bookkeeping()):
                rec[k].append(v)
            if T >= cfg["learn_start"]:
                for m in mems:                                                  # trainer.py:196-197
                    m.priority_weight = min(m.priority_weight + cfg["beta_inc"], 1)
                if T % cfg["freq"] == 0:
                    uni.table = rng.random((N * per, ATTEMPTS))
                    outs = [m.sample(per) for m in mems]                        # agent.py:72-75
                    idxs = [o[0] for o in outs]
                    rec["round_step"].append(T)
                    rec["u"].append(uni.table)
                    rec["beta"].append(mems[0].priority_weight)
                    rec["s_idx"].append(np.concatenate([np.asarray(ix, np.int64) + i * (2 * C - 1) for i, ix in enumerate(idxs)]))
                    for k, j in (("s_states", 1), ("s_actions", 2), ("s_returns", 3), ("s_next", 4), ("s_nonterm", 5),
                                 ("s_weights", 6)):
                        rec[k].append(torch.cat([o[j] for o in outs], 0).numpy())
                    loss = torch.from_numpy(rng.uniform(0.01, 4.0, size=N * per).astype(np.float32))
                    for i in range(N):                                          # agent.py:123-124
                        mems[i].update_priorities(idxs[i], loss[i * per:(i + 1) * per].detach().cpu())
                    rec["loss"].append(loss.numpy())
                    tr, _, _, mx, _ = bookkeeping()
                    rec["u_tree"].append(tr)
                    rec["u_max"].append(mx)
    finally:
        np.random.uniform = real_uniform
    assert uni.max_attempt < ATTEMPTS
    out = {k: np.stack(v) for k, v in rec.items()}
    out.update({k: np.int64(cfg[k]) for k in ("N", "C", "L", "n", "batch")})
    out["discount"], out["priority_exponent"] = np.float64(0.99), np.float64(0.5)
    out["max_attempts_used"] = np.int64(uni.max_attempt)
    return out


def main():
    mm = load_memory_module()
    for name, cfg in CONFIGS.items():
        d = record(cfg, mm)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **d)
        print(name, os.path.getsize(path), "bytes;", len(d["round_step"]), "rounds; max attempts", int(d["max_attempts_used"]))


if __name__ == "__main__":
    main()
