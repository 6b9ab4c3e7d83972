"""The CUDA kernels of irbpp_b200/csrc/ executed on host threads (tests/host_harness/cuda_emu.h: one
thread per CUDA thread of one block at a time, real barriers, warp collectives as slot exchanges) and
compared with the golden episodes of the unmodified reference.  TEST INFRASTRUCTURE ONLY: it checks the
kernel-level logic (barrier structure, hand-overs, warp collectives) where no GPU exists; the emulated
library exports ``emu_irbpp_*`` symbols, which ``irbpp_b200._lib`` cannot bind, and lives in a temp dir.
The parity tests proper are the ``-m gpu`` tests, which run the real kernels on a B200."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import lib_from_fixture, load_golden
from irbpp_b200 import _lib

pytestmark = pytest.mark.timeout(900)          # a deadlocked emulated barrier must not hang the suite

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "irbpp_b200", "csrc")
HARNESS = os.path.join(ROOT, "tests", "host_harness")


def _host_source(text):
    """Storage qualifiers and launch syntax of the device source rewritten for g++."""
    # dynamic shared memory: a pointer to the launch's heap block (sized as requested) instead of an unsized array
    text = re.sub(r"extern __shared__ __align__\(\d+\) ([\w ]+?) (\w+)\[\];",
                  r"\1* \2 = reinterpret_cast<\1*>(cuda_emu::dyn_smem);", text)
    text = re.sub(r"__shared__ __align__\((\d+)\)", r"alignas(\1) static", text)
    text = text.replace("extern __shared__", "extern").replace("__shared__", "static")
    text = re.sub(r'asm volatile\("(griddepcontrol|prefetch)[^\n]*\);', ";", text)
    text = text.replace("#include <cuda_runtime.h>", '#include "cuda_emu.h"')
    text = re.sub(r"(\w+)<<<([^;]*?)>>>\(", lambda m: "CUDA_EMU_LAUNCH(%s, %s, " % (m.group(1), m.group(2)), text, flags=re.S)
    return text


def build_emulated(tmp, defs=()):
    names = re.findall(r"\b(irbpp_[a-z_]+)\(", open(os.path.join(ROOT, "include", "irbpp.h")).read())
    csrc = os.path.join(tmp, "pkg", "csrc")               # irbpp.cu includes "../../include/irbpp.h"
    os.makedirs(csrc, exist_ok=True)
    os.makedirs(os.path.join(tmp, "include"), exist_ok=True)
    for fn in os.listdir(CSRC):
        with open(os.path.join(csrc, fn), "w") as f:
            f.write(_host_source(open(os.path.join(CSRC, fn)).read()))
    for src, dst in ((os.path.join(ROOT, "include", "irbpp.h"), os.path.join(tmp, "include", "irbpp.h")),
                     (os.path.join(HARNESS, "cuda_emu.h"), os.path.join(csrc, "cuda_emu.h"))):
        open(dst, "w").write(open(src).read())
    main = os.path.join(csrc, "emu_main.cpp")
    with open(main, "w") as f:
        f.write('#include "cuda_emu.h"\n#include "irbpp.cu"\n')
    # the C-ABI entry points get emu_ names: this library can never stand in for the product's
    rename = ["-D%s=emu_%s" % (n, n) for n in sorted(set(names))]
    out = os.path.join(tmp, "libirbpp_emulated.so")
    cmd = ["g++", "-O1", "-std=c++17", "-pthread", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared", "-fPIC",
           "-I", csrc] + rename + list(defs) + ["-o", out, main]
    subprocess.run(cmd, check=True)
    return ctypes.CDLL(out)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    return build_emulated(str(tmp_path_factory.mktemp("emu")))


class EmuEnv(object):
    """The C ABI of include/irbpp.h driven with NumPy buffers (device == host under the emulation)."""

    def __init__(self, lib, library, sequences, selected_action=500, buffer_size=1):
        self.lib, self.n = lib, len(sequences)
        cfg = _lib.IrbppConfig(self.n, library.num_rotations, selected_action, buffer_size,
                               (ctypes.c_double * 3)(0.32, 0.32, 0.30), 0.02, 0.01, 0.01, 0, 0)
        self.h = ctypes.c_void_p()
        assert lib.emu_irbpp_create(ctypes.byref(cfg), ctypes.byref(self.h)) == 0
        dims, ext, vol, maps, offsets = library.flat()
        P = ctypes.c_void_p
        assert lib.emu_irbpp_load_shapes(self.h, library.num_shapes, library.num_rotations, P(dims.ctypes.data),
                                         P(ext.ctypes.data), P(vol.ctypes.data), P(maps.ctypes.data),
                                         P(offsets.ctypes.data), ctypes.c_int64(maps.size)) == 0
        seqs = np.ascontiguousarray(sequences, dtype=np.int32)
        assert lib.emu_irbpp_set_sequences(self.h, P(seqs.ctypes.data), seqs.shape[1]) == 0
        o, l, k = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        lib.emu_irbpp_obs_len(self.h, ctypes.byref(o), ctypes.byref(l), ctypes.byref(k))
        self.obs_len, self.loc_len = o.value, l.value

    def reset(self):
        obs = np.zeros((self.n, self.obs_len), np.float32)
        assert self.lib.emu_irbpp_reset(self.h, None, ctypes.c_void_p(obs.ctypes.data), None) == 0
        return obs

    def step(self, actions):
        acts = np.ascontiguousarray(actions, dtype=np.int64)
        obs = np.zeros((self.n, self.obs_len), np.float32)
        assert self.lib.emu_irbpp_step_async(self.h, ctypes.c_void_p(acts.ctypes.data), 0, ctypes.c_void_p(obs.ctypes.data), None) == 0
        res = self.result = _lib.IrbppStepResult()
        assert self.lib.emu_irbpp_step_wait(self.h, ctypes.byref(res)) == 0, self.lib.emu_irbpp_last_error(self.h)
        view = lambda p, ct, dt: np.frombuffer((ct * self.n).from_address(p), dtype=dt).copy()
        return (obs, view(res.reward, ctypes.c_float, np.float32), view(res.done, ctypes.c_uint8, np.bool_),
                view(res.counter, ctypes.c_int32, np.int32), view(res.ratio, ctypes.c_double, np.float64))

    def get_action_candidates(self, order):
        order = np.ascontiguousarray(order, dtype=np.int64)
        loc = np.zeros((self.n, self.loc_len), np.float32)
        assert self.lib.emu_irbpp_get_action_candidates(self.h, ctypes.c_void_p(order.ctypes.data), 0,
                                                        ctypes.c_void_p(loc.ctypes.data), None) == 0
        return loc

    def get_all_possible_observation(self, k):
        out = np.zeros((self.n, k * self.loc_len), np.float32)
        assert self.lib.emu_irbpp_get_all_possible_observation(self.h, ctypes.c_void_p(out.ctypes.data), None) == 0
        return out

    def close(self):
        self.lib.emu_irbpp_destroy(self.h)


def _replay(lib, name, steps):
    d = load_golden(name)
    env = EmuEnv(lib, lib_from_fixture(d), d["sequences"], selected_action=int(d["selectedAction"]),
                 buffer_size=int(d["bufferSize"]))
    obs = env.reset()
    assert np.array_equal(obs, d["obs"][0].astype(np.float32))
    for t in range(min(steps, len(d["actions"]))):
        if int(d["bufferSize"]) > 1:
            assert np.array_equal(env.get_action_candidates(d["order"][t]), d["loc_obs"][t].astype(np.float32)), t
        obs, rew, done, counter, ratio = env.step(d["actions"][t])
        assert np.array_equal(obs, d["obs"][t + 1].astype(np.float32)), (name, t)
        assert np.array_equal(rew, d["reward"][t].astype(np.float32)) and np.array_equal(done, d["done"][t])
        for i in np.nonzero(done)[0]:
            assert counter[i] == d["counter"][t][i] and ratio[i] == d["ratio"][t][i]
    env.close()


@pytest.mark.parametrize("name,steps", [("episode_blockout", 12), ("episode_cube", 14), ("episode_irregular", 5),
                                        ("episode_truncate", 6), ("episode_buffered", 6), ("episode_buffered10", 5), ("episode_rot24", 3)])
def test_emulated_kernels_replay_reference_episodes(emu, name, steps):
    _replay(emu, name, steps)


def test_emulated_result_block_layout_matches_python_table(emu):
    """The pointers irbpp_step_wait returns sit at the offsets of _lib.RESULT_FIELDS in a block of 31 bytes per bin."""
    from irbpp_b200 import shapes
    n = 5
    lib = shapes.make_blockout_library(8, seed=1)
    env = EmuEnv(emu, lib, shapes.make_sequences(n, 8, lib.num_shapes, seed=0))
    env.reset()
    env.step(np.zeros(n, np.int64))
    offsets, size = _lib.result_offsets(n)
    res = env.result
    assert {k: getattr(res, k) - res.ratio for k in offsets} == offsets and size == 31 * n
    env.close()




@pytest.mark.parametrize("sel", [24, 96])
def test_emulated_truncation_ranking_small_tables(emu, sel):
    """Tables much smaller than the candidate set (irregular shapes, R = 8): every step truncates, the kept rows
    mix feasible and infeasible candidates and equal heights -- the bucketed ranking of phase D against the
    oracle's stable argsort (binPhy.py:209-212), random feasible-first actions, episodes restarting."""
    from irbpp_b200 import shapes
    from oracle.oracle_env import OracleConfig, OracleEnv
    lib = shapes.make_irregular_library(10, seed=5, num_rotations=8)
    n = 5
    seqs = shapes.make_sequences(n, 48, lib.num_shapes, seed=3)
    env = EmuEnv(emu, lib, seqs, selected_action=sel)
    cfg = OracleConfig(ZRotNum=8, selectedAction=sel)
    oracles = [OracleEnv(cfg, lib, seqs[i]) for i in range(n)]
    obs = env.reset()
    want = np.stack([o.reset() for o in oracles]).astype(np.float32)
    assert np.array_equal(obs, want)
    rng = np.random.default_rng(sel)
    n_trunc = 0
    for t in range(14):
        valid = obs[:, :sel * 5].reshape(n, sel, 5)[:, :, 4] == 1
        n_trunc += int((obs[:, :sel * 5].reshape(n, sel, 5)[:, sel - 1, :3].sum(1) > 0).sum())
        acts = np.argmax(rng.random((n, sel)) + valid, axis=1)
        obs, rew, done, counter, ratio = env.step(acts)
        for i in range(n):
            o, r, dn, info = oracles[i].step(int(acts[i]))
            if dn:
                o = oracles[i].reset()
            want[i] = o
            assert np.float32(r) == rew[i] and bool(dn) == bool(done[i])
        assert np.array_equal(obs, want), (sel, t)
    assert n_trunc > 0
    env.close()


def test_emulated_fused_all_possible_observation(emu):
    """get_all_possible_observation as ONE scan + ONE candidates launch over (bin, buffer slot) pairs, k = 10, vs
    the oracle's per-item loop (binPhy.py:171-180); then the protocol goes on (candidate state of slot k-1)."""
    from irbpp_b200 import shapes
    from oracle.oracle_env import OracleConfig, OracleVecEnv
    lib = shapes.make_blockout_library(12, seed=41)
    n, k = 3, 10
    seqs = shapes.make_sequences(n, 40, lib.num_shapes, seed=9)
    ora = OracleVecEnv(OracleConfig(ZRotNum=4, bufferSize=k), lib, seqs)
    env = EmuEnv(emu, lib, seqs, buffer_size=k)
    assert np.array_equal(env.reset(), ora.reset().astype(np.float32))
    rng = np.random.default_rng(2)
    for t in range(3):
        want = np.stack([e.get_all_possible_observation() for e in ora.envs])
        assert np.array_equal(env.get_all_possible_observation(k), want.astype(np.float32)), t
        order = rng.integers(0, k, size=n)
        loc_o = np.stack(ora.get_action_candidates(order))
        assert np.array_equal(env.get_action_candidates(order), loc_o.astype(np.float32)), t
        acts = np.zeros(n, dtype=np.int64)
        for i in range(n):
            valid = np.nonzero(loc_o[i][:2500].reshape(500, 5)[:, 4] == 1)[0]
            acts[i] = int(rng.choice(valid)) if len(valid) else 0
        assert np.array_equal(env.step(acts)[0], ora.step(acts)[0].astype(np.float32)), t
    env.close()


def _P(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.parametrize("tag", ["blockout", "irregular", "cube"])
def test_emulated_scan_matches_reference_golden(emu, tag):
    """Verbatim Space.get_possible_position outputs (scan goldens) through irbpp_debug_scan."""
    d = load_golden("scan_" + tag)
    lib = lib_from_fixture(d)
    n, R = len(d["item_ids"]), lib.num_rotations
    env = EmuEnv(emu, lib, np.zeros((n, 8), np.int32))
    hm = np.ascontiguousarray(d["heightmaps"], dtype=np.float64)
    assert emu.emu_irbpp_debug_set_heightmap(env.h, _P(hm)) == 0
    items = np.ascontiguousarray(d["item_ids"], dtype=np.int32)
    pz, pv, mk = np.zeros((n, R, 16, 16)), np.zeros((n, R, 16, 16)), np.zeros((n, R, 16, 16))
    cand, nh = np.zeros((n, 500, 5)), np.zeros(n, np.int32)
    assert emu.emu_irbpp_debug_scan(env.h, _P(items), _P(pz), _P(pv), _P(mk), _P(cand), _P(nh)) == 0
    assert np.array_equal(pz, d["posZmap"]) and np.array_equal(pv, d["posZValid"]) and np.array_equal(mk, d["naiveMask"])
    env.close()


def test_emulated_hull_actions_match_reference_golden(emu):
    """Verbatim cvTools.getConvexHullActions outputs (hull goldens) through irbpp_debug_hulls."""
    from irbpp_b200 import shapes
    d = load_golden("hulls")
    n = 64                                                   # the first 64 of the 160 cases (emulation speed)
    env = EmuEnv(emu, shapes.make_cube_library(seed=1, num_rotations=1, num_shapes=4), np.zeros((n, 8), np.int32),
                 selected_action=256)
    pv = np.ascontiguousarray(d["posZValid"][:n, None], dtype=np.float64)
    mk = np.ascontiguousarray(d["mask"][:n, None], dtype=np.float64)
    cand, nh = np.zeros((n, 256, 5)), np.zeros(n, np.int32)
    assert emu.emu_irbpp_debug_hulls(env.h, _P(pv), _P(mk), _P(cand), _P(nh)) == 0
    off = 0
    for k in range(n):
        c = int(d["counts"][k])
        assert nh[k] == c, k
        if c:
            assert np.array_equal(cand[k, :c], d["rows"][off:off + c]), k
        off += c
    env.close()


def test_emulated_heuristics_match_reference_golden(emu):
    """Verbatim Space.get_heuristic_action (4 scores x 4 directions) and the pose step, first steps of the
    irregular heuristic episode."""
    d = load_golden("heuristic_irregular")
    lib = lib_from_fixture(d)
    env = EmuEnv(emu, lib, d["sequences"])
    n = env.n
    assert np.array_equal(env.reset(), d["obs"][0])
    for t in range(4):
        for mi in range(4):
            for k in range(4):
                poses, index = np.zeros((n, 3), np.int32), np.zeros(n, np.int64)
                assert emu.emu_irbpp_heuristic_actions(env.h, mi, k, _P(poses), _P(index), 0, None) == 0
                assert np.array_equal(poses, d["poses"][t, mi, k]) and np.array_equal(index, d["index"][t, mi, k]), (t, mi, k)
        acts = np.ascontiguousarray(d["actions"][t], dtype=np.int64)
        obs = np.zeros((n, env.obs_len), np.float32)
        assert emu.emu_irbpp_step_poses_async(env.h, _P(acts), 0, _P(obs), None) == 0
        assert emu.emu_irbpp_step_wait(env.h, None) == 0
        assert np.array_equal(obs, d["obs"][t + 1]), t
    env.close()


def test_emulated_24_rotations(emu):
    """R = 24: run-time sized scratch, > 1024 candidates per bin, exact bucketed ranking."""
    _replay(emu, "episode_rot24", 3)


def _kat_inputs():
    """The SURVEY section 4 known-answer maps (8 x 8) embedded in the 16 x 16 action grid, masked outside."""
    d = load_golden("kats")
    names = ["rect", "pixel", "hline", "L", "ring_island", "diag", "diag_squares", "twolevel"]
    pv = np.full((len(names), 1, 16, 16), 1e3)
    mk = np.zeros((len(names), 1, 16, 16))
    for i, k in enumerate(names):
        pv[i, 0, :8, :8] = d["kat_%s_posz" % k]
        mk[i, 0, :8, :8] = d["kat_%s_mask" % k]
    pv[mk == 0] = 1e3
    return d, names, pv, mk


def check_kats(run_hulls):
    """``run_hulls(posZValid[n,1,16,16], mask) -> (cand[n,sel,5], num_hull[n])``; shared with the GPU test."""
    from test_oracle_golden import SURVEY_KATS
    d, names, pv, mk = _kat_inputs()
    cand, nh = run_hulls(pv, mk)
    for i, k in enumerate(names[:-1]):
        rows = cand[i, :int(nh[i])]
        assert [[int(r[2]), int(r[1])] for r in rows] == SURVEY_KATS[k], k          # (col, row), np.unique order
        assert np.all(rows[:, 4] == 1) and np.all(rows[:, 3] == 0.05)
    assert cand[-1, :int(nh[-1])].tolist() == d["kat_twolevel_rows"].tolist()


def test_emulated_survey_known_answers(emu):
    from irbpp_b200 import shapes
    n = 8
    env = EmuEnv(emu, shapes.make_cube_library(seed=1, num_rotations=1, num_shapes=4), np.zeros((n, 8), np.int32),
                 selected_action=256)

    def run(pv, mk):
        cand, nh = np.zeros((n, 256, 5)), np.zeros(n, np.int32)
        pv, mk = np.ascontiguousarray(pv), np.ascontiguousarray(mk)
        assert emu.emu_irbpp_debug_hulls(env.h, _P(pv), _P(mk), _P(cand), _P(nh)) == 0
        return cand, nh
    check_kats(run)
    env.close()


def check_many_start_pixels(run_hulls):
    """Level sets with > 100 start pixels per image (isolated pixels, sparse noise): more micro-tasks in a
    round than the task table lists (the search fallback) and several batches per round; vs the oracle."""
    from oracle.oracle_env import convex_hull_actions
    rng = np.random.default_rng(5)
    n = 4
    pv = np.full((n, 1, 16, 16), 1e3)
    mk = np.zeros((n, 1, 16, 16))
    xs, ys = np.meshgrid(np.arange(16), np.arange(16), indexing="ij")
    # bins 0, 1: every pixel feasible, neighbours always on different levels -> four level images of 64
    # isolated pixels each (256 start pixels per bin, 512 in the CTA's round: beyond the 256-entry table)
    for i in (0, 1):
        mk[i, 0] = 1
        pv[i, 0] = 0.015 + 0.01 * ((xs % 2) + 2 * (ys % 2)) + 0.04 * i
    for i, pat in ((2, rng.random((16, 16)) < 0.35), (3, (xs % 2 == 0) & (ys % 2 == 0))):
        mk[i, 0][pat] = 1
        pv[i, 0][pat] = 0.03 * (i - 1)
    cand, nh = run_hulls(pv, mk)
    for i in range(n):
        want = convex_hull_actions(pv[i], mk[i], 0.01, "port")
        assert nh[i] == len(want) and np.array_equal(cand[i, :len(want)], want), i


def test_emulated_many_start_pixels(emu):
    from irbpp_b200 import shapes
    env = EmuEnv(emu, shapes.make_cube_library(seed=1, num_rotations=1, num_shapes=4), np.zeros((4, 8), np.int32),
                 selected_action=256)

    def run(pv, mk):
        cand, nh = np.zeros((4, 256, 5)), np.zeros(4, np.int32)
        pv, mk = np.ascontiguousarray(pv), np.ascontiguousarray(mk)
        assert emu.emu_irbpp_debug_hulls(env.h, _P(pv), _P(mk), _P(cand), _P(nh)) == 0
        return cand, nh
    check_many_start_pixels(run)
    env.close()




def test_emulated_point_cloud_features_match_torch_fp32(emu):
    """SURVEY.md 8(f)3: sampled clouds and the fused shapeEncoder + max (csrc/irbpp_pointnet.cuh) run on host threads
    against the reference's own formulation in torch float32 (model.py:328-335).  Tolerance: the second layer sums
    128 products in a different order than torch's GEMM (and with FMA): |diff| <= 1e-5 * (1 + |want|)."""
    import torch
    from irbpp_b200.pointnet import pn_indices
    rng = np.random.default_rng(3)
    S, Pn, n_pts, B = 5, 300, 70, 9                     # 70 points: a full 64-point tile and a ragged one
    shape_array = rng.normal(0, 0.1, size=(S, Pn, 3)).astype(np.float32)
    ids = rng.integers(0, S, size=B).astype(np.int32)
    obs = np.zeros((B, 2500 + 9 + 1024), np.float32); obs[:, 2500] = ids
    enc = torch.nn.Sequential(torch.nn.Linear(3, 128), torch.nn.LeakyReLU(), torch.nn.Linear(128, 128), torch.nn.LeakyReLU())
    W1, b1, W2, b2 = [np.ascontiguousarray(t.detach().numpy()) for t in (enc[0].weight, enc[0].bias, enc[2].weight, enc[2].bias)]
    seed, counter = 77, 5
    idx = pn_indices(seed, counter, n_pts, Pn)
    want_cloud = shape_array[ids][:, idx]                                                  # model.py:330-332
    with torch.no_grad():
        want_feat = torch.max(enc(torch.from_numpy(want_cloud)), dim=1)[0].numpy()         # model.py:334-335
    cloud = np.zeros((B, n_pts, 3), np.float32); got_idx = np.zeros(n_pts, np.int32)
    U64 = ctypes.c_uint64
    assert emu.emu_irbpp_sample_point_clouds(_P(shape_array), S, Pn, _P(obs), ctypes.c_int64(obs.shape[1]), 2500, None, B, U64(seed),
                                             U64(counter), n_pts, _P(cloud), _P(got_idx), None) == 0
    assert np.array_equal(got_idx, idx) and np.array_equal(cloud, want_cloud)
    keys = np.zeros(S * 128, np.int32); feat = np.zeros((B, 128), np.float32)
    for use_ids in (False, True):
        assert emu.emu_irbpp_shape_features(_P(shape_array), S, Pn, None if use_ids else _P(obs), ctypes.c_int64(obs.shape[1]), 2500,
                                            _P(ids) if use_ids else None, B, U64(seed), U64(counter), n_pts, _P(W1), _P(b1), _P(W2),
                                            _P(b2), ctypes.c_float(0.01), _P(keys), _P(feat), None) == 0
        assert np.all(np.abs(feat - want_feat) <= 1e-5 * (1 + np.abs(want_feat))), np.abs(feat - want_feat).max()


def test_emulated_packed_observations_round_trip(emu):
    """csrc/irbpp_pack.cuh: the compact form the rollout gather sends must expand to the very same float32 observation
    (every golden BlockOut / irregular / truncation observation; ragged selectedAction)."""
    for name in ("episode_blockout", "episode_irregular", "episode_truncate"):
        d = load_golden(name)
        sel = int(d["selectedAction"])
        obs = np.ascontiguousarray(d["obs"].reshape(-1, d["obs"].shape[-1]).astype(np.float32))
        n, width = obs.shape
        nb = emu.emu_irbpp_packed_obs_bytes(sel)
        assert nb % 16 == 0 and nb < width * 4
        packed = np.zeros((n, nb), np.uint8)
        assert emu.emu_irbpp_pack_observations(_P(obs), ctypes.c_int64(width), sel, n, _P(packed), None) == 0
        back = np.full((n, width), -7.0, np.float32)
        assert emu.emu_irbpp_unpack_observations(_P(packed), sel, n, _P(back), ctypes.c_int64(width), None) == 0
        assert np.array_equal(back, obs), name
