"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container (needs ``/root/reference`` and cv2):

    python tests/golden/make_golden.py

It executes reference ``environment/physics0/space.py`` (``Space.get_possible_position``,
``space.py:98-129``) and ``environment/physics0/cvTools.py`` (``getConvexHullActions`` /
``convexHulls``, ``cvTools.py:61-103``) verbatim via ``oracle/ref_loader.py`` and stores their
outputs.  Episode fixtures drive those verbatim functions through the restated ``binPhy`` glue of
``oracle/oracle_env.py`` (``RefGeometry`` backend) -- the glue cannot run verbatim (gym / pybullet).
The GPU box has no reference tree; tests there read only the ``.npz`` files written here.
"""
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from irbpp_b200 import shapes  # noqa: E402
from oracle import ref_loader  # noqa: E402
from oracle.oracle_env import HEURISTICS, OracleConfig, OracleVecEnv, RefGeometry  # noqa: E402


def savez(path, **arrays):
    """``np.savez_compressed`` at zlib's highest level: keeps every fixture under 1 MB (episode_irregular.npz is just
    over at the default level).  ``np.load`` reads it like any .npz."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED, compresslevel=9) as z:
        for name, a in arrays.items():
            with z.open(name + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


def lib_arrays(lib, prefix="lib_"):
    dims, ext, vol, maps, offsets = lib.flat()
    return {prefix + "dims": dims, prefix + "ext": ext, prefix + "vol": vol, prefix + "maps": maps,
            prefix + "offsets": offsets, prefix + "res": np.array([lib.resolutionH, lib.resolutionAct])}


def random_heightmap(rng, kind):
    hm = np.zeros((32, 32))
    if kind == 0:
        return hm
    if kind == 1:  # stacked boxes on a 0.04 grid (BlockOut-like terrain)
        for _ in range(int(rng.integers(1, 12))):
            x0, y0 = rng.integers(0, 8, size=2) * 4
            w, h = rng.integers(1, 4, size=2) * 4
            top = hm[x0:x0 + w, y0:y0 + h].max() + 0.04 * rng.integers(1, 3)
            hm[x0:x0 + w, y0:y0 + h] = min(top, 0.30)
        return hm
    if kind == 2:  # arbitrary float64 heights
        hm = rng.uniform(0, 0.3, size=(32, 32))
        hm[rng.random((32, 32)) < 0.3] = 0.0
        return hm
    # smooth bumps with float noise
    xs, ys = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    for _ in range(int(rng.integers(1, 5))):
        cx, cy = rng.uniform(0, 32, size=2)
        hm += rng.uniform(0.02, 0.1) * np.exp(-((xs - cx) ** 2 + (ys - cy) ** 2) / rng.uniform(10, 80))
    return np.minimum(hm, 0.3)


def gen_scan_cases(space_mod):
    out = {}
    for tag, lib, R in (("blockout", shapes.make_blockout_library(12, seed=11), 4),
                        ("irregular", shapes.make_irregular_library(12, seed=12), 8),
                        ("cube", shapes.make_cube_library(seed=13, num_shapes=12), 2)):
        cfg = OracleConfig(ZRotNum=R)
        rng = np.random.default_rng(100 + R)
        sp = space_mod.Space(cfg.bin_dimension, cfg.resolutionAct, cfg.resolutionH, False, R,
                             lib.shot_info(), [100, 100, 100])
        hms, ids, pz, pv, mk = [], [], [], [], []
        for case in range(24):
            hm = random_heightmap(rng, case % 4)
            item = int(rng.integers(0, lib.num_shapes))
            sp.heightmapC = hm
            meshes = [ref_loader.MeshStandIn(lib.extents[item, r]) for r in range(R)]
            mask = sp.get_possible_position(item, meshes, 500)
            hms.append(hm.copy()); ids.append(item)
            pz.append(sp.posZmap.copy()); pv.append(sp.posZValid.copy()); mk.append(mask.copy())
        d = lib_arrays(lib)
        d.update(R=np.array(R), heightmaps=np.array(hms), item_ids=np.array(ids), posZmap=np.array(pz),
                 posZValid=np.array(pv), naiveMask=np.array(mk))
        out[tag] = d
    return out


def gen_hull_cases(cv_mod):
    """Random [16,16] posZ / mask maps -> rows [rot,row,col,H,V] of the verbatim getConvexHullActions."""
    rng = np.random.default_rng(7)
    posz, masks, rows, counts = [], [], [], []
    for case in range(160):
        kind = case % 4
        if kind == 0:   # blocky levels
            lv = np.zeros((16, 16))
            for _ in range(int(rng.integers(1, 9))):
                x0, y0 = rng.integers(0, 15, size=2); w, h = rng.integers(1, 9, size=2)
                lv[x0:x0 + w, y0:y0 + h] = rng.integers(0, 8)
            pz = lv * 0.04
        elif kind == 1:  # noisy multiples of 0.01 (floor-divide hazards 0.03//0.01 == 2 ...)
            pz = rng.integers(0, 31, size=(16, 16)) * 0.01
        elif kind == 2:  # arbitrary floats incl. negatives
            pz = rng.uniform(-0.05, 0.3, size=(16, 16))
        else:            # few levels, big regions with holes
            pz = (rng.random((16, 16)) < 0.35) * 0.05 + (rng.random((16, 16)) < 0.2) * 0.02
        mask = (rng.random((16, 16)) > (0.1 if case % 8 < 6 else 0.6)).astype(np.float64)
        if case % 16 == 15:
            mask[:] = 0
        pv = np.where(mask == 1, pz, 1e3)
        res = cv_mod.getConvexHullActions(pv[None], mask[None], 0.01)
        posz.append(pv); masks.append(mask)
        if res is None:
            counts.append(0)
        else:
            counts.append(len(res)); rows.append(res)
    return dict(posZValid=np.array(posz), mask=np.array(masks), counts=np.array(counts),
                rows=np.concatenate(rows, axis=0))


def gen_kats(cv_mod):
    """Known-answer vectors of SURVEY.md section 4, re-derived from the verbatim reference."""
    def level_img(pix):
        pz = np.full((8, 8), 1e3); m = np.zeros((8, 8))
        for (r, c) in pix:
            pz[r, c] = 0.05; m[r, c] = 1
        return pz, m
    shapes_px = {
        "rect": [(r, c) for r in range(2, 5) for c in range(1, 6)],
        "pixel": [(3, 3)],
        "hline": [(3, c) for c in range(1, 6)],
        "L": [(r, c) for r in range(1, 6) for c in range(1, 6) if not (r >= 3 and c >= 3)],
        "ring_island": [(r, c) for r in range(7) for c in range(7) if not (2 <= r <= 4 and 2 <= c <= 4)] + [(3, 3)],
        "diag": [(i, i) for i in range(5)],
        "diag_squares": [(1, 1), (1, 2), (2, 1), (2, 2), (3, 3), (3, 4), (4, 3), (4, 4)],
    }
    out = {}
    for k, pix in shapes_px.items():
        pz, m = level_img(pix)
        hulls, V = cv_mod.convexHulls(pz, m, 0.01)
        out["kat_" + k + "_posz"] = pz
        out["kat_" + k + "_mask"] = m
        out["kat_" + k + "_hulls"] = np.asarray(hulls)
    pz = np.zeros((8, 8)); pz[:, :4] = 0.02; pz[:, 4:] = 0.05
    m = np.ones((8, 8)); m[0, 0] = 0
    pv = np.where(m == 1, pz, 1e3)
    out["kat_twolevel_posz"] = pv
    out["kat_twolevel_mask"] = m
    out["kat_twolevel_rows"] = cv_mod.getConvexHullActions(pv[None], m[None], 0.01)
    # NumPy float64 floor_divide at cvTools.py:78
    vals = np.concatenate([np.arange(0, 40) * 0.01, np.arange(0, 40) * 0.01 + 1e-12,
                           np.random.default_rng(3).uniform(-0.4, 0.4, size=400),
                           np.array([0.30000000000000004, -0.0, 1e3, -0.01, -0.03])])
    out["floordiv_in"] = vals
    out["floordiv_out"] = vals // 0.01
    return out


def gen_episode(tag, lib, R, n_envs, n_steps, seed, selectedAction=500, bufferSize=1):
    cfg = OracleConfig(ZRotNum=R, selectedAction=selectedAction, bufferSize=bufferSize)
    seqs = shapes.make_sequences(n_envs, 48, lib.num_shapes, seed=seed)
    vec = OracleVecEnv(cfg, lib, seqs, lambda c, l: RefGeometry(c, l))
    rng = np.random.default_rng(seed)
    obs = vec.reset()
    obs_log = [obs.copy()]
    loc_log, act_log, ord_log, rew_log, done_log, cnt_log, ratio_log, epr_log, epl_log = [], [], [], [], [], [], [], [], []
    for t in range(n_steps):
        if bufferSize > 1:
            order = rng.integers(0, bufferSize, size=n_envs)
            loc = np.stack(vec.get_action_candidates(order))
            ord_log.append(order); loc_log.append(loc.copy())
        else:
            loc = obs
        acts = []
        for i in range(n_envs):
            cand = loc[i][:selectedAction * 5].reshape(selectedAction, 5)
            valid = np.nonzero(cand[:, 4] == 1)[0]
            if t % 7 == 6:      # now and then take an arbitrary row (padding rows / invalid rows included)
                acts.append(int(rng.integers(0, selectedAction)))
            elif len(valid):
                acts.append(int(rng.choice(valid)))
            else:
                acts.append(0)
        obs, rew, done, infos = vec.step(acts)
        act_log.append(acts); obs_log.append(obs.copy()); rew_log.append(rew); done_log.append(done)
        cnt_log.append([inf.get("counter", -1) for inf in infos])
        ratio_log.append([inf.get("ratio", -1.0) for inf in infos])
        epr_log.append([inf["episode"]["r"] if "episode" in inf else 0.0 for inf in infos])
        epl_log.append([inf["episode"]["l"] if "episode" in inf else 0 for inf in infos])
    d = lib_arrays(lib)
    d.update(R=np.array(R), selectedAction=np.array(selectedAction), bufferSize=np.array(bufferSize),
             sequences=seqs, actions=np.array(act_log), obs=np.array(obs_log), reward=np.array(rew_log),
             done=np.array(done_log), counter=np.array(cnt_log), ratio=np.array(ratio_log),
             ep_r=np.array(epr_log), ep_l=np.array(epl_log))
    if bufferSize > 1:
        d.update(order=np.array(ord_log), loc_obs=np.array(loc_log))
    print(tag, "dones", int(np.sum(done_log)), "obs", d["obs"].shape)
    return d


def gen_heuristic_episode(tag, lib, R, n_envs, n_steps, seed):
    """Episodes driven by the reference's own placement heuristics: at every step the verbatim
    ``Space.get_heuristic_action`` (space.py:162-227) is evaluated for all four scores and all four
    flip directions on every bin (stored), then the bins are stepped with the pose of one
    (method, dirIdx), rotating over the sixteen combinations."""
    cfg = OracleConfig(ZRotNum=R)
    seqs = shapes.make_sequences(n_envs, 48, lib.num_shapes, seed=seed)
    vec = OracleVecEnv(cfg, lib, seqs, lambda c, l: RefGeometry(c, l))
    obs_log = [vec.reset().copy()]
    pose_log, index_log, act_log, rew_log, done_log = [], [], [], [], []
    for t in range(n_steps):
        poses = np.zeros((4, 4, n_envs, 3), np.int32)
        index = np.zeros((4, 4, n_envs), np.int64)
        for mi, m in enumerate(HEURISTICS):
            for d in range(4):
                poses[mi, d], index[mi, d] = vec.heuristic_actions(m, d)
        pose_log.append(poses); index_log.append(index)
        p = poses[t % 4, (t // 4) % 4]
        acts = (p[:, 0].astype(np.int64) * 16 + p[:, 1]) * 16 + p[:, 2]
        obs, rew, done, _ = vec.step(acts, poses=True)
        act_log.append(acts); obs_log.append(obs.copy()); rew_log.append(rew); done_log.append(done)
    d = lib_arrays(lib)
    d.update(R=np.array(R), sequences=seqs, poses=np.array(pose_log), index=np.array(index_log),
             actions=np.array(act_log), obs=np.array(obs_log).astype(np.float32),   # as VecPyTorch casts (envs.py:151,163)
             reward=np.array(rew_log), done=np.array(done_log))
    print(tag, "dones", int(np.sum(done_log)), "poses", d["poses"].shape, "not-a-candidate", int((d["index"] < 0).sum()))
    return d


def main():
    assert ref_loader.reference_available(), "needs /root/reference"
    _, space_mod, cv_mod = ref_loader.load_reference()
    # BASELINE.json configs[3]: buffered k = 10 (--hierachical).  Added in round 2; generated on its own
    # (--buffered10-only) so the round-1 fixtures stay byte-identical.
    if "--buffered10-only" in sys.argv or "--all" in sys.argv:
        d = gen_episode("buffered10", shapes.make_blockout_library(16, seed=8), 4, 3, 36, 29, bufferSize=10)
        savez(os.path.join(HERE, "episode_buffered10.npz"), **d)
        if "--buffered10-only" in sys.argv:
            return
    heur = {
        "heuristic_blockout": gen_heuristic_episode("heur-blockout", shapes.make_blockout_library(16, seed=6), 4, 3, 64, 26),
        "heuristic_irregular": gen_heuristic_episode("heur-irregular", shapes.make_irregular_library(12, seed=7), 8, 3, 48, 27),
    }
    for k, d in heur.items():
        savez(os.path.join(HERE, k + ".npz"), **d)
    if "--heuristics-only" in sys.argv:
        return
    for tag, d in gen_scan_cases(space_mod).items():
        savez(os.path.join(HERE, "scan_%s.npz" % tag), **d)
    savez(os.path.join(HERE, "hulls.npz"), **gen_hull_cases(cv_mod))
    savez(os.path.join(HERE, "kats.npz"), **gen_kats(cv_mod))
    eps = {
        "episode_blockout": gen_episode("blockout", shapes.make_blockout_library(16, seed=1), 4, 4, 70, 21),
        "episode_irregular": gen_episode("irregular", shapes.make_irregular_library(16, seed=2), 8, 4, 50, 22),
        "episode_cube": gen_episode("cube", shapes.make_cube_library(seed=3, num_shapes=24), 2, 3, 60, 23),
        # selectedAction small enough that the >selectedAction truncation path (binPhy.py:209-212) fires
        "episode_truncate": gen_episode("truncate", shapes.make_irregular_library(12, seed=4), 8, 3, 40, 24,
                                        selectedAction=40),
        "episode_buffered": gen_episode("buffered", shapes.make_blockout_library(16, seed=5), 4, 3, 50, 25,
                                        bufferSize=5),
        # 24 rotations (BASELINE.json config 3): > 1024 candidates per bin, truncation is the normal case
        "episode_rot24": gen_episode("rot24", shapes.make_irregular_library(8, seed=9, num_rotations=24), 24, 2, 24, 28),
    }
    for k, d in eps.items():
        savez(os.path.join(HERE, k + ".npz"), **d)
    import cv2
    with open(os.path.join(HERE, "PROVENANCE.txt"), "w") as f:
        f.write("generated by tests/golden/make_golden.py from the unmodified reference at %s\n" % ref_loader.REFERENCE_ROOT)
        f.write("numpy %s, cv2 %s\n" % (np.__version__, cv2.__version__))


if __name__ == "__main__":
    main()
