"""The reference's vectorised-environment surface, served by the CUDA library.

Mirrors (paths relative to the reference root):

* ``wrapper/vec_env.py:7-26``   ``AlreadySteppingError`` / ``NotSteppingError``
* ``wrapper/vec_env.py:29-108`` ``VecEnv``: ``reset / step_async / step_wait / step / close``
* ``wrapper/shmem_vec_env.py:20-118`` ``ShmemVecEnv``: ``waiting_step``, ``get_action_candidates``,
  ``reset_specific``; auto-reset on done (``:140-144``)
* ``envs.py:142-165`` ``VecPyTorch``: observations as ``torch.float32`` on ``device``, reward as a
  CPU ``float32 [N, 1]`` tensor, ``done`` a NumPy bool array, ``infos`` a sequence of dicts
* ``wrapper/monitor.py:58-75`` episode info ``info['episode'] = {'r', 'l', 't'}`` on done

so ``agent.py`` / ``trainer.py`` can drive ``GpuVecEnv`` where they drove
``VecPyTorch(ShmemVecEnv([...PackingGame...]))``.  All N bins live on one GPU; ``step`` is one kernel
launch (see ``csrc/irbpp_kernels.cuh``).  PyTorch is used for device memory and streams only.
"""
import ctypes
import time
import weakref
from abc import ABC, abstractmethod
from collections.abc import Sequence

import numpy as np

from . import _lib


class AlreadySteppingError(Exception):
    """step_async() called while a step is pending (reference wrapper/vec_env.py:7-16)."""

    def __init__(self):
        Exception.__init__(self, "already running an async step")


class NotSteppingError(Exception):
    """step_wait() called without a pending step (reference wrapper/vec_env.py:18-26)."""

    def __init__(self):
        Exception.__init__(self, "not running an async step")


class VecEnv(ABC):
    """Abstract asynchronous vectorised environment (reference wrapper/vec_env.py:29-108)."""
    closed = False

    def __init__(self, num_envs, observation_space, action_space):
        self.num_envs = num_envs
        self.observation_space = observation_space
        self.action_space = action_space

    @abstractmethod
    def reset(self):
        pass

    @abstractmethod
    def step_async(self, actions):
        pass

    @abstractmethod
    def step_wait(self):
        pass

    def close_extras(self):
        pass

    def close(self):
        if self.closed:
            return
        self.close_extras()
        self.closed = True

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    @property
    def unwrapped(self):
        return self


class Box(object):
    """Minimal stand-in for ``gym.spaces.Box`` (gym is not a dependency of this package): the
    attributes the reference's callers read (``shape``, ``low``, ``high``, ``dtype``;
    binPhy.py:100-101)."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.low = np.full(shape, low, dtype=dtype)
        self.high = np.full(shape, high, dtype=dtype)
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)

    def __repr__(self):
        return "Box(%s, %s, %s, %s)" % (self.low.min(), self.high.max(), self.shape, self.dtype)


class Discrete(object):
    """Stand-in for ``gym.spaces.Discrete`` (binPhy.py:102)."""

    def __init__(self, n):
        self.n = int(n)
        self.shape = ()
        self.dtype = np.dtype(np.int64)

    def __repr__(self):
        return "Discrete(%d)" % self.n


class LazyInfos(Sequence):
    """``infos`` of one step: behaves like the reference's tuple of N dicts but builds a dict only
    when indexed (at N = 4096 eagerly building them would dominate the step).  Holds this step's private
    copy of the library's result block; the typed views are cut out of it on first use."""

    _FIELDS = ("valid", "counter", "ratio", "ep_reward", "ep_len")

    def __init__(self, n, block, offsets, done, t_rel, borrowed=False):
        self._n, self._block, self._offsets, self._done, self._t = n, block, offsets, done, t_rel
        self._v = None
        self._borrowed = borrowed        # `block` is the library's pinned buffer: copied (detach) before it is reused

    def detach(self):
        """Take a private copy of the result block (called by the environment before the library reuses the
        buffer, if this object is still alive by then)."""
        if self._borrowed:
            self._block = self._block.copy()
            self._v = None
            self._borrowed = False

    def _views(self):
        if self._v is None:
            n, b, o = self._n, self._block, self._offsets
            self._v = {k: b[o[k]:o[k] + n * dt.itemsize].view(np.bool_ if k == "valid" else dt)
                       for k, dt in _lib.RESULT_FIELDS if k in self._FIELDS}
        return self._v

    def __len__(self):
        return self._n

    # -- batched views (SURVEY.md 8(f)2: consume a step without a Python loop over N dicts) --
    def valid_array(self):
        """``[info['Valid'] for info in infos]`` as one bool array (``trainer.py:167-169``)."""
        return self._views()["valid"][:self._n]

    def finished(self):
        """The episodes that ended in this step: ``(indices, episode_reward, ratio, counter, valid)`` arrays over
        the bins with ``done`` -- what ``trainer.py:170-178`` collects bin by bin (``episode_reward`` rounded to
        6 decimals like ``monitor.py:60``)."""
        v = self._views()
        idx = np.nonzero(self._done)[0]
        return (idx, np.round(v["ep_reward"][idx], 6), v["ratio"][idx], v["counter"][idx], v["valid"][idx])

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        v = self._views()
        info = {"Valid": bool(v["valid"][i])}
        if self._done[i]:
            # binPhy.py:306-309 and monitor.py:58-75 (round(eprew, 6) is Python's round, as there)
            info["counter"] = int(v["counter"][i])
            info["ratio"] = float(v["ratio"][i])
            info["episode"] = {"r": round(float(v["ep_reward"][i]), 6), "l": int(v["ep_len"][i]), "t": self._t}
        return info


def _as_host_i64(a, n, what):
    arr = np.ascontiguousarray(np.asarray(a).reshape(-1), dtype=np.int64)
    if arr.shape[0] != n:
        raise ValueError("%s: expected %d entries, got %d" % (what, n, arr.shape[0]))
    return arr


class GpuVecEnv(VecEnv):
    """N packing bins resident on one B200 behind the VecEnv contract.

    Parameters mirror what ``PackingGame.__init__`` reads from ``args`` (binPhy.py:25-49):
    ``library`` is a ``shapes.ShapeLibrary`` (the ``shotInfo`` / ``shapeDict`` / ``infoDict`` data),
    ``sequences`` the per-env item ids ``[N, L]`` (replayed modulo L; what the parity tests use), or ``None``
    for i.i.d. ids generated on the device from ``item_seed`` (the stand-in for ``RandomItemCreator``,
    IRcreator.py:26-33).  ``approx_legacy`` selects the point-to-line ``approxPolyDP`` rule believed to be
    what the reference's pinned OpenCV 4.4.0.46 computes (default: the 4.13 rule, the one testable here)."""

    def __init__(self, library, sequences, num_envs=None, device="cuda:0", selected_action=500, buffer_size=1,
                 bin_dimension=(0.32, 0.32, 0.30), resolution_act=0.02, resolution_h=0.01, resolution_z=0.01,
                 approx_legacy=False, item_seed=0):
        import torch
        self._torch = torch
        self._lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("GpuVecEnv needs a CUDA device; there is no CPU path")
        if sequences is None:
            # no explicit sequences: ids are drawn on the device, i.i.d. uniform from a counter-based generator
            # seeded with ``item_seed`` (RandomItemCreator's role, IRcreator.py:26-33; no period)
            if num_envs is None:
                raise ValueError("num_envs is required when no sequences are given")
        else:
            sequences = np.ascontiguousarray(sequences, dtype=np.int32)
            if num_envs is None:
                num_envs = sequences.shape[0]
            if sequences.shape[0] != num_envs:
                raise ValueError("sequences has %d rows for %d envs" % (sequences.shape[0], num_envs))
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        cfg = _lib.IrbppConfig()
        cfg.num_envs = num_envs
        cfg.num_rotations = library.num_rotations
        cfg.selected_action = selected_action
        cfg.buffer_size = buffer_size
        for i in range(3):
            cfg.bin_dimension[i] = float(bin_dimension[i])
        cfg.resolution_act, cfg.resolution_h, cfg.resolution_z = resolution_act, resolution_h, resolution_z
        cfg.device = idx
        cfg.approx_legacy = 1 if approx_legacy else 0
        handle = ctypes.c_void_p()
        rc = self._lib.irbpp_create(ctypes.byref(cfg), ctypes.byref(handle))
        _lib.check(self._lib, None, rc)
        self._h = handle
        self._cfg = cfg
        self.buffer_size = buffer_size
        self.selected_action = selected_action
        self.library = library
        dims, ext, vol, maps, offsets = library.flat()
        self._keep = (dims, ext, vol, maps, offsets, sequences)
        rc = self._lib.irbpp_load_shapes(self._h, library.num_shapes, library.num_rotations,
                                         dims.ctypes.data, ext.ctypes.data, vol.ctypes.data, maps.ctypes.data,
                                         offsets.ctypes.data, maps.size)
        self._check(rc)
        if sequences is None:
            rc = self._lib.irbpp_set_item_rng(self._h, int(item_seed) & 0xFFFFFFFFFFFFFFFF)
        else:
            rc = self._lib.irbpp_set_sequences(self._h, sequences.ctypes.data, sequences.shape[1])
        self._check(rc)
        o, l, k = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
        self._check(self._lib.irbpp_obs_len(self._h, ctypes.byref(o), ctypes.byref(l), ctypes.byref(k)))
        self.obs_len, self.loc_obs_len, self.order_obs_len = o.value, l.value, k.value
        obs_space = Box(0.0, float(bin_dimension[2]), (self.obs_len,))                 # binPhy.py:100-101
        act_space = Discrete(buffer_size if buffer_size > 1 else selected_action)     # binPhy.py:81-85,102
        VecEnv.__init__(self, num_envs, obs_space, act_space)
        self.waiting_step = False
        self._live_infos = []
        self._obs_pending = None
        self._spare_obs = None
        self._spare_stream = None
        self._dev_index = idx
        self._raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
        self._tstart = time.time()
        self._result = _lib.IrbppStepResult()

    # -- helpers --
    def _check(self, rc):
        _lib.check(self._lib, self._h, rc)

    def _stream(self):
        """Raw handle of torch's current stream on this device (queried per call: the caller may switch
        streams); the private fast accessor when this torch has it."""
        raw = self._raw_stream
        if raw is not None:
            return raw(self._dev_index)
        return self._torch.cuda.current_stream(self.device).cuda_stream

    def _new_obs(self, width):
        return self._torch.empty((self.num_envs, width), dtype=self._torch.float32, device=self.device)

    def _actions_arg(self, actions, what):
        """Host array / list (copied through pinned staging) or a CUDA int64 tensor (used in place)."""
        torch = self._torch
        if type(actions) is np.ndarray and actions.dtype == np.int64 and actions.ndim == 1 \
                and actions.shape[0] == self.num_envs and actions.flags.c_contiguous:
            return actions, actions.ctypes.data, 0              # the common case (trainer.py:165), no conversion
        if isinstance(actions, torch.Tensor):
            if actions.is_cuda:
                a = actions.reshape(-1).to(torch.int64).contiguous()
                if a.numel() != self.num_envs:
                    raise ValueError("%s: expected %d entries" % (what, self.num_envs))
                return a, a.data_ptr(), 1
            actions = actions.cpu().numpy()
        a = _as_host_i64(actions, self.num_envs, what)
        return a, a.ctypes.data, 0

    # -- VecEnv surface --
    def reset(self):
        """``envs.reset()`` -> float32 [N, obs_len] on device (envs.py:149-152)."""
        if self.waiting_step:                     # shmem_vec_env.py:61-63
            self.step_wait()
        obs = self._new_obs(self.obs_len)
        self._check(self._lib.irbpp_reset(self._h, None, obs.data_ptr(), self._stream()))
        self._tstart = time.time()
        return obs

    def reset_specific(self, indexs, obs):
        """``ShmemVecEnv.reset_specific`` (shmem_vec_env.py:113-118): reset the listed envs, writing
        their rows of ``obs`` (a [N, obs_len] device tensor) in place."""
        which = np.zeros(self.num_envs, dtype=np.uint8)
        which[np.asarray(indexs, dtype=np.int64)] = 1
        self._check(self._lib.irbpp_reset(self._h, which.ctypes.data, obs.data_ptr(), self._stream()))
        self._torch.cuda.current_stream(self.device).synchronize()   # `which` is read asynchronously
        return obs

    def _take_obs(self):
        """Observation buffer of the step being launched: the one ``step_wait`` allocated while the GPU
        was busy with the previous step, if there is one."""
        obs, self._spare_obs = self._spare_obs, None
        if obs is not None and self._spare_stream != self._stream():
            obs = None                            # allocated under another stream: let the allocator decide
        return obs if obs is not None else self._new_obs(self.obs_len)

    def step_async(self, actions):
        if self.waiting_step:
            raise AlreadySteppingError()
        keep, ptr, on_dev = self._actions_arg(actions, "actions")
        obs = self._take_obs()
        self._release_result_block()
        self._check(self._lib.irbpp_step_async(self._h, ptr, on_dev, obs.data_ptr(), self._stream()))
        self._obs_pending = (obs, keep)
        self.waiting_step = True

    def step_wait(self):
        """-> (obs float32 [N, obs_len] on device, reward float32 [N, 1] on CPU, done bool [N], infos)
        exactly as ``VecPyTorch.step_wait`` (envs.py:161-165)."""
        if not self.waiting_step:
            raise NotSteppingError()
        torch = self._torch
        self.waiting_step = False
        obs, _ = self._obs_pending
        self._obs_pending = None
        if self._spare_obs is None:               # host work that does not need the results: while the kernels run
            self._spare_obs = self._new_obs(self.obs_len)
            self._spare_stream = self._stream()
        t_rel = round(time.time() - self._tstart, 6)
        res = self._result
        self._check(self._lib.irbpp_step_wait(self._h, ctypes.byref(res)))
        src, offs = self._result_block(res)
        n = self.num_envs
        # reward and done are returned as arrays of their own (24 KB); everything else stays in the library's pinned
        # block, which is not reused before the second next step: the infos of a step are normally consumed and dropped
        # by then (trainer.py:167-178) -- if one is still alive when its block comes up for reuse it takes a copy first
        reward = src[offs["reward"]:offs["reward"] + 4 * n].view(np.float32).copy()
        done = src[offs["done"]:offs["done"] + n].view(np.bool_).copy()
        infos = LazyInfos(n, src, offs, done, t_rel, borrowed=True)
        self._live_infos = (self._live_infos + [weakref.ref(infos)])[-2:]
        return obs, torch.from_numpy(reward).unsqueeze(dim=1), done, infos

    def _release_result_block(self):
        """The step about to be launched writes into the pinned block the second-last step used: an infos object
        of that step that is still referenced somewhere takes its private copy now."""
        if len(self._live_infos) == 2:
            old = self._live_infos[0]()
            if old is not None:
                old.detach()

    def _result_block(self, res):
        """uint8 view of the library's pinned result block that the pointers of ``irbpp_step_result`` point into,
        and the byte offset of every array in it (two blocks per handle, each view built once).  Raises when a
        pointer is not where ``_lib.RESULT_FIELDS`` puts it."""
        base = getattr(res, _lib.RESULT_FIELDS[0][0])
        cache = self.__dict__.setdefault("_block_cache", {})      # the library alternates between two blocks
        hit = cache.get(base)
        if hit is None:
            offsets, size = _lib.result_offsets(self.num_envs)
            for k, off in offsets.items():
                if getattr(res, k) != base + off:
                    raise RuntimeError("result block: %s at byte %d, expected %d" % (k, getattr(res, k) - base, off))
            buf = (ctypes.c_uint8 * size).from_address(base)
            hit = cache[base] = (np.frombuffer(buf, dtype=np.uint8), offsets)
        return hit

    def step_device(self, actions):
        """Device-resident loop: ``actions`` is a CUDA int64 tensor; nothing is copied to the host and
        nothing is synchronised.  Returns (obs, reward, done) device views valid in stream order."""
        if self.waiting_step:
            raise AlreadySteppingError()
        keep, ptr, on_dev = self._actions_arg(actions, "actions")
        if not on_dev:
            raise ValueError("step_device needs a CUDA tensor")
        obs = self._new_obs(self.obs_len)
        self._check(self._lib.irbpp_step_async(self._h, ptr, 1, obs.data_ptr(), self._stream()))
        res = self._result
        self._check(self._lib.irbpp_step_wait_device(self._h, ctypes.byref(res)))
        return obs, res

    def last_step_device(self):
        """Device views of the last step's result arrays -- ``reward`` float32 [N], ``done`` / ``valid`` uint8 [N],
        ``counter`` int32 [N], ``ratio`` float64 [N] -- as torch tensors aliasing the library's buffers (valid until
        the next step on this handle): what a device-resident replay bank appends without any host round trip."""
        torch = self._torch
        views = getattr(self, "_dev_views", None)
        if views is None:                             # the device arrays are fixed for the life of the handle: built once
            res = _lib.IrbppStepResult()
            self._check(self._lib.irbpp_device_results(self._h, ctypes.byref(res)))
            n = self.num_envs

            class _View(object):
                def __init__(self, ptr, shape, typestr):
                    self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (int(ptr), False), "version": 2}
            views = self._dev_views = {k: torch.as_tensor(_View(getattr(res, k), (n,), dt.str), device=self.device)
                                       for k, dt in _lib.RESULT_FIELDS if k != "error"}
        return views

    def get_action_candidates(self, order_actions, as_tensor=False):
        """``envs.get_action_candidates(orderAction)`` (shmem_vec_env.py:99-102 -> binPhy.py:161-169).
        Default return matches the reference (list of N float64 host arrays of length 3533, what
        ``trainer.py:267-268`` feeds to ``np.array``); ``as_tensor=True`` returns the float32 device
        tensor and skips the host copy."""
        keep, ptr, on_dev = self._actions_arg(order_actions, "order_actions")
        out = self._new_obs(self.loc_obs_len)
        self._check(self._lib.irbpp_get_action_candidates(self._h, ptr, on_dev, out.data_ptr(), self._stream()))
        if as_tensor:
            return out
        # the reference returns N float64 rows (``trainer.py:267-268`` stacks them with np.array): one D2H copy into
        # pinned memory, one widening pass, rows handed out as views of that array (no per-row copies)
        host = self._pinned_loc()
        host.copy_(out, non_blocking=False)
        wide = host.numpy().astype(np.float64)
        return list(wide)

    def _pinned_loc(self):
        buf = getattr(self, "_loc_pinned", None)
        if buf is None:
            buf = self._torch.empty((self.num_envs, self.loc_obs_len), dtype=self._torch.float32).pin_memory()
            self._loc_pinned = buf
        return buf

    def get_all_possible_observation(self):
        """``PackingGame.get_all_possible_observation`` for every env (binPhy.py:171-180):
        float32 [N, k * 3533] on device."""
        out = self._new_obs(self.buffer_size * self.loc_obs_len)
        self._check(self._lib.irbpp_get_all_possible_observation(self._h, out.data_ptr(), self._stream()))
        return out

    HEURISTICS = ("MINZ", "DBLF", "FIRSTFIT", "HM")     # space.py:168-199; ids = IRBPP_HEUR_* (include/irbpp.h)

    def get_heuristic_actions(self, method, dirIdx=0, as_tensor=False):
        """``Space.get_heuristic_action(dirIdx, method, ...)`` (space.py:162-227) for every env, on the
        scan of the env's current item.  Returns ``(poses, index)``: int32 [N, 3] (rotIdx, lx, ly) and
        int64 [N], the row of that pose in the env's candidate table (a valid ``step`` action) or -1
        when the pose is not a candidate (use ``step_poses`` then).  NumPy arrays, or CUDA tensors
        without any synchronisation when ``as_tensor``."""
        if method not in self.HEURISTICS:
            raise ValueError("unknown heuristic %r (the reference's RANDOM branch raises too)" % (method,))
        m = self.HEURISTICS.index(method)
        if as_tensor:
            torch = self._torch
            poses = torch.empty((self.num_envs, 3), dtype=torch.int32, device=self.device)
            index = torch.empty((self.num_envs,), dtype=torch.int64, device=self.device)
            self._check(self._lib.irbpp_heuristic_actions(self._h, m, int(dirIdx), poses.data_ptr(), index.data_ptr(),
                                                          1, self._stream()))
            return poses, index
        poses = np.empty((self.num_envs, 3), dtype=np.int32)
        index = np.empty((self.num_envs,), dtype=np.int64)
        self._check(self._lib.irbpp_heuristic_actions(self._h, m, int(dirIdx), poses.ctypes.data, index.ctypes.data,
                                                      0, self._stream()))
        return poses, index

    def step_poses(self, poses):
        """``step`` with explicit poses: int64 [N] flat ``(rotIdx * Ax + lx) * Ay + ly`` or an [N, 3]
        array / tensor of (rotIdx, lx, ly) -- what ``action_to_position`` (binPhy.py:234-236) would
        have read from ``candidates[action]``.  Same return tuple as ``step``."""
        if self.waiting_step:
            raise AlreadySteppingError()
        torch = self._torch
        if isinstance(poses, torch.Tensor):
            if poses.dim() == 2:
                poses = (poses[:, 0].to(torch.int64) * 16 + poses[:, 1].to(torch.int64)) * 16 + poses[:, 2].to(torch.int64)
        else:
            poses = np.asarray(poses)
            if poses.ndim == 2:
                poses = (poses[:, 0].astype(np.int64) * 16 + poses[:, 1]) * 16 + poses[:, 2]
            poses = np.ascontiguousarray(poses, dtype=np.int64)
        keep, ptr, on_dev = self._actions_arg(poses, "poses")
        obs = self._take_obs()
        self._release_result_block()
        self._check(self._lib.irbpp_step_poses_async(self._h, ptr, on_dev, obs.data_ptr(), self._stream()))
        self._obs_pending = (obs, keep)
        self.waiting_step = True
        return self.step_wait()

    def close_extras(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.irbpp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- parity / debugging views (float64, host) --
    def launch_count(self):
        return int(self._lib.irbpp_launch_count(self._h))

    def debug_phase_cycles(self, enable=True):
        """Read-and-clear the per-phase SM-cycle counters (see include/irbpp.h) and set the switch."""
        out = np.zeros(8, dtype=np.uint64)
        self._check(self._lib.irbpp_debug_phase_cycles(self._h, 1 if enable else 0, out.ctypes.data))
        return out

    def debug_state(self):
        n, k = self.num_envs, max(self.buffer_size, 1)
        hm = np.zeros((n, 32, 32)); queue = np.zeros((n, k), np.int32)
        cursor = np.zeros(n, np.int32); packed = np.zeros(n, np.int32)
        self._check(self._lib.irbpp_debug_state(self._h, hm.ctypes.data, queue.ctypes.data, cursor.ctypes.data,
                                                packed.ctypes.data))
        return {"heightmap": hm, "queue": queue, "cursor": cursor, "packed": packed}

    def debug_set_heightmap(self, heightmap):
        hm = np.ascontiguousarray(heightmap, dtype=np.float64).reshape(self.num_envs, 32, 32)
        self._check(self._lib.irbpp_debug_set_heightmap(self._h, hm.ctypes.data))

    def debug_scan(self, item_ids):
        n, R, sel = self.num_envs, self.library.num_rotations, self.selected_action
        items = np.ascontiguousarray(item_ids, dtype=np.int32).reshape(n)
        pz = np.zeros((n, R, 16, 16)); pv = np.zeros((n, R, 16, 16)); mk = np.zeros((n, R, 16, 16))
        cand = np.zeros((n, sel, 5)); nh = np.zeros(n, np.int32)
        self._check(self._lib.irbpp_debug_scan(self._h, items.ctypes.data, pz.ctypes.data, pv.ctypes.data,
                                               mk.ctypes.data, cand.ctypes.data, nh.ctypes.data))
        return {"posZmap": pz, "posZValid": pv, "naiveMask": mk, "cand": cand, "num_hull": nh}

    def debug_hulls(self, posZValid, mask):
        n, R, sel = self.num_envs, self.library.num_rotations, self.selected_action
        pv = np.ascontiguousarray(posZValid, dtype=np.float64).reshape(n, R, 16, 16)
        mk = np.ascontiguousarray(mask, dtype=np.float64).reshape(n, R, 16, 16)
        cand = np.zeros((n, sel, 5)); nh = np.zeros(n, np.int32)
        self._check(self._lib.irbpp_debug_hulls(self._h, pv.ctypes.data, mk.ctypes.data, cand.ctypes.data,
                                                nh.ctypes.data))
        return {"cand": cand, "num_hull": nh}
