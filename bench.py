#!/usr/bin/env python
"""bench.py -- env-steps/s of the packing-environment hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--dump-outputs DIR]   # B200 arm, one JSON line on rank 0
    python bench.py --impl reference [--gpus N] --steps K --warmup W [--config NAME]   # reference CPU arm (oracle port)

``--dump-outputs DIR`` writes what the last timed step returned to its caller (rank 0's bins) as ``DIR/<name>.npy``, so
that two builds can be compared output for output: the inputs are seeded and identical from run to run.

``--config`` selects one of BASELINE.json's configurations (default ``blockout`` = configs[1], the one the
metric is quoted on):

    blockout    BlockOut polycubes, 4096 bins/GPU, online, selectedAction=500, R=4           (configs[1], headline)
    cube1       Cube boxes, 1 bin, R=2, online                                                 (configs[0])
    general     irregular height-field shapes, 4096 bins/GPU, R=8 (arguments.py default for General)  (configs[2])
    general24   the same with 24 rotations per shape (configs[2] as BASELINE.json words it)
    buffered10  BlockOut, buffered k=10: one step = get_action_candidates(order) + step(location)     (configs[3])
    abc32k      irregular R=8, 4096 bins/GPU -- meant for --gpus 8 (32768 bins, rollout-end gather)    (configs[4])

A "step" is one batched ``step()`` over all bins of a GPU.  For N > 1 the driver launches one rank per GPU
with torch.distributed.run; bins are sharded by index (weak scaling), there is no collective inside a step,
and ONE gather of the observations per rollout (NCCL all-gather; IRBPP_GATHER selects the measured alternatives:
copy-engine pulls through torch symmetric memory, the packed form, send/recv pairs).  That gather is pipelined (SURVEY.md 8e): the gather of the previous
rollout's observations is started with this rollout's first timed step and runs on a side stream beside the steps.  Its
cost enters the timed total twice: the steps it overlaps are timed with it running (whatever it slows them down by is in
their event pairs), and `gather_exposed_ms` is added -- the part after the last step in full, the part that fell into the
benchmark's own L2-flush gaps at the price it would have beside further steps (see gather_account), plus the pack / expand
kernels of the compact form.  `gather_hidden_ms`, `gather_beside_flush_ms`, `gather_tail_ms` are reported next to it.

Timing: every timed step is bracketed by CUDA events on the launching stream; between timed steps the L2 is
flushed by writing a 256 MiB buffer (outside the event pairs).  ``value`` uses actions that are already on the
device; ``e2e`` calls the public ``GpuVecEnv.step`` with HOST actions (pinned H2D copy, kernels, D2H of
reward/done/info arrays) and is timed with the host clock around the call.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEL = 500
SEQ_LEN = 128
CPU_BURN_IN = 40         # untimed batched steps of the CPU arm before its timed samples
BURN_IN = 150            # untimed steps before the W warm-up steps so episodes are in steady state
UNIT = "env-steps/s"
CPU_ENVS_PER_CORE = 2    # bins per worker process of the CPU arm (same in cpu_baseline and --impl reference)
CPU_SAMPLES = 3          # the CPU arm reports the median of this many timed samples
DEFAULT_NCCL_CHANNELS = 0   # channels (= SMs) of the rollout all-gather; 0 = NCCL's default (see main_gpu)
DUMP_LIMIT_BYTES = 64 * 10 ** 6   # --dump-outputs: larger outputs are written as a seeded sample of bins

CONFIGS = {
    "blockout": dict(bins=4096, k=1, R=4, metric="env steps/sec (4096 bins, BlockOut)",
                     workload="BlockOut-like polycubes (32 shapes, 2-5 cells of 0.04 m), 4096 bins per GPU, online "
                              "(bufferSize=1), selectedAction=500, R=4, bin 0.32x0.32x0.30, random-valid policy"),
    "cube1": dict(bins=1, k=1, R=2, metric="env steps/sec (1 bin, Cube)",
                  workload="Cube boxes (125 shapes, edges 0.03-0.15 m), 1 bin, online, selectedAction=500, R=2, "
                           "random-valid policy (BASELINE.json configs[0])"),
    "general": dict(bins=4096, k=1, R=8, metric="env steps/sec (4096 bins, General irregular R=8)",
                    workload="irregular height-field shapes (32 shapes, non-flat bottoms, holes, off-grid extents), 4096 "
                             "bins per GPU, online, selectedAction=500, R=8, random-valid policy (BASELINE.json configs[2])"),
    "general24": dict(bins=4096, k=1, R=24, metric="env steps/sec (4096 bins, General irregular R=24)",
                      workload="irregular height-field shapes (32 shapes), 4096 bins per GPU, online, selectedAction=500, "
                               "24 rotations per shape, random-valid policy (BASELINE.json configs[2], 24-rotation wording)"),
    "buffered10": dict(bins=4096, k=10, R=4, metric="env steps/sec (4096 bins, BlockOut buffered k=10)",
                       workload="BlockOut-like polycubes, 4096 bins per GPU, buffered k=10 (--hierachical): one step = "
                                "get_action_candidates(random order action) + step(random-valid location action), "
                                "selectedAction=500, R=4 (BASELINE.json configs[3])"),
    "abc32k": dict(bins=4096, k=1, R=8, metric="env steps/sec (4096 bins per GPU, ABC-like irregular R=8)",
                   workload="irregular height-field shapes (ABC stand-in, 32 shapes), 4096 bins per GPU (32768 at --gpus 8), "
                            "online, selectedAction=500, R=8, rollout-end all-gather (BASELINE.json configs[4])"),
}


def make_library(config):
    from irbpp_b200 import shapes
    if config in ("blockout", "buffered10"):
        return shapes.make_blockout_library(32, seed=1, num_rotations=4)
    if config == "cube1":
        return shapes.make_cube_library(seed=3)
    if config in ("general", "abc32k"):
        return shapes.make_irregular_library(32, seed=2, num_rotations=8)
    if config == "general24":
        return shapes.make_irregular_library(32, seed=2, num_rotations=24)
    raise SystemExit("unknown config %r" % config)


def algorithmic_bytes_per_env_step(lib, k=1, sel=SEL):
    """SURVEY.md 8(d): 2*Hx*Hy*8 [hm r+w] + R*Ax*Ay*16 [posZ+mask] + sum_r 2*w_r*h_r*8 [B, maskB of the
    next item] + 2*w*h*8 [T, maskT of the placed rotation] + obs_len*4 [float32 observation], averaged
    over the shape library (ids are uniform).  Buffered (k > 1): the candidate pass reads the heightmap
    once more and writes the location observation; the step writes the order observation [k + 1024]."""
    R = lib.num_rotations
    wh = (lib.dims[:, :, 0].astype(np.float64) * lib.dims[:, :, 1])
    loc_len = sel * 5 + 9 + 1024
    base = 2 * 32 * 32 * 8 + R * 16 * 16 * 16 + float(wh.sum(axis=1).mean()) * 16 + float(wh.mean()) * 16 + loc_len * 4
    if k > 1:
        base += 32 * 32 * 8 + (k + 1024) * 4
    return base


class ClockSampler(object):
    """SM clock and throttle reasons sampled while the benchmark loop runs: NVML queries from a thread of this process
    (pynvml; a few microseconds each), or an `nvidia-smi -lms` subprocess when pynvml is missing.  (Round 2: the
    nvidia-smi loop at 20 ms was replaced after single steps of 1-30 ms showed up on multi-GPU boxes.)"""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, period_s=0.025):
        self.index, self.rows, self.proc, self.period = index, [], None, period_s
        self._stop = threading.Event()
        self.thread = None
        self.how = None

    def _nvml_loop(self, nv, handle):
        masks = [(nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                 (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")]
        smax = nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                bits = nv.nvmlDeviceGetCurrentClocksEventReasons(handle)
                self.rows.append((float(sm), float(smax), [nm for m, nm in masks if bits & m]))
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # torch numbers the devices like CUDA does; NVML by PCI order: resolve through the UUID-free common case
            # (CUDA_VISIBLE_DEVICES unset, CUDA_DEVICE_ORDER default = fastest first == PCI order on a homogeneous box)
            handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.how = "nvml"
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.how = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) < 6:
                continue
            try:
                self.rows.append((float(parts[0]), float(parts[1]),
                                  [nm for nm, v in zip(self.NAMES, parts[2:6]) if v.lower().startswith("active")]))
            except ValueError:
                continue

    def stop(self):
        if self.how is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"]}
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        sm = [r[0] for r in self.rows]
        reasons = set()
        for r in self.rows:
            reasons.update(r[2])
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.rows[-1][1] if self.rows else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.how}


def device_policy(torch, obs, gen):
    """Stand-in for the agent (trainer.py:161-162): a uniformly random candidate with V == 1 (row 0 if
    none), computed on the device from the observation's mask column."""
    n = obs.shape[0]
    mask = obs[:, :SEL * 5].view(n, SEL, 5)[:, :, 4] == 1
    score = torch.rand((n, SEL), device=obs.device, generator=gen) + mask.float()
    return torch.argmax(score, dim=1)


def step_outputs(env, state):
    """Host copies of what the last device-resident step handed its caller: the observation, the location candidates
    it chose from (buffered) and the per-bin result arrays.  Integer and flag arrays become float64, which is exact."""
    out = {"obs": state["obs"]}
    if "loc" in state:
        out["candidates"] = state["loc"]
    out.update(env.last_step_device())
    out = {k: v.cpu().numpy() for k, v in out.items()}
    return {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in out.items()}


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES, seed=0):
    """Write every [N, ...] array of `arrays` as out_dir/<name>.npy and the bin index of each row as bins.npy.  When the
    whole would exceed `limit` bytes, every array is cut to the same fixed, seeded sample of bins."""
    n = len(arrays["obs"])
    row_bytes = 8 + sum(a[:1].nbytes for a in arrays.values())
    rows = min(n, (limit - 4096) // row_bytes)            # 4096: room for the .npy headers
    bins = np.arange(n) if rows == n else np.sort(np.random.default_rng(seed).choice(n, rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "bins.npy"), bins.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[bins])


def host_policy(rng, obs):
    n = obs.shape[0]
    mask = obs[:, :SEL * 5].reshape(n, SEL, 5)[:, :, 4] == 1
    score = rng.random((n, SEL)) + mask
    return np.argmax(score, axis=1).astype(np.int64)


# ---------------------------------------------------------------------------------------------------
# CPU reference arm / baseline (oracle port; the reference itself is Python that cannot be installed:
# it imports trimesh / gym / pybullet which are absent, see DESIGN.md)
# ---------------------------------------------------------------------------------------------------

def _spin(q, seconds):
    t_end = time.perf_counter() + seconds
    n = 0
    x = 1.0
    while time.perf_counter() < t_end:
        for _ in range(20000):
            x = x * 1.0000001 + 1e-9
        n += 1
    q.put(n)


def host_cores():
    """How many host cores this process may really use.  ``os.cpu_count()`` is the machine's count; a
    container is usually limited by the affinity mask and / or a cgroup CPU quota (round 1's 1-GPU lease
    ran 128 workers on a fraction of the 128 advertised cores).  Besides reading those limits the
    parallel speed-up of a spin loop is measured, which also catches limits that are not visible here."""
    import multiprocessing as mp
    info = {"cpu_count": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["cpu_count"]
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            q, p = open(path).read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
        except Exception:
            pass
    if quota is None:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    info["cgroup_quota"] = quota
    declared = info["affinity"]
    if quota is not None:
        declared = max(1, min(declared, int(quota + 0.5)))
    # measured: throughput of `declared` concurrent spinners relative to one spinner
    ctx = mp.get_context("fork")

    def rate(nproc, seconds=0.8):
        q = ctx.Queue()
        ps = [ctx.Process(target=_spin, args=(q, seconds)) for _ in range(nproc)]
        for p in ps:
            p.start()
        tot = sum(q.get() for _ in ps)
        for p in ps:
            p.join()
        return tot / seconds
    try:
        one = max(rate(1), rate(1))                  # best of two: a busy neighbour must not look like a quota
        many = max(rate(declared), rate(declared))
        info["measured_parallelism"] = round(many / one, 1)
    except Exception:
        info["measured_parallelism"] = None
    cores = declared
    mp_ = info["measured_parallelism"]
    if mp_ is not None and mp_ < 0.6 * declared:           # far fewer real cores than declared: do not oversubscribe
        cores = max(1, int(mp_ + 0.5))
    info["cores_used"] = cores
    return info


def run_cpu_arm(config, steps, warmup, max_seconds=None):
    """The reference-style CPU vector env on this box's host cores: one worker process per usable core
    (ShmemVecEnv shape), CPU_ENVS_PER_CORE bins each, CPU_SAMPLES timed samples of `steps` batched steps
    (or until max_seconds per sample); the median sample is reported."""
    from irbpp_b200 import shapes
    from oracle.cpu_vec_env import SubprocOracleVecEnv
    spec = CONFIGS[config]
    lib = make_library(config)
    hc = host_cores()
    cores = hc["cores_used"]
    k = spec["k"]
    if spec["bins"] == 1:
        cores = 1
        n = 1
    else:
        n = cores * CPU_ENVS_PER_CORE
    seqs = shapes.make_sequences(n, SEQ_LEN, lib.num_shapes, seed=0)
    vec = SubprocOracleVecEnv(dict(ZRotNum=spec["R"], selectedAction=SEL, bufferSize=k), lib, seqs, num_procs=cores)
    rng = np.random.default_rng(0)
    obs = vec.reset()

    def one(obs):
        if k > 1:
            loc = vec.get_action_candidates(rng.integers(0, k, size=n))
            acts = host_policy(rng, loc)
        else:
            acts = host_policy(rng, obs)
        return vec.step(acts)[0]

    t_burn = time.perf_counter()
    for i in range(CPU_BURN_IN + warmup):            # untimed: reach a steady mix of episode phases
        obs = one(obs)
        if max_seconds is not None and time.perf_counter() - t_burn > max_seconds and i >= 5:
            break
    samples = []
    for _ in range(CPU_SAMPLES):
        t_total, done_steps = 0.0, 0
        for _ in range(steps):
            if k > 1:
                order = rng.integers(0, k, size=n)
                t0 = time.perf_counter()
                loc = vec.get_action_candidates(order)
                t_total += time.perf_counter() - t0
                acts = host_policy(rng, loc)
            else:
                acts = host_policy(rng, obs)
            t0 = time.perf_counter()
            obs = vec.step(acts)[0]
            t_total += time.perf_counter() - t0
            done_steps += 1
            if max_seconds is not None and t_total > max_seconds:
                break
        samples.append((n * done_steps / t_total, done_steps, t_total))
    vec.close()
    samples.sort()
    value, done_steps, t_total = samples[len(samples) // 2]
    return {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d bins (%d per worker) x %d batched steps per sample, median of %d samples (%s env-steps/s), one worker "
                      "process per usable core over pipes (ShmemVecEnv shape), oracle port with reference-style loops + cv2, "
                      "no PyBullet; host cores: cpu_count %s, affinity %s, cgroup quota %s, measured parallel speed-up %s -> %d "
                      "workers (round 1 spawned cpu_count workers, which oversubscribed quota-limited boxes)"
                      % (n, n // cores, done_steps, len(samples), "/".join("%.0f" % s[0] for s in samples), hc["cpu_count"],
                         hc["affinity"], hc["cgroup_quota"], hc["measured_parallelism"], cores),
            "per_core": value / cores, "host": hc,
            "steps": done_steps, "ms_per_step": 1e3 * t_total / done_steps, "n_envs": n}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    spec = CONFIGS[args.config]
    res = run_cpu_arm(args.config, max(args.steps, 1), max(args.warmup, 1), max_seconds=args.cpu_seconds * 4)
    line = {"impl": "reference", "metric": spec["metric"], "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": res["steps"], "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": spec["workload"] + " [CPU arm: bounded sample of %d bins on %d host cores]"
                                   % (res["n_envs"], res["cores"]), "name": args.config},
            "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": res["kind"],
                             "sample": res["sample"], "per_core": res["per_core"]},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------

def overlap_ms(origin, a0, a1, spans):
    """Milliseconds of [a0, a1] that ran concurrently with any of `spans` (pairs of CUDA events);
    all positions measured from `origin`."""
    g0, g1 = origin.elapsed_time(a0), origin.elapsed_time(a1)
    tot = 0.0
    for s0, s1 in spans:
        x0, x1 = origin.elapsed_time(s0), origin.elapsed_time(s1)
        tot += max(0.0, min(g1, x1) - max(g0, x0))
    return tot, g1 - g0


def gather_account(origin, gev, steps, others):
    """Where one rollout gather [gev] ran, relative to the timed `steps` (event pairs) and the `others` spans (agent stand-in):
      hidden        beside a step or the agent
      tail          after the last step ended                                   -> exposed in full
      beside_flush  in the gaps the benchmark's L2 flushes open between steps; a training loop has no such gaps, this part
                    of the transfer would run beside the following steps instead -> charged what it would cost there:
                    (beside_flush / undisturbed step time) further steps, each slowed like the steps the gather did overlap
    Returns (gather_ms, hidden, tail, beside_flush, exposed)."""
    hidden, g = overlap_ms(origin, gev[0], gev[1], list(steps) + list(others))
    hidden = min(hidden, g)
    g0, g1 = origin.elapsed_time(gev[0]), origin.elapsed_time(gev[1])
    spans = [(origin.elapsed_time(a), origin.elapsed_time(b)) for a, b in steps]
    last_end = max(b for _, b in spans)
    tail = max(0.0, g1 - max(last_end, g0))
    beside_flush = max(0.0, g - hidden - tail)
    touched = [b - a for a, b in spans if min(g1, b) - max(g0, a) > 0.0]
    free = [b - a for a, b in spans if min(g1, b) - max(g0, a) <= 0.0]
    slow = max(0.0, float(np.mean(touched)) - float(np.mean(free))) if touched and free else 0.0
    base = float(np.mean(free)) if free else float(np.mean([b - a for a, b in spans]))
    exposed = tail + (beside_flush / base) * slow
    return g, hidden, tail, beside_flush, exposed


def main_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    spec = CONFIGS[args.config]
    n_envs, k = spec["bins"], spec["k"]

    cpu_base = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        # before CUDA is initialised in this process (workers are forked)
        cpu_base = run_cpu_arm(args.config, steps=10 ** 9, warmup=2, max_seconds=args.cpu_seconds / CPU_SAMPLES)
        for key in ("steps", "ms_per_step", "n_envs", "host"):
            cpu_base.pop(key, None)

    import torch
    import torch.distributed as dist
    import irbpp_b200
    from irbpp_b200 import shapes, sharding
    from irbpp_b200.vec_env import GpuVecEnv

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # The rollout gather runs beside the next rollout's steps.  NCCL's default all-gather takes up to 32 SMs with
        # one fat CTA each for its whole duration; the candidates kernel's grid fits the 148 SMs exactly once, so any
        # SM it loses costs it a second wave (8 GPUs: steps 0.108 -> 0.145 ms while the gather ran).  Fewer channels make
        # the gather slower but narrower; it has the whole rollout to finish.  IRBPP_NCCL_CHANNELS overrides (0: NCCL's choice).
        ch = int(os.environ.get("IRBPP_NCCL_CHANNELS", str(DEFAULT_NCCL_CHANNELS)))
        if ch > 0:
            os.environ["NCCL_MAX_NCHANNELS"] = str(ch)
            os.environ["NCCL_MIN_NCHANNELS"] = str(min(ch, 4))
        dist.init_process_group("nccl", device_id=dev)

    lib = make_library(args.config)
    n_total = n_envs * world
    seqs_all = shapes.make_sequences(n_total, SEQ_LEN, lib.num_shapes, seed=0)
    seqs = sharding.shard_sequences(seqs_all, rank, world)
    env = GpuVecEnv(lib, seqs, device=dev, selected_action=SEL, buffer_size=k)
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    state = {"obs": None}

    def choose():
        """the stand-in agent (outside the timed intervals): -> what one_step consumes"""
        if k > 1:
            return torch.randint(0, k, (n_envs,), device=dev, generator=gen)
        return device_policy(torch, state["obs"], gen)

    def one_step(choice, ev=None):
        """one batched env step on the device-resident path; `ev` brackets the library's work"""
        if k > 1:
            if ev is not None:
                ev[0].record()
            state["loc"] = env.get_action_candidates(choice, as_tensor=True)
            acts = device_policy(torch, state["loc"], gen)   # the location agent needs the candidates: inside the interval
            state["obs"], _ = env.step_device(acts)
        else:
            if ev is not None:
                ev[0].record()
            state["obs"], _ = env.step_device(choice)
        if ev is not None:
            ev[1].record()

    # ---- device-resident loop ("value") ----
    import gc
    gc.collect()
    gc.disable()                                    # a generation-2 collection inside a timed step showed up as a 1-30 ms "step"
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                             # sampled from burn-in through the timed steps (same load)
    state["obs"] = env.reset()
    for _ in range(BURN_IN + args.warmup):          # burn-in: bins spread over all episode phases
        one_step(choose())
    gatherer = None
    if world > 1:
        # IRBPP_GATHER: nccl (default: plain all-gather on the side stream) | symm (copy-engine pulls over torch symmetric
        # memory) | compact (all-gather of the packed observations, expanded on arrival) | sendrecv | peer (CUDA IPC pushes).
        # 8 x B200, 4096 bins each, same box (profiles/README.md): nccl 0.1165 ms/step, compact 0.1212, symm 0.1288 -- the
        # copy-engine pulls leave the SMs alone but one step beside them took 0.33 ms, the all-gather kernel costs less.
        kind = os.environ.get("IRBPP_GATHER", "nccl")
        gatherer = (sharding.PeerCopyGather(world) if kind == "peer" else sharding.SymmMemGather(world) if kind == "symm" else
                    sharding.CompactRolloutGather(SEL, world) if kind == "compact" and k == 1 else
                    sharding.AsyncRolloutGather(world, point_to_point=(kind == "sendrecv")))
    gather_alone_ms = 0.0
    if world > 1:                                   # warm-up of the rollout-end collective (NCCL channel setup) + its stand-alone time
        for _ in range(2):
            gatherer.start(state["obs"]); gatherer.finish()
        torch.cuda.synchronize(dev)
        gather_alone_ms = gatherer.events[0].elapsed_time(gatherer.events[1])
    # rehearsal: a few untimed iterations shaped exactly like the timed ones (L2 flush, event records), so that nothing
    # is done for the first time inside the timed region (a first-use stall showed up as one 60 ms step on a fresh box)
    for i in range(3):
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        choice = choose()
        flush.fill_(float(i))
        one_step(choice, (r0, r1))
    torch.cuda.synchronize(dev)
    launches0 = env.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    origin = torch.cuda.Event(enable_timing=True)
    tail0, tail1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.perf_counter()
    # runway: the GPU spins for ~30 ms while the host enqueues all K iterations, so the event intervals below are GPU time
    # only -- a host hiccup between two launches of a step (seen as single "steps" of 1-30 ms) cannot land inside them
    torch.cuda._sleep(int(0.030 * 1.9e9))
    origin.record()
    prev_rollout_obs = state["obs"]
    ev_pol = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)] if world > 1 else None
    for i in range(args.steps):
        if world > 1:
            ev_pol[i][0].record()
        choice = choose()
        if world > 1:
            ev_pol[i][1].record()
        flush.fill_(float(i))                       # L2 flush, outside the event pair
        if i == 0 and world > 1:                    # the previous rollout's observations go out while this rollout's
            gatherer.start(prev_rollout_obs)        # first steps run (side stream; starts with the first timed step)
        one_step(choice, ev[i])
    gathered = None
    if world > 1:
        tail0.record()
        gathered = gatherer.finish()
        tail1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches_timed = env.launch_count() - launches0
    outputs = step_outputs(env, state) if args.dump_outputs and rank == 0 else None   # before any further step
    # the timed region lasts ~10-30 ms: keep the same loop running (untimed) until nvidia-smi has
    # delivered enough clock samples under this load
    extra_steps = 0
    if rank == 0:
        t_end = time.perf_counter() + 2.5
        while len(sampler.rows) < 20 and time.perf_counter() < t_end:
            for _ in range(20):
                one_step(choose())
            torch.cuda.synchronize(dev)
            extra_steps += 20
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "burn-in + timed steps + %d further untimed steps of the same loop" % extra_steps
    step_ms = [a.elapsed_time(b) for a, b in ev]
    gather_ms = gather_exposed = gather_hidden = gather_tail = gather_flush = gather_extra = 0.0
    if world > 1:
        assert gathered.shape[0] == n_total
        gather_ms, gather_hidden, gather_tail, gather_flush, gather_exposed = gather_account(origin, gatherer.events, ev, ev_pol)
        for evs in (getattr(gatherer, "pack_events", None), getattr(gatherer, "unpack_events", None)):
            if evs is not None:                     # pack / expansion of the compact form run on the step stream: always exposed
                gather_extra += evs[0].elapsed_time(evs[1])
        gather_exposed += gather_extra
    t_dev_ms = float(sum(step_ms)) + gather_exposed
    t_strict_ms = float(sum(step_ms)) + (gather_ms - gather_hidden) + gather_extra     # every ms outside a step / the agent charged
    t = torch.tensor([t_dev_ms, float(np.mean(step_ms)), gather_ms, gather_exposed, gather_alone_ms, gather_hidden, gather_tail, gather_flush,
                      t_strict_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_dev_ms, kern_ms, gather_ms, gather_exposed, gather_alone_ms, gather_hidden, gather_tail, gather_flush, t_strict_ms = [float(v) for v in t.tolist()]
    value = n_total * args.steps / (t_dev_ms * 1e-3)

    # ---- end-to-end loop through the public API with host actions ----
    e2e_steps = args.steps
    t_e2e = 0.0

    def e2e_step(timed, gather_obs=None):
        if k > 1:
            order = torch.randint(0, k, (n_envs,), device=dev, generator=gen).cpu().numpy()
        else:
            acts = device_policy(torch, state["obs"], gen).cpu().numpy()   # agent -> action.cpu().numpy() (trainer.py:165)
        if timed is not None:
            flush.fill_(1.0)
            torch.cuda.synchronize(dev)
            if gather_obs is not None:
                gatherer.start(gather_obs)          # the previous rollout's gather runs beside this rollout's first steps
            timed[0].record()
        t0 = time.perf_counter()
        if k > 1:
            loc = env.get_action_candidates(order, as_tensor=True)       # H2D order actions, kernels; stays on device
            acts = device_policy(torch, loc, gen).cpu().numpy()            # location agent -> host actions (trainer.py:272-281)
        out = env.step(acts)                                               # H2D actions, kernels, D2H results
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if timed is not None:
            timed[1].record()
        state["obs"] = out[0]
        return dt

    for _ in range(min(args.warmup, 3)):
        e2e_step(None)
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(e2e_steps)]
    origin2 = torch.cuda.Event(enable_timing=True)
    barrier()
    origin2.record()
    prev_rollout_obs = state["obs"]
    for i in range(e2e_steps):
        t_e2e += e2e_step(ev2[i], prev_rollout_obs if (i == 0 and world > 1) else None)
    e2e_gather_exposed = 0.0
    if world > 1:
        gatherer.finish()
        torch.cuda.synchronize(dev)
        e2e_gather_exposed = gather_account(origin2, gatherer.events, ev2, [])[4]
        for evs in (getattr(gatherer, "pack_events", None), getattr(gatherer, "unpack_events", None)):
            if evs is not None:
                e2e_gather_exposed += evs[0].elapsed_time(evs[1])
    te = torch.tensor([t_e2e + e2e_gather_exposed * 1e-3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    t_e2e = float(te.item())
    e2e_value = n_total * e2e_steps / t_e2e
    h2d = n_envs * 8 * (2 if k > 1 else 1)                          # int64 actions (+ order actions when buffered)
    d2h = n_envs * (8 + 8 + 4 + 4 + 4 + 1 + 1 + 1)                  # ratio, ep_reward, reward, counter, ep_len, done, valid, error
    if k > 1:
        d2h += n_envs * 8                                           # the location agent's actions come back to the host

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        bytes_step = algorithmic_bytes_per_env_step(lib, k) * n_envs
        achieved = bytes_step / (kern_ms * 1e-3) / 1e9
        traffic, traffic_note = None, "no ncu capture of this kernel version / config committed"
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")))
            entry = prof.get(args.config)
            if entry and entry.get("kernel_version") == irbpp_b200.KERNEL_VERSION:
                traffic = entry.get("dram_bytes_per_launch")
                traffic_note = "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of the step's kernels, %s (%s)" % (
                    entry.get("source", "profiles/"), entry.get("kernel_version"))
            elif entry:
                traffic_note = "committed capture is of kernel version %s, this is %s" % (entry.get("kernel_version"), irbpp_b200.KERNEL_VERSION)
        except Exception:
            pass
        line = {"metric": spec["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": t_dev_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": spec["workload"], "name": args.config, "bins_per_gpu": n_envs, "burn_in_steps": BURN_IN,
                           "parallelism": "env-shard x%d" % world, "kernel_version": irbpp_b200.KERNEL_VERSION,
                           "l2": "flushed between timed steps by a 256 MiB write outside the event pairs",
                           "timing": "sum of per-step CUDA-event intervals on the launching stream"
                                     + (" + the part of the pipelined rollout all-gather that overlapped neither a timed step nor the agent stand-in" if world > 1 else "")
                                     + ", max over ranks"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                             "kernel": "irbpp_scan_kernel + irbpp_candidates_kernel (one step = both launches"
                                       + ("; buffered: a candidates pass + the order-level step" if k > 1 else "") + ")",
                             "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": bytes_step},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": 1e3 * t_e2e / e2e_steps,
                        "note": "GpuVecEnv.step(host int64 actions): pinned staging, kernels, reward/done/info arrays back to the "
                                "host, stream sync; observations stay on the device as in the reference (envs.py:163)"
                                + ("; includes the exposed part of the rollout all-gather" if world > 1 else "")},
                "gpu_launches": int(launches_timed), "clocks": clocks, "wall_s_timed_region": t_wall,
                "step_ms": {"median": float(np.median(step_ms)), "min": float(np.min(step_ms)), "max": float(np.max(step_ms))}}
        if world > 1:
            line["gather_ms"] = gather_ms
            line["gather_exposed_ms"] = gather_exposed
            line["gather_hidden_ms"] = gather_hidden
            line["gather_beside_flush_ms"] = gather_flush
            line["gather_tail_ms"] = gather_tail
            line["value_charging_flush_gaps"] = n_total * args.steps / (t_strict_ms * 1e-3)   # round-1 accounting, for comparison
            line["gather_alone_ms"] = gather_alone_ms
            line["gather_kind"] = getattr(gatherer, "kind", "nccl all-gather")
            line["nccl_channels"] = os.environ.get("NCCL_MAX_NCHANNELS", "default")
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line))
    env.close()
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="blockout", choices=sorted(CONFIGS))
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="bound of the cpu_baseline timed samples (wall seconds, all samples)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: only the B200 arm has a timed device step to dump")
        return main_reference(args)
    return main_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
