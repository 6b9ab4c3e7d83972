#!/usr/bin/env python
"""Times of the prioritized replay bank (irbpp_b200/replay.py) at the reference's learner sizes: N = 4096 bins,
C = 1e5 / 4096 = 24 transitions per bin, L = 3533 (location observation), batch 64.  GPU only.

    python tools/replay_bench.py [--iters 200] [--loop-iters 60] [--port-steps 3]

* append / sample / update: mean wall time per call over --iters calls (CUDA events; sample includes the host check of
  the per-row error flags, update the host np.power and the copy of 64 priorities), after a warm-up;
* actor loop: tools/actor_loop.py's batched loop (mask -> act -> env.step -> episode stats -> append, sample every 4th
  iteration) with the prioritized bank (sample + update_priorities) and with the uniform learner_glue.ReplayBank,
  alternated in the same process;
* CPU port: N one-bank ReplayPort objects driven as trainer.py:184-186 drives N ReplayMemory objects (a Python loop of
  appends per step), and one draw + update from each of 64 of them.
Prints one JSON line, with the GPU's name and power limit."""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from irbpp_b200 import shapes, learner_glue as glue
from irbpp_b200.replay import PrioritizedReplayBank
from irbpp_b200.vec_env import GpuVecEnv

SEL = 500


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else torch.cuda.get_device_name(0)
    except Exception:
        return torch.cuda.get_device_name(0)


def time_calls(fn, iters):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters          # us per call


def actor_loop(env, state, bank, iters, prioritized, gen, batch=64, freq=4):
    stats = glue.EpisodeStats()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for T in range(1, iters + 1):
        mask = glue.get_mask_from_state(state, SEL)
        q = torch.rand(mask.shape, device=state.device, generator=gen)
        q[(1 - mask).bool()] = -float("inf")
        action = q.argmax(1)
        next_state, reward, done, infos = env.step(action.cpu().numpy())
        stats.update(done, infos)
        bank.append_from_env(env, state, action, reward_clip=10.0)
        if T % freq == 0:
            if prioritized:
                idx = bank.sample(batch)[0]
                bank.update_priorities(idx, torch.rand(batch, generator=torch.Generator().manual_seed(T)))
            else:
                bank.sample(batch)
        state = next_state
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return state, {"iters_per_s": iters / dt, "env_steps_per_s": env.num_envs * iters / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--loop-iters", type=int, default=60)
    ap.add_argument("--port-steps", type=int, default=3)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    N, C, L, B = 4096, 24, 3533, 64
    out = {"gpu": gpu_info(), "bins": N, "capacity": C, "obs_len": L, "batch": B}
    g = torch.Generator(device=dev); g.manual_seed(0)
    bank = PrioritizedReplayBank(N, C, L, dev, priority_weight=0.4)
    state = torch.randn((N, L), device=dev, generator=g)
    action = torch.randint(0, SEL, (N,), device=dev, generator=g)
    reward = torch.rand(N, device=dev, generator=g)
    done = (torch.rand(N, device=dev, generator=g) < 0.05).to(torch.uint8)
    for _ in range(C + 4):
        bank.append_batch(state, action, reward, done)
    out["append_us"] = time_calls(lambda: bank.append_batch(state, action, reward, done), a.iters)
    out["append_bytes"] = N * L * 4 * 2                       # the state rows read and written
    out["append_GBps"] = out["append_bytes"] / (out["append_us"] * 1e-6) / 1e9
    out["sample_us"] = time_calls(lambda: bank.sample(B), a.iters)
    idx = bank.sample(B)[0]
    loss = torch.rand(B)
    out["update_us"] = time_calls(lambda: bank.update_priorities(idx, loss), a.iters)

    # actor loop: prioritized bank vs the uniform ReplayBank, alternated
    env = GpuVecEnv(shapes.make_blockout_library(32, seed=1), None, num_envs=N, device=dev, item_seed=1)
    s = env.reset()
    pbank = PrioritizedReplayBank(N, C, env.obs_len, dev, priority_weight=0.4)
    ubank = glue.ReplayBank(N, C, env.obs_len, dev)
    s, _ = actor_loop(env, s, pbank, 2 * C, True, g)            # fill both banks, warm every shape
    s, _ = actor_loop(env, s, ubank, 2 * C, False, g)
    loops = {"prioritized": [], "uniform": []}
    for rep in range(2):
        s, r = actor_loop(env, s, pbank, a.loop_iters, True, g); loops["prioritized"].append(r)
        s, r = actor_loop(env, s, ubank, a.loop_iters, False, g); loops["uniform"].append(r)
    env.close()
    out["actor_loop"] = loops

    # CPU port as trainer.py uses N ReplayMemory objects
    from oracle.replay_port import ReplayPort
    mems = [ReplayPort(1, C, L, 0.99, 3) for _ in range(N)]
    st = state.cpu().numpy(); ac = action.cpu().numpy(); rw = reward.cpu().numpy(); dn = done.cpu().numpy().astype(bool)
    for _ in range(C):
        for i in range(N):
            mems[i].append(st[i:i + 1], ac[i:i + 1], rw[i:i + 1], dn[i:i + 1])
    t0 = time.perf_counter()
    for _ in range(a.port_steps):
        for i in range(N):
            mems[i].append(st[i:i + 1], ac[i:i + 1], rw[i:i + 1], dn[i:i + 1])
    out["cpu_port_append_ms_per_step"] = (time.perf_counter() - t0) * 1e3 / a.port_steps
    rng = np.random.default_rng(0)
    t0 = time.perf_counter()
    for i in rng.choice(N, B, replace=False):
        r = mems[i].sample(1, rng.random((1, 64)))
        mems[i].update_priorities(r[0], np.float32([1.0]))
    out["cpu_port_sample_update_ms"] = (time.perf_counter() - t0) * 1e3
    print(json.dumps(out))


if __name__ == "__main__":
    main()
