"""Time per step with uint8 against packed (obs_dtype="bits", WF_OBS_BITS) observations, variants alternating on one GPU.
    python tools/obs_bits_timing.py [blocks]
Prints the card's name and power limit first, then one line per measurement and block:
  - wf_rollout of C4 (1024 x 256x256), C5 (64 x 1024x1024) and C2 (4096 x 14x14) at bench.py's launch sizes
    (CUDA events around back-to-back launches into preallocated outputs, about 0.3 s per block);
  - wf_step_host of C2 with the step-server session (wf_host_session mode 1), uint8 against bits, same host threads;
  - wf_step_host of C4 (tile family, no session), uint8 against bits.
The observation bytes per step follow from the shapes and are printed beside the times."""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import WORKLOADS  # noqa: E402
from wildfire_control_python_b200 import BatchedForestFire, obs_bits_words  # noqa: E402

BLOCKS = int(sys.argv[1]) if len(sys.argv) > 1 else 3
LAUNCHES = {"c4": 100, "c5": 200, "c2": 600}  # about 0.3 s of GPU time per block
VARIANTS = (torch.uint8, "bits")


def name(dt):
    return "bits" if dt == "bits" else "uint8"


def obs_bytes(n, w, h, dt):
    return n * (obs_bits_words(w, h) * 4 if dt == "bits" else w * h * 3)


def card():
    r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else torch.cuda.get_device_name()


def make(wl, dt, n=None):
    env = BatchedForestFire(n or wl["n_envs"], obs_dtype=dt, auto_reset=True, seed=0, **wl["meta"])
    env.reset()
    return env


def rollout_timing(w):
    wl = WORKLOADS[w]
    N, K, (W, H) = wl["n_envs"], wl["chunk"], (wl["meta"]["width"], wl["meta"]["height"])
    arms = {}
    for dt in VARIANTS:
        env = make(wl, dt)
        shape = (K, N, obs_bits_words(W, H)) if dt == "bits" else (K, N, W, H, 3)
        out = (torch.empty(shape, dtype=torch.int32 if dt == "bits" else dt, device="cuda"),
               torch.empty((K, N), dtype=torch.float64, device="cuda"), torch.empty((K, N), dtype=torch.uint8, device="cuda"))
        for _ in range(3):
            env.rollout(K, out=out)
        arms[dt] = (env, out)
    res = {dt: [] for dt in VARIANTS}
    for b in range(BLOCKS):
        for dt in VARIANTS:
            env, out = arms[dt]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(LAUNCHES[w]):
                env.rollout(K, out=out)
            e1.record()
            torch.cuda.synchronize()
            res[dt].append(e0.elapsed_time(e1) * 1e3 / (LAUNCHES[w] * K))
    for dt in VARIANTS:
        mb = obs_bytes(N, W, H, dt) / 1e6
        print(f"rollout {w} N={N} K={K} {name(dt):5s} obs {mb:8.2f} MB/step  us/step: " + " ".join(f"{x:.2f}" for x in res[dt]),
              flush=True)
    for env, _ in arms.values():
        env.close()
    del arms
    torch.cuda.empty_cache()


def step_host_timing(w, session, steps):
    wl = WORKLOADS[w]
    N, (W, H) = wl["n_envs"], (wl["meta"]["width"], wl["meta"]["height"])
    envs = {dt: make(wl, dt) for dt in VARIANTS}
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 4, (steps, N)).astype(np.int32)
    res = {dt: [] for dt in VARIANTS}
    for b in range(BLOCKS):
        for dt in VARIANTS:
            env = envs[dt]
            if session:  # one resident step server at a time: the other handle's is parked
                assert env.host_session(True)
            for k in range(5):
                env.step_host(acts[k])
            t0 = time.perf_counter()
            for k in range(steps):
                env.step_host(acts[k])
            res[dt].append((time.perf_counter() - t0) * 1e6 / steps)
            if session:
                env.host_session(False)
    threads = {name(dt): envs[dt].host_threads for dt in VARIANTS}
    for dt in VARIANTS:
        mb = obs_bytes(N, W, H, dt) / 1e6
        print(f"step_host {w} N={N} {'session mode 1' if session else 'no session'} {name(dt):5s} obs {mb:8.2f} MB/step  "
              f"host threads {threads[name(dt)]}  us/step: " + " ".join(f"{x:.2f}" for x in res[dt]), flush=True)
    for env in envs.values():
        env.close()
    torch.cuda.empty_cache()


if __name__ == "__main__":
    if not torch.cuda.is_available():
        sys.exit("obs_bits_timing.py needs a CUDA device")
    print(f"card: {card()}", flush=True)
    for w in ("c4", "c5", "c2"):
        rollout_timing(w)
    step_host_timing("c2", True, 2000)
    step_host_timing("c4", False, 50)
