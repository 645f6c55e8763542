"""Timing of the in-kernel Q-network on the tile family (grids larger than 32x32; needs a CUDA device).

- microseconds per step of rollouts with K = 16 steps per launch and packed observations, the stream, walk and mlp
  (hidden 50, eps 0.1) policies alternating, at 48x48 x 4096 envs, 64x64 x 2048, 128x128 x 512 and C4 (256x256 x 1024,
  bench.py's workload); with the mean step of the running episodes and the mean number of burning cells at the end, since
  the policy pass's cost grows with the fire and fm_inf cells;
- episodes/s of DQN.evaluate_batched in the kernel against the torch path at 48x48 and 64x64;
- env-steps/s and replays/s of DQN.learn_batched at 48x48 (replays as torch fit_batch calls on these grids);
- microseconds per set_policy_mlp_dev call (the refresh learn_batched queues before every launch) at 48x48, 128x128 and
  256x256: its all-free base is a float64 sum over W*H cells, one thread per hidden unit.
Prints the card's name and power limit read in the same run.

    python tools/tile_policy_timing.py [--out FILE] [--quick]
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import WORKLOADS  # noqa: E402
from wildfire_control_python_b200 import BatchedForestFire, ForestFire, _lib, agents as A  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def glorot_net(W, H, n_actions, hidden=50, seed=0):
    rng = np.random.default_rng(seed)
    n_in = W * H * 3
    lim1, lim2 = np.sqrt(6.0 / (n_in + hidden)), np.sqrt(6.0 / (hidden + n_actions))
    return [x.astype(np.float32) for x in (rng.uniform(-lim1, lim1, (n_in, hidden)), np.zeros(hidden),
                                           rng.uniform(-lim2, lim2, (hidden, n_actions)), np.zeros(n_actions))]


def step_times(name, N, meta, rounds, launches):
    W, H, K = meta["width"], meta["height"], 16
    env = BatchedForestFire(N, obs_dtype="bits", auto_reset=True, seed=0, **meta)
    env.set_policy_mlp(*glorot_net(W, H, env.n_actions), eps=0.1)
    env.reset()
    out = (torch.empty((K, N, env.obs_words), dtype=torch.int32, device="cuda"),
           torch.empty((K, N), dtype=torch.float64, device="cuda"), torch.empty((K, N), dtype=torch.uint8, device="cuda"))
    pols = ("stream", "walk", "mlp")
    for _ in range(4):  # warm-up: module loads, and fires that have burned a while
        for p in pols:
            env.rollout(K, policy=p, out=out)
    res = {p: [] for p in pols}
    for _ in range(rounds):
        for p in pols:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                env.rollout(K, policy=p, out=out)
            e1.record()
            torch.cuda.synchronize()
            res[p].append(e0.elapsed_time(e1) * 1e3 / (launches * K))
    sc = env.get_state()["scalars"].double()
    running = sc[:, _lib.S_RUNNING] != 0
    t_mean = float(sc[running, _lib.S_T].mean()) if running.any() else 0.0
    burning = float(sc[:, _lib.S_N_BURNING].mean())
    env.close()
    cols = "  ".join(f"{p} " + " ".join(f"{v:.2f}" for v in res[p]) for p in pols)
    return (f"{name} ({W}x{H} x {N} envs, K={K}, bits): {cols} us/step; mlp / walk = "
            f"{np.median(res['mlp']) / np.median(res['walk']):.2f}; at the end: running episodes at step {t_mean:.0f} on "
            f"average, {burning:.0f} burning cells per env")


def refresh_time(W, H, reps):
    env = BatchedForestFire(8, auto_reset=True, seed=0, width=W, height=H)
    k1, b1, k2, b2 = (torch.from_numpy(x).cuda() for x in glorot_net(W, H, env.n_actions))
    w1, w2 = k1.t().contiguous(), k2.t().contiguous()
    env.set_policy_mlp_dev(w1, b1, w2, b2, eps=0.1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        env.set_policy_mlp_dev(w1, b1, w2, b2, eps=0.1)
    e1.record()
    torch.cuda.synchronize()
    env.close()
    return e0.elapsed_time(e1) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes and few repetitions (a smoke run of the script)")
    args = ap.parse_args()
    q = args.quick
    lines = [f"card: {card()}"]
    print(lines[0], flush=True)
    c4 = WORKLOADS["c4"]
    sizes = [("48x48", 4096, dict(width=48, height=48)), ("64x64", 2048, dict(width=64, height=64)),
             ("128x128", 512, dict(width=128, height=128)), ("C4", c4["n_envs"], c4["meta"])]
    for name, N, meta in sizes:
        lines.append(step_times(name, 64 if q else N, meta, 1 if q else 3, 2 if q else 20))
        print(lines[-1], flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        for W in (48, 64):
            torch.manual_seed(0)
            ag = A.DQN(ForestFire(width=W, height=W, seed=0), verbose=False)
            ag.out_dir = tmp
            N = 64 if q else 2048
            rates = {}
            for rep in range(2):  # the first round warms up
                for in_kernel in (True, False):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    rets, _ = ag.evaluate_batched(n_envs=N, eps=0.1, seed=rep, in_kernel=in_kernel)
                    rates[in_kernel] = len(rets) / (time.perf_counter() - t0)
            lines.append(f"evaluate_batched {W}x{W} N={N} eps=0.1: in-kernel {rates[True]:.3g} episodes/s, torch path "
                         f"{rates[False]:.3g} episodes/s ({rates[True] / rates[False]:.1f}x)")
            print(lines[-1], flush=True)
        W, N, K = 48, (64 if q else 1024), 16
        torch.manual_seed(0)
        ag = A.DQN(ForestFire(width=W, height=W, seed=3), verbose=False)
        ag.out_dir = tmp
        ag.learn_batched(50 if q else 300, n_envs=N, k_steps=K, seed=0)  # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        steps = ag.learn_batched(100 if q else 3000, n_envs=N, k_steps=K, seed=1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        launches = steps // (N * K)
        lines.append(f"DQN learn_batched {W}x{W} N={N} K={K} B={ag.METADATA['batch_size']}: {steps / dt:.3g} env-steps/s, "
                     f"{launches * K / dt:.3g} replays/s (torch fit_batch; {steps} env-steps, {launches} launches in {dt:.2f} s)")
        print(lines[-1], flush=True)
    for W in (48, 128, 256):
        lines.append(f"set_policy_mlp_dev {W}x{W} hidden 50: {refresh_time(W, W, 2 if q else 20):.1f} us per refresh")
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
