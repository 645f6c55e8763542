"""Timing of the learner paths (needs a CUDA device): microseconds per replay of the torch fit_batch loop against
wf_replay_fit (DQN.fit_batches_fused) at n_replays = 1, 64 and 1024 for DQN and DQN_BOTH at 14x14, B = 32; env-steps/s and
replays/s of learn_batched at N = 4096, K = 16; episodes/s of the single-env learn() loop.  Prints the card's name and power
limit read in the same run.

    python tools/learn_timing.py [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from wildfire_control_python_b200 import ForestFire, agents as A, pack_obs, unpack_obs  # noqa: E402


def random_replays(ag, n_frames, n, seed):
    """n transitions over n_frames random packed observations (about a third of the bits set, like a real map)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    W, H = ag.obs_shape[0], ag.obs_shape[1]
    frames = pack_obs((torch.rand((n_frames, W, H, 3), device="cuda", generator=g) < 0.35).to(torch.uint8))
    rows = lambda: torch.randint(0, n_frames, (n,), device="cuda", generator=g)  # noqa: E731
    acts = lambda: torch.randint(0, ag.action_size, (n,), device="cuda", generator=g)  # noqa: E731
    return (frames, rows(), rows(), acts(), acts(), torch.randn((n,), device="cuda", generator=g) * 3,
            torch.rand((n,), device="cuda", generator=g) < 0.1)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    args = ap.parse_args()
    lines = [f"card: {card()}"]
    W, B = 14, 32
    for name in ("DQN", "DQN_BOTH"):
        torch.manual_seed(0)
        ag = getattr(A, name)(ForestFire(width=W, height=W, seed=0), verbose=False)
        frames, s, sp, a, ap_, r, d = random_replays(ag, 4096, 1024 * B, seed=1)
        su = unpack_obs(frames, W, W, s[:B], torch.uint8)
        spu = unpack_obs(frames, W, W, sp[:B], torch.uint8)
        batch = (su, a[:B], r[:B], spu, ap_[:B], d[:B])
        t = timed(lambda: ag.fit_batch(batch), 200)
        lines.append(f"{name} {W}x{W} B={B} torch fit_batch: {t * 1e6:.1f} us per replay")
        for n in (1, 64, 1024):
            t = timed(lambda: ag.fit_batches_fused(frames, s[:n * B], sp[:n * B], a[:n * B], ap_[:n * B], r[:n * B],
                                                   d[:n * B], n), max(3, 2048 // n))
            lines.append(f"{name} {W}x{W} B={B} wf_replay_fit n_replays={n}: {t / n * 1e6:.2f} us per replay")
    with tempfile.TemporaryDirectory() as tmp:
        for name in ("DQN", "DQN_BOTH"):
            sim = ForestFire(width=W, height=W, seed=3)
            ag = getattr(A, name)(sim, verbose=False)
            ag.out_dir = tmp
            ag.learn_batched(500, n_envs=4096, k_steps=16, seed=0)  # warm-up (module loads, allocations)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            steps = ag.learn_batched(100000, n_envs=4096, k_steps=16, seed=1)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            launches = steps // (4096 * 16)
            lines.append(f"{name} learn_batched N=4096 K=16 B={B}: {steps / dt:.3g} env-steps/s, {launches * 16 / dt:.3g} "
                         f"replays/s ({steps} env-steps, {launches} launches in {dt:.2f} s)")
            ag2 = getattr(A, name)(ForestFire(width=W, height=W, seed=3), verbose=False)
            ag2.out_dir = tmp
            t0 = time.perf_counter()
            ag2.learn(20)
            lines.append(f"{name} learn() single env: {20 / (time.perf_counter() - t0):.3g} episodes/s")
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
