"""Timing of population training (needs a CUDA device): aggregate replays/s of wf_replay_fit_many with M = 1 ... 32
learners in one launch against M back-to-back wf_replay_fit calls (14x14, B = 32, R = 256 replays per learner, DQN and
DQN_BOTH shapes), and the wall time of learn_population with 8 agents against 8 sequential learn_batched runs of the same
configuration.  Prints the card's name and power limit read in the same run.

    python tools/population_timing.py [--out FILE]     (default profiles/r05_population_timing.txt)
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from wildfire_control_python_b200 import _lib, agents as A, pack_obs  # noqa: E402
from wildfire_control_python_b200.compat import ForestFire  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def fit_setup(M, W, hid, A_, dueling, B, R, seed):
    """M learners' random state and R * B random transitions each over one shared table of 4096 random frames."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    P = _lib.mlp_param_count(W, W, hid, A_, dueling)
    frames = pack_obs((torch.rand((4096, W, W, 3), device="cuda", generator=g) < 0.35).to(torch.uint8))
    n, keep, desc = R * B, [], (_lib.WfFitLearner * M)()
    for j in range(M):
        st = [torch.randn(P, device="cuda", generator=g) * 0.05, torch.randn(P, device="cuda", generator=g) * 0.05,
              torch.zeros(P, device="cuda"), torch.zeros(P, device="cuda")]
        data = [torch.randint(0, 4096, (n,), device="cuda", generator=g), torch.randint(0, 4096, (n,), device="cuda", generator=g),
                torch.randint(0, A_, (n,), device="cuda", generator=g, dtype=torch.int32),
                torch.randint(0, A_, (n,), device="cuda", generator=g, dtype=torch.int32),
                torch.randn(n, device="cuda", generator=g), (torch.rand(n, device="cuda", generator=g) < 0.1).to(torch.uint8)]
        keep.append(st + data)
        hp = _lib.WfFitParams(gamma=0.999, lr=0.005, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipvalue=1.0, adam_t=0,
                              target_every=20, phase=20)
        desc[j] = _lib.WfFitLearner(*[t.data_ptr() for t in st], *[t.data_ptr() for t in data], None, hp)
    sh = _lib.WfMlpShape(width=W, height=W, hidden=hid, n_actions=A_, dueling=dueling, batch=B)
    return sh, desc, frames, keep


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_population_timing.txt"))
    args = ap.parse_args()
    L = _lib.lib()
    lines = [f"card: {card()}"]
    W, B, R = 14, 32, 256
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for name, dueling in (("DQN", 0), ("DQN_BOTH", 1)):
        for M in (1, 2, 4, 8, 16, 32):
            sh, desc, frames, keep = fit_setup(M, W, 50, 4, dueling, B, R, seed=M)
            many = lambda: _lib.check(L.wf_replay_fit_many(C.byref(sh), M, desc, R, frames.data_ptr(), 4096, stream))  # noqa: E731

            def apart():
                for j in range(M):
                    _lib.check(L.wf_replay_fit_many(C.byref(sh), 1, C.byref(desc[j]), R, frames.data_ptr(), 4096, stream))
            reps = 3
            t_many, t_apart = [], []
            for _ in range(2):  # alternating
                t_many.append(timed(many, reps))
                t_apart.append(timed(apart, reps))
            tm, ta = min(t_many), min(t_apart)
            lines.append(f"{name} {W}x{W} B={B} R={R} M={M:2d}: wf_replay_fit_many {M * R / tm:8.0f} replays/s "
                         f"({tm * 1e3:7.1f} ms per launch) | {M} x wf_replay_fit {M * R / ta:8.0f} replays/s "
                         f"({ta * 1e3:7.1f} ms) | x{ta / tm:.2f}")
            del keep
    # learn_population against sequential learn_batched: 8 DQN agents, 10x10, 64 envs each, K = 16, R = 256
    M, G, K, R, n_ep = 8, 64, 16, 256, 1000
    with tempfile.TemporaryDirectory() as tmp:
        def agents():
            out = []
            for j in range(M):
                torch.manual_seed(j)
                ag = A.DQN(ForestFire(width=10, height=10, seed=0), verbose=False)
                ag.out_dir = tmp
                out.append(ag)
            return out
        A.learn_population(agents()[:2], 50, envs_per_learner=G, k_steps=K, replays_per_launch=R, seed=0)  # warm-up
        for rep in range(2):
            ags = agents()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            steps = A.learn_population(ags, n_ep, envs_per_learner=G, k_steps=K, replays_per_launch=R, seed=rep)
            torch.cuda.synchronize()
            t_pop = time.perf_counter() - t0
            ags = agents()
            t0 = time.perf_counter()
            for j, ag in enumerate(ags):
                ag.learn_batched(n_ep, n_envs=G, k_steps=K, replays_per_launch=R, seed=rep, replay_seed=rep + j)
            torch.cuda.synchronize()
            t_seq = time.perf_counter() - t0
            lines.append(f"DQN 10x10 {M} agents x {n_ep} episodes, {G} envs each, K={K}, R={R}: learn_population "
                         f"{t_pop:.2f} s ({sum(steps)} env-steps) | {M} sequential learn_batched {t_seq:.2f} s | "
                         f"x{t_seq / t_pop:.2f}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
