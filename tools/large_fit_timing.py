"""Timing of wf_replay_fit_large, the replay kernel of grids larger than 32x32 (needs a CUDA device).

- microseconds per replay of DQN and DQN_BOTH (hidden 50, B = 32) at 48x48, 128x128 and 256x256: the torch fit_batch loop
  (unpacking each minibatch to float32, as learn_batched did on these grids before the kernel) against
  wf_replay_fit_large called through the C ABI with n_replays = 1 (64 calls) and 64 (one call), arms alternating; with
  the first layer's Adam bytes per replay (24 * units * n_in, plus 4 * units * n_in on a target sync) and their share of
  the 7.7 TB/s HBM bound, and whether the model, target and moments fit the 126 MB L2;
- 14x14 and 32x32: wf_replay_fit against wf_replay_fit_large (n_replays 64, DQN and DQN_BOTH, B = 32);
- env-steps/s and replays/s of DQN.learn_batched at 48x48, N = 1024, K = 16, B = 32.
Prints the card's name and power limit read in the same run.

    python tools/large_fit_timing.py [--out FILE] [--quick]
"""
import argparse
import ctypes
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from wildfire_control_python_b200 import ForestFire, _lib, agents as A, pack_obs, unpack_obs  # noqa: E402
from wildfire_control_python_b200.batched import _ptr  # noqa: E402
from wildfire_control_python_b200.compat import get_name  # noqa: E402
from wildfire_control_python_b200.constants import make_metadata  # noqa: E402

HBM = 7.7e12  # bytes/s, B200 data sheet
L2 = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


class _World:
    DEPTH = 3
    agents = []

    def __init__(self, W, H):
        self.WIDTH, self.HEIGHT = W, H


class _Sim:
    """The surface DQN.__init__ reads, without creating environments."""

    def __init__(self, W, H):
        self.METADATA = make_metadata(width=W, height=H)
        self.n_actions, self.DEBUG, self.get_name = int(self.METADATA["n_actions"]), 1, get_name
        self.W = _World(W, H)


class Case:
    """A warmed agent, R * B random transitions over 4 * B frames, and flat copies of its state for the C ABI."""

    def __init__(self, name, W, B, R, seed=0):
        torch.manual_seed(seed)
        self.ag = getattr(A, name)(_Sim(W, W), verbose=False, device="cuda")
        self.W, self.B, self.R = W, B, R
        g = torch.Generator(device="cuda").manual_seed(seed)
        n_frames, n = 4 * B, R * B
        self.frames = pack_obs((torch.rand((n_frames, W, W, 3), device="cuda", generator=g) < 0.35).to(torch.uint8))
        self.s, self.sp = (torch.randint(0, n_frames, (n,), device="cuda", generator=g) for _ in range(2))
        self.a = torch.randint(0, self.ag.action_size, (n,), device="cuda", generator=g, dtype=torch.int32)
        self.ap = torch.randint(0, self.ag.action_size, (n,), device="cuda", generator=g, dtype=torch.int32)
        self.r = torch.randn((n,), device="cuda", generator=g) * 3
        self.d = (torch.rand((n,), device="cuda", generator=g) < 0.1).to(torch.uint8)
        for i in range(3):  # Adam at t > 0
            self.ag.fit_batch(self.batch(i))
        p2v = torch.nn.utils.parameters_to_vector
        ps = list(self.ag.model.parameters())
        st = [self.ag.optimizer.state[p] for p in ps]
        self.flat = [p2v(x).detach().clone() for x in (ps, list(self.ag.target.parameters()), [s["m"] for s in st],
                                                        [s["v"] for s in st])]
        self.loss = torch.empty(R, device="cuda")
        self.units = self.ag.model.dense_1.out_features * (2 if hasattr(self.ag.model, "dense_3") else 1)

    def batch(self, i):
        sl = slice(i * self.B, (i + 1) * self.B)
        W = self.W
        return (unpack_obs(self.frames, W, W, self.s[sl]), self.a[sl].long(), self.r[sl], unpack_obs(self.frames, W, W, self.sp[sl]),
                self.ap[sl].long(), self.d[sl].bool())

    def torch_loop(self, n):
        for i in range(n):
            self.ag.fit_batch(self.batch(i))

    def kernel(self, fn, n_replays, calls):
        ag = self.ag
        g = ag.optimizer.param_groups[0]
        hp = _lib.WfFitParams(gamma=float(ag.gamma), lr=g["lr"], beta_1=g["beta_1"], beta_2=g["beta_2"], epsilon=g["epsilon"],
                              clipvalue=g["clipvalue"], adam_t=3, target_every=int(ag.target_update_freq), phase=7)
        sh = ag._flat_shape(self.B)
        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        P, T, M, V = (_ptr(x) for x in self.flat)
        for c in range(calls):
            i = c * n_replays * self.B
            _lib.check(fn(ctypes.byref(sh), ctypes.byref(hp), n_replays, P, T, M, V, _ptr(self.frames), self.frames.shape[0],
                          _ptr(self.s[i:]), _ptr(self.sp[i:]), _ptr(self.a[i:]), None, _ptr(self.r[i:]), _ptr(self.d[i:]),
                          _ptr(self.loss), stream))


def timed(f):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--quick", action="store_true", help="small sizes and few repetitions (a smoke run of the script)")
    args = ap.parse_args()
    q = args.quick
    L = _lib.lib()
    lines = [f"card: {card()}"]
    print(lines[0], flush=True)
    R, B, rounds = 64, 32, (1 if q else 3)
    for W in ((48,) if q else (48, 128, 256)):
        for name in ("DQN", "DQN_BOTH"):
            c = Case(name, W, B, R)
            arms = {"torch fit_batch loop": lambda: c.torch_loop(R),
                    "wf_replay_fit_large n_replays=1": lambda: c.kernel(L.wf_replay_fit_large, 1, R),
                    "wf_replay_fit_large n_replays=64": lambda: c.kernel(L.wf_replay_fit_large, R, 1)}
            for f in arms.values():  # warm-up: module loads, cuBLAS algorithm choice, the memory pool
                f()
            res = {k: [] for k in arms}
            for _ in range(rounds):
                for k, f in arms.items():
                    res[k].append(timed(f) / R)
            n_in = W * W * 3
            by = 24 * c.units * n_in + 4 * c.units * n_in / c.ag.target_update_freq
            state = 16 * c.units * n_in
            best = min(res["wf_replay_fit_large n_replays=64"])
            where = (f"model + target + m + v = {state / 1e6:.1f} MB fit the 126 MB L2, so HBM does not bound it"
                     if state <= L2 else f"model + target + m + v = {state / 1e6:.0f} MB exceed the L2: HBM-bound")
            cols = "; ".join(f"{k} " + " ".join(f"{v:.1f}" for v in res[k]) for k in arms)
            lines.append(f"{name} {W}x{W} B={B} hidden 50: {cols} us/replay; speed-up at n_replays=64 "
                         f"{np.median(res['torch fit_batch loop']) / np.median(res['wf_replay_fit_large n_replays=64']):.1f}x; "
                         f"first-layer Adam bytes/replay {by / 1e6:.2f} MB -> {by / HBM * 1e6:.1f} us at 7.7 TB/s, "
                         f"{by / HBM * 1e6 / best:.0%} of that bound reached; {where}")
            print(lines[-1], flush=True)
            del c
            torch.cuda.empty_cache()
    for W in ((14,) if q else (14, 32)):
        for name in ("DQN", "DQN_BOTH"):
            c = Case(name, W, B, R)
            arms = {"wf_replay_fit": lambda: c.kernel(L.wf_replay_fit, R, 1),
                    "wf_replay_fit_large": lambda: c.kernel(L.wf_replay_fit_large, R, 1)}
            for f in arms.values():
                f()
            res = {k: [] for k in arms}
            for _ in range(rounds * 3):
                for k, f in arms.items():
                    res[k].append(timed(f) / R)
            cols = "; ".join(f"{k} " + " ".join(f"{v:.1f}" for v in res[k]) for k in arms)
            lines.append(f"{name} {W}x{W} B={B} n_replays={R}: {cols} us/replay")
            print(lines[-1], flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        W, N, K = 48, (64 if q else 1024), 16
        torch.manual_seed(0)
        ag = A.DQN(ForestFire(width=W, height=W, seed=3), verbose=False)
        ag.out_dir = tmp
        ag.learn_batched(50 if q else 300, n_envs=N, k_steps=K, seed=0)  # warm-up
        for rep in range(1 if q else 2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            steps = ag.learn_batched(100 if q else 3000 * (1 + rep), n_envs=N, k_steps=K, seed=1 + rep)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            launches = steps // (N * K)
            lines.append(f"DQN learn_batched {W}x{W} N={N} K={K} B={ag.METADATA['batch_size']}: {steps / dt:.3g} env-steps/s, "
                         f"{launches * K / dt:.3g} replays/s (wf_replay_fit_large; {steps} env-steps, {launches} launches "
                         f"in {dt:.2f} s); r07 with torch fit_batch replays: 9.99e+05 env-steps/s, 975 replays/s")
            print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
