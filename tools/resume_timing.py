"""Cost of checkpoints in the training loops (needs a CUDA device).

- checkpoint size and the time of a stop and a resume for DQN.learn_batched at 14x14 with N = 4096 and at 48x48 with
  N = 1024 (K = 16), and for a 32-learner learn_population at 14x14 (64 envs each): each run is stopped after one launch
  (time_limit=0), then resumed and stopped twice more.  "save" is the whole stop, from reading the env state to the
  renamed file; "write" the part inside the file write (serialise, fsync, rename); "load" reading the file back with its
  fingerprint check; "restore" the env's set_state and the replay ring's copy to the device.
- the training rate with checkpoint=None against the parent commit's agents.py (--parent FILE, e.g.
  ``git show HEAD~1:wildfire_control_python_b200/agents.py > build_ab/parent_agents.py``), both on this library, arms
  alternating, with a check that both compute the same weights and step counts.
Prints the card's name and power limit read in the same run.

    python tools/resume_timing.py [--parent FILE] [--out FILE] [--quick]     (default out: profiles/r09_resume_timing.txt)
"""
import argparse
import importlib.util
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from wildfire_control_python_b200 import agents as A  # noqa: E402
from wildfire_control_python_b200.batched import BatchedForestFire  # noqa: E402
from wildfire_control_python_b200.compat import get_name  # noqa: E402
from wildfire_control_python_b200.constants import make_metadata  # noqa: E402


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

    def __init__(self, W):
        self.METADATA = make_metadata(width=W, height=W)
        self.n_actions, self.DEBUG, self.get_name = int(self.METADATA["n_actions"]), 1, get_name
        self.W = _World(W, W)


def agents(mod, W, M, out):
    ags = []
    for j in range(M):
        torch.manual_seed(j)
        ag = mod.DQN(_Sim(W), verbose=False, device="cuda")
        ag.out_dir = out
        ags.append(ag)
    return ags


class Clock:
    """Timers around the checkpoint steps of agents.py (what each one covers: the module docstring)."""

    def __init__(self):
        self.t = {k: [] for k in ("save", "write", "load", "restore")}
        self.start = {}
        self._orig = []

    def _wrap(self, owner, name, start=None, stop=None):
        fn = getattr(owner, name)
        self._orig.append((owner, name, fn))

        def wrapped(*args, **kwargs):
            if start:
                self.start[start] = time.perf_counter()
            out = fn(*args, **kwargs)
            if stop:
                torch.cuda.synchronize()
            for k in stop or ():
                if k != "load" or out is not None:  # a load without a file is a fresh start
                    self.t[k].append(time.perf_counter() - self.start[k])
            return out
        setattr(owner, name, wrapped)

    def __enter__(self):
        self._wrap(A, "_env_state", start="save")  # the first thing a stop reads
        self._wrap(A._RunCheckpoint, "save", start="write", stop=("write", "save"))
        self._wrap(A._RunCheckpoint, "load", start="load", stop=("load",))
        self._wrap(BatchedForestFire, "set_state", start="restore")
        self._wrap(A._PackedReplayRing, "load_state_dict", stop=("restore",))
        return self

    def __exit__(self, *exc):
        for owner, name, fn in reversed(self._orig):
            setattr(owner, name, fn)


def checkpoint_costs(label, run, tmp):
    path = os.path.join(tmp, "run.ckpt")
    with Clock() as c:
        for _ in range(3):
            assert run(path) is None
    size = os.path.getsize(path)
    ms = lambda xs: " ".join(f"{x * 1e3:.0f}" for x in xs)  # noqa: E731
    os.remove(path)
    return (f"{label}: checkpoint {size} bytes ({size / 1e6:.1f} MB); save {ms(c.t['save'])} ms (write {ms(c.t['write'])}); "
            f"load {ms(c.t['load'])} ms; restore {ms(c.t['restore'])} ms")


def weights(ags):
    return [b"".join(p.detach().cpu().numpy().tobytes() for p in a.model.parameters()) for a in ags]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="the parent commit's wildfire_control_python_b200/agents.py")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_resume_timing.txt"))
    ap.add_argument("--quick", action="store_true", help="small sizes and one round (a smoke run of the script)")
    args = ap.parse_args()
    q = args.quick
    lines = [f"card: {card()}"]
    print(lines[0], flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        for W, N in ((14, 4096), (48, 1024)):
            N = 256 if q else N
            lines.append(checkpoint_costs(
                f"DQN learn_batched {W}x{W} N={N} K=16",
                lambda path: agents(A, W, 1, tmp)[0].learn_batched(10**6, n_envs=N, k_steps=16, checkpoint=path, time_limit=0),
                tmp))
            print(lines[-1], flush=True)
        M = 4 if q else 32
        lines.append(checkpoint_costs(
            f"DQN learn_population {M} learners 14x14 64 envs each K=16",
            lambda path: A.learn_population(agents(A, 14, M, tmp), 10**5, envs_per_learner=64, k_steps=16, checkpoint=path,
                                            time_limit=0),
            tmp))
        print(lines[-1], flush=True)

        if not args.parent:
            lines.append("training rate against the parent commit: not measured (no --parent)")
        else:
            spec = importlib.util.spec_from_file_location("wildfire_control_python_b200._parent_agents", args.parent)
            parent = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(parent)
            n_b, n_p, M = (20000, 300, 4) if q else (400000, 3000, 32)

            def batched(mod, n):
                ags = agents(mod, 14, 1, tmp)
                return ags, [ags[0].learn_batched(n, n_envs=4096, k_steps=16, seed=1)]

            def population(mod, n):
                ags = agents(mod, 14, M, tmp)
                return ags, mod.learn_population(ags, n, envs_per_learner=64, k_steps=16, seed=1)

            work = {f"DQN learn_batched 14x14 N=4096 K=16, {n_b} episodes": batched,
                    f"DQN learn_population {M} learners 14x14 64 envs each K=16, {n_p} episodes each": population}
            for (label, fn), n in zip(work.items(), (n_b, n_p)):
                for mod in (A, parent):  # warm-up
                    fn(mod, max(n // 20, 50))
                rates = {"this commit": [], "parent": []}
                results = {}
                for _ in range(1 if q else 3):
                    for arm, mod in (("this commit", A), ("parent", parent)):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        ags, steps = fn(mod, n)
                        torch.cuda.synchronize()
                        rates[arm].append(sum(steps) / (time.perf_counter() - t0))
                        results[arm] = (steps, weights(ags))
                same = results["this commit"] == results["parent"]
                cols = "; ".join(f"{arm} " + " ".join(f"{r:.3g}" for r in rs) for arm, rs in rates.items())
                lines.append(f"{label}, checkpoint=None: {cols} env-steps/s (arms alternating); same weights and steps: {same}")
                print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
