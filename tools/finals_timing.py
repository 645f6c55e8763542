"""Cost of final-state capture (rollout(finals=True)) on the step kernels, capture on and off, against a parent build.

Arms, each in a process of its own (the library is loaded once per process), alternating over --rounds:
  base   the tree given by --base-tree (e.g. a built checkout of the parent commit: its own package and library), capture off
  off    this tree's library, capture off
  on     this tree's library, capture on
Workloads: a C3-like rollout (14x14, 8192 envs, the in-kernel MLP policy, eps 0.1, 64 steps per launch, uint8 obs), a
C4-like rollout (256x256, wind [0.85, (1, 0)], 32 extra ignitions, 1024 envs, ACTION-stream actions, 64 steps per launch):
time per step from CUDA events around --launches launches after --warmup launches; and DQN.learn_batched with
record_maps off / on (14x14 with 4096 envs and 48x48 with 1024 envs, K = 16): time per env-step of one whole call, after a
short warm-up call.  Writes a table to --out and prints it.

    python tools/finals_timing.py --base-tree build_ab/parent --out profiles/r10_finals_timing.txt
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKLOADS = {
    "c3-like mlp 14x14 N=8192": dict(n=8192, meta=dict(width=14, height=14), chunk=64, policy="mlp"),
    "c4-like 256x256 N=1024": dict(n=1024, meta=dict(width=256, height=256, wind=[0.85, (1, 0)], extra_ignitions=32), chunk=64,
                                   policy="stream"),
    "learn_batched 14x14 N=4096 K=16": dict(learn=True, n=4096, W=14, episodes=20000),
    "learn_batched 48x48 N=1024 K=16": dict(learn=True, n=1024, W=48, episodes=1500),
}


def child_learn(wl, capture):
    import torch

    from wildfire_control_python_b200 import DQN, ForestFire
    kw = dict(record_maps=True) if capture else {}  # (a tree without the option runs the off arm only)

    def run(n_ep):
        torch.manual_seed(0)
        ag = DQN(ForestFire(width=wl["W"], height=wl["W"]), verbose=False)
        ag.write_data = lambda: None
        torch.cuda.synchronize()
        t0 = time.time()
        steps = ag.learn_batched(n_ep, n_envs=wl["n"], k_steps=16, seed=0, **kw)
        torch.cuda.synchronize()
        return steps, time.time() - t0, len(ag.logs.get("maps", []))

    run(wl["n"] // 4)
    steps, dt, n_maps = run(wl["episodes"])
    return dict(us_per_step=dt * 1e6 / (steps / wl["n"]), records_per_launch=n_maps)


def child(name: str, capture: bool, launches: int, warmup: int, tree: str) -> dict:
    sys.path.insert(0, tree)
    import numpy as np
    import torch

    from wildfire_control_python_b200 import BatchedForestFire

    wl = WORKLOADS[name]
    if wl.get("learn"):
        return child_learn(wl, capture)
    N, K = wl["n"], wl["chunk"]
    W, H = wl["meta"]["width"], wl["meta"]["height"]
    env = BatchedForestFire(N, auto_reset=True, seed=0, **wl["meta"])
    env.reset()
    if wl["policy"] == "mlp":
        z = np.load(os.path.join(ROOT, "bench_inputs", "c3_policy_sarsa9_14s.npz"))  # (this tree's copy: the same file)
        env.set_policy_mlp(z["kernel1"], z["bias1"], z["kernel2"], z["bias2"], eps=0.1)
    out = (torch.empty((K, N, W, H, 3), dtype=torch.uint8, device="cuda"), torch.empty((K, N), dtype=torch.float64, device="cuda"),
           torch.empty((K, N), dtype=torch.uint8, device="cuda"))
    records = 0

    def one():
        nonlocal records
        if capture:
            res = env.rollout(K, policy=wl["policy"], out=out, finals=True)
            records += len(res[-1])
        else:
            env.rollout(K, policy=wl["policy"], out=out)

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    records = 0
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(launches):
        one()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    return dict(us_per_step=ms * 1e3 / (launches * K), records_per_launch=records / launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-tree", default=None, help="built tree of the comparison build (capture off); omitted: no base arm")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--capture", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--tree", default=ROOT, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        print(json.dumps(child(a.child, bool(a.capture), a.launches, a.warmup, a.tree)))
        return
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    arms = ([("base", os.path.abspath(a.base_tree), 0)] if a.base_tree else []) + [("off", ROOT, 0), ("on", ROOT, 1)]
    res = {}
    for r in range(a.rounds):
        for name in WORKLOADS:
            for arm, tree, cap in arms:
                env = dict(os.environ)
                env.pop("WILDFIRE_B200_LIB", None)
                p = subprocess.run([sys.executable, __file__, "--child", name, "--capture", str(cap), "--launches", str(a.launches),
                                    "--warmup", str(a.warmup), "--tree", tree], capture_output=True, text=True, env=env)
                if p.returncode != 0:
                    raise RuntimeError(f"{name} / {arm} failed:\n{p.stderr[-3000:]}")
                res.setdefault((name, arm), []).append(json.loads(p.stdout.strip().splitlines()[-1]))
    lines = [f"# final-state capture cost; {gpu}; {a.rounds} alternating rounds x {a.launches} launches of 64 steps, CUDA events",
             "| workload | arm | us per step of the batch (each round) | records per launch (learn_batched: maps logged) |",
             "|---|---|---|---|"]
    for name in WORKLOADS:
        for arm, _, _ in arms:
            rs = res[(name, arm)]
            lines.append(f"| {name} | {arm} | {' / '.join(f'{x['us_per_step']:.2f}' for x in rs)} | "
                         f"{rs[-1]['records_per_launch']:.1f} |")
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
