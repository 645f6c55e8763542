#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched fire-spread step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE ForestFire.step over the whole batch of the workload (default c2 = BASELINE.json
configs[1]: 4096 envs of 14x14 per GPU, Logs/14-sized constants, actions from the shared Philox
ACTION stream, auto-reset on done).  Prints one JSON line (rank 0); DESIGN.md section 5 explains
every field.

  value         device-resident throughput: exactly K = --steps timed steps, launched `launch.steps_per_launch` steps
                at a time (the last launch shorter when that does not divide K), after `warmup` un-timed steps (W
                rounded up to whole launches, the last of them queued in front of the first event so that the GPU
                never idles inside the region); CUDA events on the launching stream, max over ranks.  Obs/reward/done
                of EVERY step are written to HBM.  ms_per_step = region / K.  Every other timed region of the line
                (e2e, per_step_launch, secondary, via_torch) is K steps too, each behind un-timed warm-up steps.
  e2e           the same metric through the host-buffer C-ABI call (wf_step_host, page-locked host buffers): per
                step actions H2D, step, obs + reward + done D2H, all inside the timed region; wall clock over
                K steps.  `session` says whether the handle's persistent step-server kernel was used.
  per_step_launch   one wf_step per step with device-resident actions (Python loop, and CUDA graph).
  roofline      dominant kernel.  `achieved` / `frac` count the bytes THIS layout must move per env-step
                (`bytes_per_unit`); `survey_accounting` is the same throughput in SURVEY.md 8(d)'s byte-per-cell
                accounting (15 B per cell-update); `traffic` = DRAM bytes per launch from the committed ncu capture.
  cpu_baseline  the C oracle (a port of the reference step, oracle/) on ONE host core, bounded sample, plus
                `python_ref`: the UNMODIFIED Python reference in os.cpu_count() processes (oracle/ref_bench.py).
  secondary     (default workload only) c4 (256x256 stencil stress), c5 (1024x1024, 64 envs/GPU) and c3 (8192
                envs/GPU, the reference's DQN network in the loop), each measured the same way with its own roofline.
--impl reference times the reference's own Python step (oracle/_ref snapshot or the reference tree) on all host
cores, and the C port beside it; its line carries "impl": "reference".

--dump-outputs DIR writes, after the timed steps, what the timed path returned for its last step: per workload
<workload>_reward.npy (float64) and <workload>_done.npy (float32) of every env and <workload>_obs.npy (float32) of the
envs listed in <workload>_obs_env_index.npy (all of them, or a fixed seeded sample so that the files stay within
64 MiB in all).  The step count is fixed by --warmup / --steps and every input is seeded, so two builds of the
project run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: 14x14 (Logs/14-sized constants) batched 4096 envs, random actions
    # 256 steps per launch: the ~15 us a launch costs beyond its steps (launch gap, state load/store, table set-up,
    # the tail of the slowest warp) falls from 9 % of a 64-step launch to 2.5 % (tools/ab_rollout.py, r01)
    "c2": dict(n_envs=4096, meta=dict(width=14, height=14), chunk=256,
               desc="14x14 Logs/14-sized constants, 4096 envs/GPU, ACTION-stream random actions, auto-reset"),
    # configs[2]: 14x14 batched 65536 envs (8192 per GPU on 8 GPUs) with a DQN-policy rollout:
    # Flatten -> Dense(50, sigmoid) -> Dense(4) (DQN.py:209-233), epsilon-greedy 0.1
    "c3": dict(n_envs=8192, meta=dict(width=14, height=14), chunk=64, policy=True,
               desc="14x14 Logs/14-sized constants, 8192 envs/GPU, DQN MLP policy 588-50-4 in the loop (eps 0.1), auto-reset"),
    # configs[3]: 256x256, 1024 envs, wind enabled, multi-ignition stress of the stencil
    # 64 steps per launch: 45.9 / 45.1 / 44.8 / 44.5 us per step with 16 / 32 / 64 / 128 (r02; c5 does not care: 86.4 ... 85.6)
    "c4": dict(n_envs=1024, meta=dict(width=256, height=256, wind=[0.85, (1, 0)], extra_ignitions=32), chunk=64,
               desc="256x256, wind [0.85,(1,0)], 32 extra ignitions, 1024 envs/GPU, ACTION-stream actions, auto-reset"),
    # configs[4]: 1024x1024 grid, 64 envs per GPU
    "c5": dict(n_envs=64, meta=dict(width=1024, height=1024, extra_ignitions=256), chunk=16,
               desc="1024x1024, no wind, 256 extra ignitions, 64 envs/GPU, ACTION-stream actions, auto-reset"),
}
BYTES_PER_CELL_UPDATE = 15  # SURVEY.md 8(d): 6 B state read + 6 B state write + 3 B uint8 observation
CPU_BASELINE_SECONDS = 10.0  # bounded sample of the cpu_baseline (port) leg
PYTHON_REF_STEPS = 20        # bounded sample of the python_ref leg: the workload's envs (at most 4096) x this many steps
DUMP_BYTES = 64 << 20        # --dump-outputs writes at most this much in all
C3_POLICY = os.path.join(ROOT, "bench_inputs", "c3_policy_sarsa9_14s.npz")


def workload_config(name):
    """The `config` object of the JSON line: a function of the workload only, identical in both arms."""
    wl = WORKLOADS[name]
    return {"workload": f"{name}: {wl['desc']}", "grid": [wl["meta"]["width"], wl["meta"]["height"]], "envs_per_gpu": wl["n_envs"]}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def launch_sizes(steps: int, chunk: int) -> list:
    """`steps` steps as launches of `chunk` steps, the last one shorter when `chunk` does not divide `steps`."""
    return [chunk] * (steps // chunk) + ([steps % chunk] if steps % chunk else [])


def warmup_steps(W: int, chunk: int) -> int:
    """The un-timed steps in front of a timed region: W rounded up to whole launches, at least one."""
    return max(1, -(-W // chunk)) * chunk


def last_step_outputs(obs, reward, done, budget: int) -> dict:
    """What a caller of the timed path received for its last step, as float32 / float64 numpy arrays of at most
    `budget` bytes: reward and done of every env, and the observation of as many envs as fit (a fixed seeded sample
    when not all of them do, listed in obs_env_index)."""
    import numpy as np
    import torch
    N = reward.shape[0]
    keep = min(N, max(1, (budget - 20 * N) // (obs[0].numel() * 4)))  # 20 B per env: reward, done, index
    idx = np.arange(N) if keep == N else np.sort(np.random.default_rng(0).choice(N, keep, replace=False))
    sel = obs.index_select(0, torch.as_tensor(idx, device=obs.device))
    return {"reward": reward.double().cpu().numpy(), "done": done.float().cpu().numpy(),
            "obs": sel.float().cpu().numpy(), "obs_env_index": idx.astype(np.float64)}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.1)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower() == "active" for r in self.rows)]
        # median over the samples taken under load (the top half of the sorted list: idle samples between legs sit low)
        busy = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def oracle_cfg(meta):
    return dict(seed=0, **meta)


def port_baseline(wl, threads: int, seconds: float):
    """The C port of the reference step (oracle/) on `threads` host threads, bounded to ~`seconds`."""
    from oracle import wf_oracle as wo  # the checker, timed as a CPU baseline (allowed use)
    ob = wo.OracleBatch(oracle_cfg(wl["meta"]), min(wl["n_envs"], 1024 if threads == 1 else 4096), threads)
    t0 = time.perf_counter(); n = ob.step(2); rate = n / (time.perf_counter() - t0)
    steps_cpu = max(1, int(rate * seconds / ob.n_envs))
    t0 = time.perf_counter(); n = ob.step(steps_cpu); dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "env-steps/s", "cores": ob.n_threads, "kind": "port",
            "sample": f"{ob.n_envs} envs x {steps_cpu} steps of the same workload, {ob.n_threads} thread(s), {dt:.1f} s"}


def python_ref_baseline(wl, steps: int, warmup: int, budget_s: float = 60.0):
    """The UNMODIFIED Python reference in os.cpu_count() processes (oracle/ref_bench.py), or None if it is not there."""
    try:
        from oracle import ref_bench
        if not ref_bench.available():
            return None
        cores = os.cpu_count() or 1
        probe = ref_bench.run(wl["meta"], cores, 10, 2, cores)
        n_envs = int(max(cores, min(wl["n_envs"], probe["value"] * budget_s / max(1, steps + warmup))))
        r = ref_bench.run(wl["meta"], n_envs, steps, warmup, cores)
        return {"value": r["value"], "unit": "env-steps/s", "cores": r["procs"], "kind": "_ref",
                "sample": f"{r['envs']} of {wl['n_envs']} envs x {steps} steps (+{warmup} warm-up), the reference's own ForestFire.step "
                          f"in {r['procs']} processes, random actions, reset on done, {r['seconds']:.1f} s",
                "source": "oracle/_ref snapshot of the unmodified Simulation/ package (or /root/reference); its A* compiled from "
                          "pyastar/astar.cpp"}
    except Exception as exc:  # a missing snapshot or a broken worker must not take the bench line down
        return {"error": repr(exc)[:300], "kind": "_ref"}


def run_reference(args, wl):
    """The reference's CPU implementation of the path on the box's host cores: the UNMODIFIED Python step when the
    snapshot is there (kind "_ref"), and the C port of it (oracle/, test infrastructure: this is one of the two places
    bench.py may execute it) beside it / instead of it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    W, H = wl["meta"]["width"], wl["meta"]["height"]
    port = port_baseline(wl, cores, min(30.0, 0.5 * (args.steps + args.warmup)))
    py = python_ref_baseline(wl, args.steps, args.warmup)
    main = py if (py and "value" in py) else port
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": main["value"], "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wl["n_envs"] / main["value"],  # what one step over the full batch would take at this rate
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args.workload),
        "cell_updates_per_sec": main["value"] * W * H,
        "cpu_baseline": dict(main, port=port) if main is not port else port,
        "e2e": {"value": main["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": ("value = the reference's own Python ForestFire.step (unmodified, oracle/_ref) on all host cores; "
                 "cpu_baseline.port = the C port of it (oracle/wf_oracle.c, validated step-by-step against the Python reference) "
                 "on all host threads" if main is not port else
                 "C oracle port of Simulation/forest_fire.py + environment.py (validated step-by-step against the Python "
                 "reference); the Python reference snapshot (oracle/_ref) is not present on this box"),
    }
    if py and "error" in py:
        line["python_ref_error"] = py["error"]
    print(json.dumps(line), flush=True)


class Dist:
    def __init__(self, gpus):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world == 1 and gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run --nproc-per-node N")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def timed_region(D: Dist, launch, K: int, chunk: int, W: int):
    """Time exactly K steps of `launch(n)` (n <= chunk steps per call) after warmup_steps(W, chunk) un-timed steps, the
    last `chunk` of them queued in front of the first event.  Returns (ms, n_launches) of the region."""
    torch = D.torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup_steps(W, chunk) // chunk - 1):
        launch(chunk)
    D.barrier()
    launch(chunk)     # un-timed: the GPU is busy when ev0 is reached, so no host launch latency sits in the region
    ev0.record()
    sizes = launch_sizes(K, chunk)
    for n in sizes:
        launch(n)
    ev1.record()
    D.barrier()
    return D.max_over_ranks(ev0.elapsed_time(ev1)), len(sizes)


def measure(D: Dist, name: str, K: int, Wm: int, chunk_arg: int, with_e2e: bool, with_per_step: bool, dump_budget: int = 0):
    """Time workload `name` on this rank's GPU; every rank calls this, results are max-reduced.  dump_budget > 0: keep
    the last timed step's outputs (last_step_outputs) as res["outputs"]."""
    import numpy as np
    torch = D.torch
    from wildfire_control_python_b200 import BatchedForestFire

    wl = WORKLOADS[name]
    dev, rank, world = D.dev, D.rank, D.world
    N, W, H = wl["n_envs"], wl["meta"]["width"], wl["meta"]["height"]
    chunk = max(1, chunk_arg or wl["chunk"])
    env = BatchedForestFire(N, device=dev, auto_reset=True, seed=0, env_id_base=rank * N, **wl["meta"])
    env.reset()
    obs_buf = torch.empty((chunk, N, W, H, 3), dtype=torch.uint8, device=dev)
    rew_buf = torch.empty((chunk, N), dtype=torch.float64, device=dev)
    done_buf = torch.empty((chunk, N), dtype=torch.uint8, device=dev)

    def launch(n):
        env.rollout(n, actions=None, out=(obs_buf[:n], rew_buf[:n], done_buf[:n]))

    launches0 = env.launch_count
    ms_max, n_launch = timed_region(D, launch, K, chunk, Wm)
    res = {"name": name, "wl": wl, "N": N, "W": W, "H": H, "K": K, "warmup": warmup_steps(Wm, chunk), "chunk": chunk,
           "ms": ms_max, "launches": int(n_launch), "launches_total": int(env.launch_count - launches0),
           "value": world * N * K / (ms_max * 1e-3), "obs_mb": obs_buf.numel() / 1e6, "family": env.kernel_family,
           "state_bytes": env.state_bytes_per_env, "tile_geometry": list(env.tile_geometry)}
    if dump_budget:
        last = launch_sizes(K, chunk)[-1] - 1
        res["outputs"] = last_step_outputs(obs_buf[last], rew_buf[last], done_buf[last], dump_budget)

    if with_per_step:
        g = torch.Generator(device=dev).manual_seed(99 + rank)
        acts = torch.randint(0, 4, (K, N), dtype=torch.int32, device=dev, generator=g)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        for k in range(res["warmup"]):
            env.step(acts[k % K])
        ev0.record()
        for k in range(K):
            env.step(acts[k])
        ev1.record()
        D.barrier()
        t2 = D.max_over_ranks(ev0.elapsed_time(ev1))
        per_step = {"value": world * N * K / (t2 * 1e-3), "unit": "env-steps/s", "steps": K, "us_per_step": t2 * 1e3 / K,
                    "issue": "python loop over BatchedForestFire.step, actions resident in HBM"}
        try:  # the same per-step launches replayed from a CUDA graph (no host work between launches)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                env.step(acts[0])
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2, stream=side):
                    for k in range(K):
                        env.step(acts[k])
            torch.cuda.current_stream(dev).wait_stream(side)
            D.barrier()
            g2.replay()  # un-timed, queued in front of the first event
            ev0.record()
            g2.replay()
            ev1.record()
            D.barrier()
            t3 = D.max_over_ranks(ev0.elapsed_time(ev1))
            per_step["cuda_graph"] = {"value": world * N * K / (t3 * 1e-3), "unit": "env-steps/s", "steps": K,
                                      "us_per_step": t3 * 1e3 / K,
                                      "note": "obs written to the same buffer every step (may stay in L2)"}
        except Exception as exc:  # a convenience measurement, never the headline
            per_step["cuda_graph"] = {"error": repr(exc)[:200]}
        res["per_step"] = per_step

    if with_e2e:
        rng = np.random.default_rng(7 + rank)
        host_actions = rng.integers(0, 4, size=(512, N), dtype=np.int32)
        def time_e2e(persistent_obs):
            session = False
            if hasattr(env, "host_session") and not os.environ.get("WF_BENCH_NO_SESSION"):
                session = bool(env.host_session(True, persistent_obs=persistent_obs))
            D.barrier()  # before the warm-up: a synchronise would wait until the resident step server parks
            for k in range(res["warmup"]):
                env.step_host(host_actions[k & 511])
            t0 = time.perf_counter()
            for k in range(K):
                env.step_host(host_actions[k & 511])
            te = D.max_over_ranks(time.perf_counter() - t0)  # each call returns with its results in the host arrays
            if session:
                env.host_session(False)
            return session, te

        session, te = time_e2e(False)
        obs_bytes = N * W * H * 3
        if env.host_threads:  # packed path: one record of ceil(e * W*H*3 / 32) words per e envs (e = 2 if W <= 16 else 1)
            epw = 2 if W <= 16 else 1
            records, rec_words = (N + epw - 1) // epw, (epw * W * H * 3 + 31) // 32
            if session:  # + one status word (reward code, done) per record, four records per 128-byte-aligned CTA block
                d2h = ((records + 3) // 4) * ((4 * (rec_words + 1) + 31) // 32 * 32) * 4
            else:
                d2h = records * rec_words * 4 + N * 8 + N
        else:
            d2h = obs_bytes + N * 8 + N
        res["e2e"] = {"value": world * N * K / te, "unit": "env-steps/s", "h2d_bytes_per_step": N * 4,
                      "d2h_bytes_per_step": d2h, "obs_bytes_delivered_per_step": obs_bytes,
                      "steps": K, "us_per_step": te * 1e6 / K,
                      "host_threads": env.host_threads, "session": session,
                      "api": ("wf_step_host, page-locked host buffers: actions/reward/done zero-copy; observation sent as a bit "
                              "stream and expanded to the caller's uint8 [N][W][H][3] array by the library's host threads"
                              + ("; resident step-server kernel (wf_host_session): the kernel polls the tagged actions in mapped "
                                 "host memory and raises a completion flag there, no launch and no stream synchronise per step" if session else "")
                              if env.host_threads else
                              "wf_step_host, page-locked host buffers (actions/reward/done zero-copy, obs one DMA copy)")}
        if session and not os.environ.get("WF_BENCH_NO_PERSISTENT"):
            # The same call with wf_host_session mode 2 (a vectorised Gym env's copy=False convention: step_host hands out
            # the same array every call and the caller does not write to it): only the elements that changed cross PCIe and
            # are patched in place.  Reported beside the headline, which re-delivers the whole array every step.
            _, tp = time_e2e(True)
            ctas = ((N + epw - 1) // epw + 3) // 4
            res["e2e"]["persistent_obs"] = {
                "value": world * N * K / tp, "unit": "env-steps/s", "us_per_step": tp * 1e6 / K,
                "d2h_bytes_per_step": ctas * 128,
                "note": "wf_host_session(env, 2): one 128-byte change-list block per 8 envs + the full record (160 B) of every "
                        "pair of envs with more than 13 changed elements (about 4 % of them per step: resets, large fire ticks); "
                        "the array is complete and equal to the headline's after every call (tests/test_host_api_gpu.py)"}
    res["stats"] = env.stats()
    env.close()
    del obs_buf, rew_buf, done_buf, env
    torch.cuda.empty_cache()
    return res


def load_c3_policy(torch, dev, W, H, n_actions):
    """The policy of configs[2]: a network the REFERENCE trained (Models/14-sized/SARSA9-..., converted to .npz by
    oracle/gen_keras_fixture.py), else fixed-seed random weights of the same architecture (DQN.py:209-233)."""
    import numpy as np
    if os.path.isfile(C3_POLICY) and (W, H) == (14, 14):
        z = np.load(C3_POLICY)
        w1, b1, w2, b2 = (torch.as_tensor(z[k]).to(dev) for k in ("kernel1", "bias1", "kernel2", "bias2"))
        return (w1, b1, w2, b2), "the reference's trained DQN_SARSA network SARSA9-14s-10k-47298m (Keras weights)"
    g = torch.Generator(device=dev).manual_seed(1234)  # same weights on every rank
    w1 = torch.randn(W * H * 3, 50, device=dev, generator=g) * 0.05
    b1 = torch.zeros(50, device=dev)
    w2 = torch.randn(50, n_actions, device=dev, generator=g) * 0.05
    b2 = torch.zeros(n_actions, device=dev)
    return (w1, b1, w2, b2), "random-weight network"


def measure_policy(D: Dist, name: str, K: int, Wm: int, dump_budget: int = 0):
    """configs[2]: the reference's DQN network picks the actions (DQN.py:188-233).  Headline: the network evaluated
    INSIDE the step kernel (WF_POLICY_MLP); beside it, afterwards, the same policy through torch ops, one wf_step per
    step, the whole step (obs -> float -> MLP -> epsilon-greedy -> wf_step) captured in CUDA graphs."""
    torch = D.torch
    from wildfire_control_python_b200 import BatchedForestFire
    wl = WORKLOADS[name]
    dev, rank, world = D.dev, D.rank, D.world
    N, W, H = wl["n_envs"], wl["meta"]["width"], wl["meta"]["height"]
    env = BatchedForestFire(N, device=dev, auto_reset=True, seed=0, env_id_base=rank * N, **wl["meta"])
    env.reset()
    (w1, b1, w2, b2), policy_name = load_c3_policy(torch, dev, W, H, env.n_actions)
    # The policy evaluated INSIDE the step kernel (WF_POLICY_MLP): first layer kept incrementally as a sum of weight rows
    # of the observation bits, `chunk` steps per launch, obs/reward/done of every step still written.
    chunk = wl["chunk"]
    env.set_policy_mlp(w1, b1, w2, b2, eps=0.1)
    out = (torch.empty((chunk, N, W, H, 3), dtype=torch.uint8, device=dev), torch.empty((chunk, N), dtype=torch.float64, device=dev),
           torch.empty((chunk, N), dtype=torch.uint8, device=dev))
    l0 = env.launch_count
    ms, n_launch = timed_region(D, lambda n: env.rollout(n, policy="mlp", out=tuple(o[:n] for o in out)), K, chunk, Wm)
    res = {"name": name, "wl": wl, "N": N, "W": W, "H": H, "K": K, "warmup": warmup_steps(Wm, chunk), "chunk": chunk, "ms": ms,
           "launches": int(n_launch), "launches_total": int(env.launch_count - l0), "value": world * N * K / (ms * 1e-3),
           "obs_mb": out[0].numel() / 1e6, "family": env.kernel_family, "state_bytes": env.state_bytes_per_env,
           "tile_geometry": [0, 0],
           "policy": f"MLP 588-50(sigmoid)-4 = {policy_name}, eps-greedy 0.1, evaluated inside the step kernel (WF_POLICY_MLP); "
                     "`via_torch` is the same policy through torch ops"}
    if dump_budget:
        last = launch_sizes(K, chunk)[-1] - 1
        res["outputs"] = last_step_outputs(out[0][last], out[1][last], out[2][last], dump_budget)

    obs = env.observe()
    actions = torch.zeros(N, dtype=torch.int32, device=dev)

    def one_step():
        q = torch.sigmoid(obs.view(N, -1).float() @ w1 + b1) @ w2 + b2
        greedy = q.argmax(1).to(torch.int32)
        explore = torch.rand(N, device=dev) < 0.1
        rnd = torch.randint(0, env.n_actions, (N,), device=dev, dtype=torch.int32)
        actions.copy_(torch.where(explore, rnd, greedy))
        env.step(actions)  # writes the handle's persistent obs buffer, which `obs` aliases

    for _ in range(3):
        one_step()
    G_STEPS = 16
    graphs = {}
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        one_step()
        for n in {G_STEPS, *launch_sizes(K, G_STEPS)}:
            graphs[n] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphs[n], stream=side):
                for _ in range(n):
                    one_step()
    torch.cuda.current_stream(dev).wait_stream(side)
    for g in graphs.values():  # a graph's first replay uploads it: keep that out of the region
        g.replay()
    ms_torch, _ = timed_region(D, lambda n: graphs[n].replay(), K, G_STEPS, Wm)
    res["via_torch"] = {"value": world * N * K / (ms_torch * 1e-3), "unit": "env-steps/s", "steps": K,
                        "us_per_step": ms_torch * 1e3 / K,
                        "how": "obs -> float -> torch MLP -> eps-greedy -> wf_step, 16 steps per CUDA-graph replay"}
    res["stats"] = env.stats()
    env.close()
    del out, env
    torch.cuda.empty_cache()
    return res


def ncu_traffic_per_step(name):
    """DRAM bytes (read + write) per step of the workload's rollout kernel, from the committed ncu --set full capture."""
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.isfile(tpath):
        return None, None
    t = json.load(open(tpath)).get(name)
    if not t:
        return None, None
    return float(t["dram_bytes_per_step"]), t.get("source")


def roofline_of(res, world):
    peak, peak_src = load_peaks()
    N, W, H, chunk = res["N"], res["W"], res["H"], res["chunk"]
    per_gpu_steps = res["value"] / world
    survey = W * H * BYTES_PER_CELL_UPDATE
    if res["family"] == "warp":  # state stays in registers across a launch: only outputs (+ state once per launch) touch HBM
        own = W * H * 3 + 8 + 1 + 2 * res["state_bytes"] / chunk
        kernel = "wf::warp_kernel"
        note = (f"bytes_per_unit = what this layout must move per env-step: {W * H * 3} B uint8 observation + 8 B reward + 1 B done "
                f"+ the env's {res['state_bytes']} B of bit-planes loaded and stored once per {chunk}-step launch (they live in "
                "registers in between).  The kernel is issue/latency-bound, not HBM-bound, so `frac` is low by design; "
                "SURVEY 8(d)'s byte-per-cell accounting is in `survey_accounting`")
    else:  # dense pass per step: G, B, S read + S_next written (tick), F, I read + 96 B written (observation) per 32 cells
        own = W * H * (3 * 4 / 32 + 4 / 32 + 2 * 4 / 32 + 3)
        kernel = "wf::tile_rollout_kernel"
        note = ("bytes_per_unit = what this layout must move per env-step: per 32 cells the plane words G, B, S read + S_next "
                "written (tick) + F, I read (observation) + 96 B of uint8 observation written = 3.75 B per cell; fuel records "
                "and hit counters are touched only along the fire front (not counted).  HBM-bound by the observation write; "
                "SURVEY 8(d)'s byte-per-cell accounting (15 B per cell-update, which this layout does not move) is in "
                "`survey_accounting`")
    achieved = per_gpu_steps * own / 1e9
    t_step, t_src = ncu_traffic_per_step(res["name"])
    traffic = None if t_step is None else t_step * chunk
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_over_algorithmic": None if traffic is None else traffic / (own * N * chunk), "traffic_source": t_src,
            "peak_source": peak_src, "kernel": kernel, "bytes_per_unit": own, "unit_name": "env-step",
            "units_per_launch": N * chunk, "avg_launch_ms": res["ms"] / max(1, res["launches"]),
            "survey_accounting": {"bytes_per_unit": survey, "achieved": per_gpu_steps * survey / 1e9,
                                  "frac": per_gpu_steps * survey / 1e9 / peak,
                                  "what": "SURVEY.md 8(d): 6 B/cell state read + 6 B written + 3 B observation = 15 B per cell-update"},
            "note": note}


def launch_info(res):
    return {"steps_per_launch": res["chunk"], "kernel_family": res["family"],
            "tile_threads_x_cluster": res["tile_geometry"] if res["family"] == "tile" else None,
            "timing": f"{res['K']} steps = {res['launches']} launches in one CUDA-event interval, after {res['warmup']} "
                      "un-timed steps whose last launch is queued in front",
            "l2": f"outputs of one launch ({res['obs_mb']:.0f} MB obs) exceed the 126 MB L2; "
                  + ("state is register/L2 resident by design" if res["family"] == "warp"
                     else f"state ({res['state_bytes'] * res['N'] / 1e6:.0f} MB) exceeds L2 too")}


def secondary_entry(sec, world):
    e = {"workload": WORKLOADS[sec["name"]]["desc"], "config": workload_config(sec["name"]), "value": sec["value"],
         "unit": "env-steps/s", "steps": sec["K"], "repeats": 1, "warmup": sec["warmup"],
         "ms_per_step": sec["ms"] / sec["K"],
         "cell_updates_per_sec_per_gpu": sec["value"] * sec["W"] * sec["H"] / world, "gpu_launches": sec["launches"],
         "launch": launch_info(sec), "roofline": roofline_of(sec, world)}
    if "via_torch" in sec:
        e["via_torch"], e["policy"] = sec["via_torch"], sec["policy"]
    return e


def run_ours(args, wl):
    D = Dist(args.gpus)
    secondary = []
    if args.workload == "c2" and not args.no_secondary and not args.only_value:
        secondary = [s for s in args.secondary.split(",") if s]
    # rank 0's outputs only; every workload of the line gets the same share
    budget = DUMP_BYTES // (1 + len(secondary)) if args.dump_outputs and D.rank == 0 else 0
    secs = []
    with ClockSampler(D.local) as clk:
        if wl.get("policy"):
            res = measure_policy(D, args.workload, args.steps, args.warmup, budget)
        else:
            res = measure(D, args.workload, args.steps, args.warmup, args.chunk, not args.only_value, not args.only_value, budget)
        for name in secondary:
            if WORKLOADS[name].get("policy"):
                secs.append(measure_policy(D, name, args.steps, args.warmup, budget))
            else:
                secs.append(measure(D, name, args.steps, args.warmup, 0, False, False, budget))
    clocks = clk.summary()
    if D.rank != 0:
        D.close()
        return
    world, W, H, K = D.world, res["W"], res["H"], res["K"]
    if budget:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for r in [res] + secs:
            for key, arr in r["outputs"].items():
                np.save(os.path.join(args.dump_outputs, f"{r['name']}_{key}.npy"), arr)

    cpu_baseline = None
    if world == 1 and not args.only_value:
        cpu_baseline = port_baseline(wl, 1, CPU_BASELINE_SECONDS)
        cpu_baseline["host_cpus"] = os.cpu_count()
        if not args.no_python_ref:
            cpu_baseline["python_ref"] = python_ref_baseline(wl, PYTHON_REF_STEPS, 3, 20.0)

    config = workload_config(args.workload)
    config["l2"] = launch_info(res)["l2"]
    line = {
        "metric": "env_steps_per_sec", "value": res["value"], "unit": "env-steps/s", "n_gpus": world, "steps": K,
        "repeats": 1, "warmup": res["warmup"], "ms_per_step": res["ms"] / K,
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32-bitplanes+u8", "data": "synthetic",
        "config": config, "launch": launch_info(res),
        "cell_updates_per_sec": res["value"] * W * H,
        "cell_updates_per_sec_per_gpu": res["value"] * W * H / world,
        "e2e": res.get("e2e"), "per_step_launch": res.get("per_step"),
        "gpu_launches": res["launches"],
        "roofline": roofline_of(res, world),
        "cpu_baseline": cpu_baseline,
        "clocks": clocks,
        "stats": res["stats"],
    }
    if "policy" in res:
        line["policy"] = res["policy"]
        line["via_torch"] = res["via_torch"]
    if secs:
        line["secondary"] = {s["name"]: secondary_entry(s, world) for s in secs}
    print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2048)
    ap.add_argument("--warmup", type=int, default=256)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--chunk", type=int, default=0, help="steps per fused launch (default: the workload's)")
    ap.add_argument("--secondary", default="c4,c5,c3", help="workloads measured beside the default one (comma separated)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary measurements in the default line")
    ap.add_argument("--no-python-ref", action="store_true", help="skip the Python-reference leg of cpu_baseline")
    ap.add_argument("--only-value", action="store_true",
                    help="profiling runs: only the fused-rollout measurement (no per-step, e2e, CPU baseline legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs of every measured workload to DIR/<workload>_<array>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computed")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
