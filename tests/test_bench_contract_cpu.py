"""bench.py's JSON line, assembled on the CPU from canned measurements: every key the bench contract names must be there
and consistent (value = envs x steps / time, roofline.frac = achieved / peak, ...).  The GPU legs are stubbed; the
cpu_baseline leg runs the real C oracle for a fraction of a second."""
import json
import sys
import types

import pytest

import bench


class _FakeDist:
    rank, world, local = 0, 1, 0

    def __init__(self, gpus):
        pass

    def close(self):
        pass


class _NoClocks:
    def __init__(self, index):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        pass

    def summary(self):
        return {"sm_mhz": 1965, "sm_max_mhz": 1965, "reasons": [], "samples": 3}


def _canned(name, K, Wm=5):
    wl = bench.WORKLOADS[name]
    N, W, H = wl["n_envs"], wl["meta"]["width"], wl["meta"]["height"]
    chunk = wl["chunk"]
    us = 2.5 if W <= 32 else 50.0
    ms = us * 1e-3 * K
    fam = "warp" if W <= 32 else "tile"
    n_launch = len(bench.launch_sizes(K, chunk))
    out = {"name": name, "wl": wl, "N": N, "W": W, "H": H, "K": K, "warmup": bench.warmup_steps(Wm, chunk), "chunk": chunk,
           "ms": ms, "launches": n_launch, "launches_total": n_launch + 4, "value": N * K / (ms * 1e-3),
           "obs_mb": chunk * N * W * H * 3 / 1e6, "family": fam, "state_bytes": 1280 if fam == "warp" else 409664,
           "tile_geometry": [0, 0] if fam == "warp" else [256, 1],
           "stats": {"env_steps": N * K, "episodes": 1, "deaths": 1, "contained": 0, "burnouts": 0, "ticks": N * K},
           "e2e": {"value": 9e7, "unit": "env-steps/s", "h2d_bytes_per_step": N * 4, "d2h_bytes_per_step": 1, "steps": K, "repeats": 3},
           "per_step": {"value": 3e8, "unit": "env-steps/s", "steps": 3}}
    if wl.get("policy"):
        out["via_torch"] = {"value": 1e8, "unit": "env-steps/s"}
        out["policy"] = "canned"
    return out


def test_launch_sizes_time_exactly_the_requested_steps():
    for K, chunk in [(20, 256), (20, 16), (2048, 256), (7, 64), (20000, 256), (1, 256), (64, 64), (65, 64)]:
        sizes = bench.launch_sizes(K, chunk)
        assert sum(sizes) == K and all(0 < n <= chunk for n in sizes)
        assert len(sizes) == -(-K // chunk) and sizes[:-1] == [chunk] * (len(sizes) - 1)  # the fewest launches, all full but the last
    assert bench.warmup_steps(5, 256) == 256 and bench.warmup_steps(0, 16) == 16 and bench.warmup_steps(33, 16) == 48


@pytest.mark.parametrize("argv", [[], ["--workload", "c4", "--steps", "64", "--warmup", "8"], ["--steps", "20", "--warmup", "5"],
                                  ["--only-value", "--steps", "512"], ["--workload", "c3", "--steps", "20"]],
                         ids=["default", "c4", "driver_20_5", "only_value", "c3"])
def test_bench_line_has_the_contract_keys(monkeypatch, capsys, argv):
    monkeypatch.setattr(bench, "Dist", _FakeDist)
    monkeypatch.setattr(bench, "ClockSampler", _NoClocks)
    monkeypatch.setattr(bench, "CPU_BASELINE_SECONDS", 0.2)
    monkeypatch.setattr(bench, "python_ref_baseline", lambda wl, steps, warmup, budget_s=60.0: None)
    monkeypatch.setattr(bench, "measure", lambda D, name, K, Wm, chunk, e2e, per_step, dump_budget=0: {
        k: v for k, v in _canned(name, K, Wm).items() if (k != "e2e" or e2e) and (k != "per_step" or per_step)})
    monkeypatch.setattr(bench, "measure_policy", lambda D, name, K, Wm, dump_budget=0: {
        k: v for k, v in _canned(name, K, Wm).items() if k not in ("e2e", "per_step")})
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "repeats", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "launch", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert key in line, key
    assert line["metric"] == "env_steps_per_sec" and line["unit"] == "env-steps/s" and line["scaling"] == "weak"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["n_gpus"] == 1
    name = argv[argv.index("--workload") + 1] if "--workload" in argv else "c2"
    wl = bench.WORKLOADS[name]
    assert "model" not in line["config"] and "l2" in line["config"]
    assert {k: line["config"][k] for k in ("workload", "grid", "envs_per_gpu")} == bench.workload_config(name)
    assert line["warmup"] >= 3 and line["gpu_launches"] >= 1
    assert line["steps"] == (int(argv[argv.index("--steps") + 1]) if "--steps" in argv else 2048)
    assert line["value"] == pytest.approx(wl["n_envs"] / (line["ms_per_step"] * 1e-3))
    chunk = line["launch"]["steps_per_launch"]
    assert line["repeats"] == 1 and line["gpu_launches"] == len(bench.launch_sizes(line["steps"], chunk))  # --steps steps timed
    assert line["ms_per_step"] * line["steps"] == pytest.approx(_canned(name, line["steps"])["ms"])
    assert line["warmup"] == bench.warmup_steps(int(argv[argv.index("--warmup") + 1]) if "--warmup" in argv else 256, chunk)
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    assert r["achieved"] == pytest.approx(line["value"] * r["bytes_per_unit"] / 1e9)
    assert r["units_per_launch"] == wl["n_envs"] * line["launch"]["steps_per_launch"]
    sa = r["survey_accounting"]
    assert sa["bytes_per_unit"] == wl["meta"]["width"] * wl["meta"]["height"] * 15
    assert sa["frac"] == pytest.approx(line["value"] * sa["bytes_per_unit"] / 1e9 / r["peak"])
    if r["traffic"] is not None:
        assert r["traffic_over_algorithmic"] == pytest.approx(r["traffic"] / (r["bytes_per_unit"] * r["units_per_launch"]))
    if name in ("c2", "c4", "c5"):
        assert r["traffic"] is not None  # profiles/ncu_traffic.json covers every non-policy workload
    if "--only-value" in argv or name == "c3":
        assert line["e2e"] is None and "secondary" not in line
    else:
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
        cb = line["cpu_baseline"]
        assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] > 0 and "sample" in cb and "python_ref" in cb
        assert ("secondary" in line) == ("--workload" not in argv)
        if "secondary" in line:
            assert set(line["secondary"]) == {"c4", "c5", "c3"}
            for k, e in line["secondary"].items():
                assert e["config"] == bench.workload_config(k) and e["roofline"]["frac"] > 0 and e["value"] > 0
            assert "via_torch" in line["secondary"]["c3"]


def test_reference_arm_line(monkeypatch, capsys):
    """--impl reference: the reference's Python step (when the snapshot / tree is there) and the oracle port on the host
    cores; same metric / unit / config as our arm, impl = reference."""
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "3", "--warmup", "1"])
    monkeypatch.setitem(bench.WORKLOADS, "c2", dict(bench.WORKLOADS["c2"], n_envs=64))
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "env_steps_per_sec" and line["unit"] == "env-steps/s"
    assert line["config"] == bench.workload_config("c2")
    cb = line["cpu_baseline"]
    assert line["value"] > 0 and cb["value"] == line["value"]
    from oracle import ref_bench
    if ref_bench.available():
        assert cb["kind"] == "_ref" and cb["port"]["kind"] == "port" and cb["port"]["value"] > cb["value"]
    else:
        assert cb["kind"] == "port"
    assert line["e2e"] == {"value": line["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["higher_is_better"] is True


def test_dump_outputs_writes_every_workload_within_64_mib(monkeypatch, capsys, tmp_path):
    """--dump-outputs DIR: reward, done and observations of the last timed step of every workload of the line as float32 /
    float64 .npy files, 64 MiB in all; workloads whose observations do not fit keep a fixed seeded sample of envs."""
    import numpy as np
    import torch

    def with_outputs(name, K, Wm, budget):
        res = _canned(name, K, Wm)
        N, W, H = res["N"], res["W"], res["H"]
        g = torch.Generator().manual_seed(len(name))
        obs = torch.randint(0, 2, (1, W, H, 3), dtype=torch.uint8, generator=g).expand(N, -1, -1, -1)
        reward = torch.arange(N, dtype=torch.float64) - 0.5
        done = (torch.arange(N) % 3 == 0).to(torch.uint8)
        assert budget > 0
        res["outputs"] = bench.last_step_outputs(obs, reward, done, budget)
        return res

    monkeypatch.setattr(bench, "Dist", _FakeDist)
    monkeypatch.setattr(bench, "ClockSampler", _NoClocks)
    monkeypatch.setattr(bench, "CPU_BASELINE_SECONDS", 0.2)
    monkeypatch.setattr(bench, "python_ref_baseline", lambda wl, steps, warmup, budget_s=60.0: None)
    monkeypatch.setattr(bench, "measure", lambda D, name, K, Wm, chunk, e2e, per_step, dump_budget=0: {
        k: v for k, v in with_outputs(name, K, Wm, dump_budget).items() if (k != "e2e" or e2e) and (k != "per_step" or per_step)})
    monkeypatch.setattr(bench, "measure_policy", lambda D, name, K, Wm, dump_budget=0: {
        k: v for k, v in with_outputs(name, K, Wm, dump_budget).items() if k not in ("e2e", "per_step")})
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "20", "--warmup", "5", "--dump-outputs", str(tmp_path / "out")])
    bench.main()
    assert json.loads(capsys.readouterr().out.strip().splitlines()[-1])["steps"] == 20
    files = sorted(p.name for p in (tmp_path / "out").iterdir())
    assert files == sorted(f"{w}_{a}.npy" for w in ("c2", "c3", "c4", "c5") for a in ("obs", "reward", "done", "obs_env_index"))
    assert sum(p.stat().st_size for p in (tmp_path / "out").iterdir()) <= 64 << 20
    for w in ("c2", "c3", "c4", "c5"):
        wl = bench.WORKLOADS[w]
        N, W, H = wl["n_envs"], wl["meta"]["width"], wl["meta"]["height"]
        a = {k: np.load(tmp_path / "out" / f"{w}_{k}.npy") for k in ("obs", "reward", "done", "obs_env_index")}
        assert all(v.dtype in (np.float32, np.float64) for v in a.values())
        assert a["reward"].dtype == np.float64 and np.array_equal(a["reward"], np.arange(N) - 0.5)
        assert np.array_equal(a["done"], (np.arange(N) % 3 == 0).astype(np.float32))
        idx = a["obs_env_index"].astype(np.int64)
        assert a["obs"].shape == (len(idx), W, H, 3) and np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < N
        assert (len(idx) == N) == (w == "c2")  # c2's 4096 observations fit whole; the others are sampled
    # the sample is a function of the shapes and the budget only
    obs = torch.zeros((100, 4, 4, 3), dtype=torch.uint8)
    one = bench.last_step_outputs(obs, torch.zeros(100, dtype=torch.float64), torch.zeros(100, dtype=torch.uint8), 20 * 100 + 10 * 192)
    two = bench.last_step_outputs(obs, torch.zeros(100, dtype=torch.float64), torch.zeros(100, dtype=torch.uint8), 20 * 100 + 10 * 192)
    assert len(one["obs_env_index"]) == 10 and np.array_equal(one["obs_env_index"], two["obs_env_index"])
