"""Phase timing of one probe CTA of the tile rollout kernel (needs tools/_dbg/libwf_timing.so, -DWF_TILE_TIMING)."""
import ctypes as C
import os
import sys
os.environ["WILDFIRE_B200_LIB"] = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_dbg", "libwf_timing.so")
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import WORKLOADS
from wildfire_control_python_b200 import BatchedForestFire, _lib

name = sys.argv[1] if len(sys.argv) > 1 else "c4"
with_obs = (sys.argv[2] != "0") if len(sys.argv) > 2 else True
wl = WORKLOADS[name]
N, W, H = wl["n_envs"], wl["meta"]["width"], wl["meta"]["height"]
env = BatchedForestFire(N, auto_reset=True, seed=0, **wl["meta"])
env.reset()
K = 16
obs = torch.empty((K, N, W, H, 3), dtype=torch.uint8, device="cuda") if with_obs else None
rew = torch.empty((K, N), dtype=torch.float64, device="cuda")
done = torch.empty((K, N), dtype=torch.uint8, device="cuda")
L = _lib.lib()
buf = (C.c_ulonglong * 16)()
for _ in range(3):
    env.rollout(K, out=(obs, rew, done), obs=with_obs)
L.wf_debug_tile_timing(buf, 1)
R = 10
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(R):
    env.rollout(K, out=(obs, rew, done), obs=with_obs)
e1.record()
torch.cuda.synchronize()
L.wf_debug_tile_timing(buf, 0)
names = ["barrier X", "flood + tick", "CTA barrier", "Y + finish + agent", "observation", "closing sync", "slow + reset"]
tot = sum(buf[i] for i in range(len(names)))
print(f"{name} obs={with_obs}: {e0.elapsed_time(e1) * 1e3 / (R * K):.2f} us/step; probe CTA per step:")
for i, n in enumerate(names):
    print(f"  {n:12s} {buf[i] / (R * K) / 1e3:7.2f} us")
print(f"  {'sum':12s} {tot / (R * K) / 1e3:7.2f} us")
