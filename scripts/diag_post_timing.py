"""Debug-build diagnostic (HB_EXTRA_NVCC_FLAGS=-DHB_POST_TIMING): phase timeline of post_physics_kernel per role warp.

    python scripts/diag_post_timing.py [num_envs] [post_warps: 4 or 8, default 4]
"""
import ctypes as C
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from isaac_b200 import _lib
from isaac_b200.envs.hector_config import HectorCfg
from isaac_b200.envs.hector_env import HectorFreeEnvB200
from isaac_b200.physics import SyntheticPhysics
from isaac_b200.synthetic import make_tape

n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
warps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
dev = torch.device("cuda:0")
lib = _lib.load(check_device=True)
_lib.check(lib.hb_set_option(b"post_warps", warps), "post_warps")
tape = make_tape(n, 2, seed=1, fall_prob=0.005)
phys = SyntheticPhysics(n, device=dev)
phys.load_frame(tape.physics[0].to(dev))
env = HectorFreeEnvB200(HectorCfg(), sim_device="cuda:0", physics=phys, statics=tape.statics, initial_noise=tape.noise[0].to(dev))
nzf = tape.noise[1].to(dev)
flush = torch.empty(64 * 1024 * 1024, device=dev)
for i in range(4):
    env.inject_noise(nzf)
    flush.fill_(i)
    env.step(nzf.actions)
torch.cuda.synchronize()
tiles = min((n + 31) // 32, 4096)
buf = np.zeros(tiles * 8 * 8, dtype=np.int64)
fn = lib.hb_debug_post_stamps
fn.restype, fn.argtypes = C.c_int, [C.c_void_p, C.c_int]
assert fn(buf.ctypes.data, buf.size) == 0
s = buf.reshape(tiles, 8, 8)[:, :warps].astype(np.float64)
t0 = s[:, :, 0].min(axis=1)[:, None, None]
rel = (s - t0) / 1.965e3            # us at 1965 MHz
names = ["start", "tile staged", "phase A done", "past barrier 1", "phase B done", "past barrier 2", "stores done"]
print(f"n={n} tiles={tiles} post_warps={warps}: median [p10, p90] in us since the CTA's first stamp, per role warp")
roles = ("base", "joints", "feet", "ledger") if warps == 4 else ("base", "joints", "feet", "base'", "joints'", "feet'", "ledger",
                                                                  "ledger'")
for w, role in enumerate(roles):
    parts = []
    for k in range(7):
        v = rel[:, w, k]
        if k == 1 and role.startswith("ledger") or k == 5 and role.startswith("ledger"):
            parts.append("   -   ")
            continue
        parts.append(f"{np.median(v):5.1f} [{np.percentile(v,10):4.1f},{np.percentile(v,90):5.1f}]")
    print(f"  {role:7s} " + " | ".join(parts))
print("  columns: " + " | ".join(names))

gt = np.zeros(tiles * 3, dtype=np.uint64)
fn2 = lib.hb_debug_post_globaltimes
fn2.restype, fn2.argtypes = C.c_int, [C.c_void_p, C.c_int]
assert fn2(gt.ctypes.data, gt.size) == 0
gt = gt.reshape(tiles, 3).astype(np.float64)
t_first = gt[:, 0].min()
start, done = (gt[:, 0] - t_first) / 1e3, (gt[:, 1] - t_first) / 1e3
print(f"  global timeline (us): first CTA start 0.0, last CTA start {start.max():.1f}, last stores done {done.max():.1f}; "
      f"CTA lifetime median {np.median(done - start):.1f}")
hist, edges = np.histogram(start, bins=8)
print("  CTA start histogram:", " ".join(f"{e:.0f}us:{h}" for h, e in zip(hist, edges)))
