"""A/B of the post-physics kernel width (hb_set_option("post_warps", 4 | 8)) in ONE process, rounds interleaved.

    python scripts/ab_post_physics.py [--envs 4096,8192,16384,65536] [--rounds 5] [--steps 30]

Per shard size, one hector env per width (bench.py's workload: synthetic physics, device generator, CUDA-graph replay),
each captured with its width.  Each round times, for both widths in turn:
  step   env.step() from CUDA events, L2 flushed before every step (outside the events), mean over --steps steps
  post   post-physics alone, chain-timed: a graph of 4 launches replayed 10 times, L2 flushed before each replay
"""
import argparse
import os
import subprocess
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import torch

import bench
from isaac_b200 import _lib
from isaac_b200.envs.hector_config import HectorCfg
from isaac_b200.envs.hector_env import HectorFreeEnvB200
from isaac_b200.physics import SyntheticPhysics

ap = argparse.ArgumentParser()
ap.add_argument("--envs", default="4096,8192,16384,65536")
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--steps", type=int, default=30)
args = ap.parse_args()
dev = torch.device("cuda:0")
lib = _lib.load(check_device=True)
stream = torch.cuda.current_stream(dev)
flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)     # > 126 MB L2
flush_sink = torch.zeros(1, device=dev)


def flush_l2(i):
    flush.fill_(float(i))
    flush_sink.copy_(flush.sum())


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                          text=True).stdout.strip()


def make_env(n, warps, frames=4):
    _lib.check(lib.hb_set_option(b"post_warps", warps), "post_warps")
    tape = bench.make_workload(n, frames, 1234)
    phys_frames = [f.to(dev) for f in tape.physics]
    noise_frames = [f.to(dev) for f in tape.noise]
    phys = SyntheticPhysics(n, device=dev)
    phys.load_frame(phys_frames[0])
    env = HectorFreeEnvB200(HectorCfg(), sim_device=str(dev), physics=phys, statics=tape.statics, initial_noise=noise_frames[0])
    env.episode_length_buf.copy_(tape.statics.episode_length0)
    for _ in range(3):
        env.step(noise_frames[0].actions)
    env.enable_cuda_graph()
    env.prepare_action_buffers(*[f.actions for f in noise_frames])
    (o_cur, p_cur) = env._own[1][:2]
    env._draw_noise(False)

    def post(st):
        return lib.hb_env_post_physics(env._pp, env._pb, env._pn, o_cur.data_ptr(), p_cur.data_ptr(), _lib.HB_STAGE_STEP, st)
    post_graph = _lib.LaunchGraph(dev).record(lambda st: [_lib.check(post(st), "post") for _ in range(4)])
    return env, phys, phys_frames, noise_frames, post_graph


def step_us(case, steps):
    env, phys, phys_frames, noise_frames, _ = case
    tot = 0.0
    for i in range(steps + 2):
        f = i % len(phys_frames)
        phys.load_frame(phys_frames[f])
        flush_l2(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        env.step(noise_frames[f].actions)
        b.record(stream)
        b.synchronize()
        if i >= 2:
            tot += a.elapsed_time(b)
    return 1e3 * tot / steps


def post_us(case, reps=10):
    g = case[4]
    tot = 0.0
    for r in range(reps + 2):
        flush_l2(r)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        g.replay(stream.cuda_stream)
        b.record(stream)
        b.synchronize()
        if r >= 2:
            tot += a.elapsed_time(b)
    return 1e3 * tot / reps / 4


print(f"GPU: {gpu_info()}  (name, power limit, SM clock, max SM clock)", flush=True)
try:
    for n in [int(v) for v in args.envs.split(",")]:
        cases = {w: make_env(n, w) for w in (4, 8)}
        res = {w: [] for w in cases}
        for rnd in range(args.rounds):
            for w, case in cases.items():
                res[w].append((step_us(case, args.steps), post_us(case)))
        tiles = (n + 31) // 32
        print(f"n={n} ({tiles} tiles, {tiles / torch.cuda.get_device_properties(dev).multi_processor_count:.2f} per SM)", flush=True)
        for w, rs in res.items():
            st, po = [r[0] for r in rs], [r[1] for r in rs]
            print(f"  post_warps={w}: step us " + " ".join(f"{v:6.1f}" for v in st) + f" | median {sorted(st)[len(st) // 2]:6.1f}"
                  f" [{min(st):.1f}, {max(st):.1f}]   post-physics us " + " ".join(f"{v:5.2f}" for v in po) +
                  f" | median {sorted(po)[len(po) // 2]:5.2f} [{min(po):.2f}, {max(po):.2f}]", flush=True)
        del cases
        torch.cuda.empty_cache()
    print(f"GPU after: {gpu_info()}", flush=True)
finally:
    lib.hb_set_option(b"post_warps", 0)
