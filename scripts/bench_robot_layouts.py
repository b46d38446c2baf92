"""Env step time of robots described by a TaskLayout, against the three built robots on their compiled kernels.

    python scripts/bench_robot_layouts.py [--sizes 4096 16384 65536] [--rounds 5] [--steps 20] [--json PATH]

Cases: hector, hector_full and humanoid_ppo (XBot-L) on their compiled post-physics kernel and, with
hb_set_option("env_runtime_task", 1), on the kernel that reads the layout at run time; the made-up robots of
tests/test_robot_layouts.py (XBot kind 6 / 11 / 20 / 23 DOF, hector kind 8 / 14 / 22 with arms), which only have the latter.
Every case is built once per size; the rounds then alternate over the cases in one process, so that the spread over rounds
shows what the machine does to each of them alike.  Per case and round:

    step_ms   graph replay of the whole env step, L2 flushed between steps as bench.py does (256 MiB write + read)
    post_ms   hb_env_post_physics alone (single-node graph, L2 flushed before each replay)
    stack_ms  hb_env_stack_finalize alone (frame-stack shift of both histories + reset finalisation)

Bytes per env-step are the algorithmic traffic of SURVEY.md §8d (16 450 B for hector) computed from the layout by
`env_step_bytes`; the step's rate is reported against DESIGN.md's measured 6 540.5 GB/s.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

HBM_GBS = 6540.5            # DESIGN.md: measured HBM bandwidth of the B200


def env_step_bytes(cfg, nbody, decimation=10):
    """SURVEY.md §8d's accounting for a layout: n joints, frames O / P, stacks S / CS, nbody contact rows."""
    from isaac_b200._lib import HB_TASK_XBOT
    from isaac_b200.envs.tasks import layout_for
    lay = layout_for(cfg)
    n, O, P, S, CS = lay.ndof, lay.num_single_obs, lay.num_single_priv, cfg.env.frame_stack, cfg.env.c_frame_stack
    pd = decimation * (8 * n + 4 * n * 3 + 4 * n)              # R dof_state, actions, kp, kd; W torques
    ref = 4 * n if lay.kind == HB_TASK_XBOT else 0              # the reference trajectory (joint_pos reward, privileged frame)
    read = (52 + 8 * n + 12 * nbody + 64 + 12 * n + 4 * n + 24 + 4 * n + 16 + 8 + 26 + 72 + 28 + 4 * O
            + 4 * (S - 1) * O + 4 * (CS - 1) * P + ref)
    write = 4 * S * O + 4 * CS * P + 6 + 8 + 12 * n + 24 + 26 + 72 + 4 + 48 + ref
    return pd + read + write


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def cases():
    from isaac_b200.envs import TASKS
    from test_robot_layouts import NEW, new_cfg
    out = []
    for task in ("hector", "hector_full", "humanoid_ppo"):
        out += [(task, TASKS[task][1], 0), (task, TASKS[task][1], 1)]
    out += [(key, new_cfg(key), 1) for key in NEW]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 16384, 65536])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_robot_layouts: needs a CUDA device")
    from isaac_b200 import _lib
    from isaac_b200.synthetic import make_tape, task_dims
    from test_env_parity import make_cuda_env
    dev = torch.device("cuda:0")
    lib = _lib.load(check_device=True)
    stream = torch.cuda.current_stream(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    sink = torch.zeros(1, device=dev)

    def flush_l2(i):
        flush.fill_(float(i))
        sink.copy_(flush.sum())

    def elapsed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b)

    info = {"card (name, power limit, max SM clock)": card(), "hbm_gbs": HBM_GBS, "rounds": args.rounds,
            "steps_per_round": args.steps, "results": []}
    print(json.dumps({k: v for k, v in info.items() if k != "results"}), flush=True)
    for n in args.sizes:
        built = []
        for name, cfg_cls, rt in cases():
            _lib.check(lib.hb_set_option(b"env_runtime_task", rt), "env_runtime_task")
            tape = make_tape(n, 4, seed=1234, fall_prob=0.005, cfg=cfg_cls())
            frames = [f.to(dev) for f in tape.physics]
            acts = [f.actions.to(dev) for f in tape.noise]
            env, phys = make_cuda_env(tape, dev, cfg=cfg_cls())
            env.seed(5)
            for i in range(3):
                env.step(acts[i % 4])
            env.enable_cuda_graph()
            env.prepare_action_buffers(*acts)
            for i in range(4):          # both ping-pong graphs captured under this case's option
                phys.load_frame(frames[i % 4])
                env.step(acts[i % 4])
            (o_prev, p_prev), (o_cur, p_cur) = env._own[0][:2], env._own[1][:2]
            env._draw_noise(False)
            P, B = env._pp, env._pb
            g_post = _lib.LaunchGraph(dev).record(lambda st: _lib.check(lib.hb_env_post_physics(
                P, B, env._pn, o_cur.data_ptr(), p_cur.data_ptr(), _lib.HB_STAGE_STEP, st), "post"))
            g_stack = _lib.LaunchGraph(dev).record(lambda st: _lib.check(lib.hb_env_stack_finalize(
                P, B, o_prev.data_ptr(), p_prev.data_ptr(), o_cur.data_ptr(), p_cur.data_ptr(), env._host_count.data_ptr(),
                None, st), "stack"))
            dims = task_dims(cfg_cls())
            built.append(dict(name=name, path="runtime" if rt else "compiled", env=env, phys=phys, frames=frames, acts=acts,
                              g_post=g_post, g_stack=g_stack, bytes=env_step_bytes(cfg_cls(), dims.nbody), step=[], post=[],
                              stack=[]))
        _lib.check(lib.hb_set_option(b"env_runtime_task", 0), "env_runtime_task")
        torch.cuda.synchronize()
        for r in range(args.rounds):
            for c in built:
                env, phys = c["env"], c["phys"]
                tot = 0.0
                for i in range(args.steps):
                    phys.load_frame(c["frames"][i % 4])
                    flush_l2(i)
                    tot += elapsed(lambda: env.step(c["acts"][i % 4]))
                c["step"].append(tot / args.steps)
                for key in ("post", "stack"):
                    t = 0.0
                    for i in range(4):
                        flush_l2(i)
                        t += elapsed(lambda: c["g_" + key].replay(stream.cuda_stream))
                    c[key].append(t / 4)
        for c in built:
            med = lambda v: sorted(v)[len(v) // 2]
            row = {"envs": n, "robot": c["name"], "post_physics": c["path"], "bytes_per_env_step": c["bytes"]}
            for key in ("step", "post", "stack"):
                row[f"{key}_ms"] = round(med(c[key]), 4)
                row[f"{key}_ms_min_max"] = [round(min(c[key]), 4), round(max(c[key]), 4)]
            row["M_env_steps_per_s"] = round(n / row["step_ms"] / 1e3, 2)
            row["of_hbm"] = round(c["bytes"] * n / (row["step_ms"] * 1e-3) / (HBM_GBS * 1e9), 3)
            info["results"].append(row)
            print(json.dumps(row), flush=True)
        del built
        torch.cuda.empty_cache()
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
