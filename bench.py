#!/usr/bin/env python
"""Benchmark of the hector hot path on B200 (contract: one JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--impl reference] [--dump-outputs DIR]

A "step" is one `env.step(actions)` over E environments per GPU with the opaque physics stage
stubbed (SURVEY.md §8d): action prologue + `decimation`=10 PD-torque sub-steps (10 launches), the fused
post-physics kernel (termination, 18 reward terms, resets, newest observation frames) and the
frame-stacking + reset-finalisation kernel (ids, count to pinned host memory, episode means): 12 launches,
replayed from CUDA graphs.
metric = env-steps/s summed over all GPUs (weak scaling: E envs per GPU, no data-path collective).
The same run also reports GAE over [T=24, E] ("gae"), the PPO update on [24, E] rollouts with 5 epochs x 4
minibatches ("ppo": samples/s, TF32 TFLOP/s), the rollout side (PPO.act + process_env_step per step) and a whole
learning iteration ("ppo.iteration", the reference's Perf/total_fps definition).

value      device time: per-step CUDA events on the launching stream, all inputs resident in HBM,
           L2 flushed between steps (a 256 MiB write, then a 256 MiB read so that no dirty flush lines are written
           back inside the timed region; both outside the timed events), max over ranks.
e2e        the public `HectorFreeEnvB200.step()` with HOST buffers: per step the physics state and the
           actions are copied from pinned host memory, the env draws its own noise, and obs /
           privileged obs / rewards / resets are copied back to pinned host memory; wall clock.
roofline   the dominant kernel (frame stacking of both observation histories, with the reset finalisation riding in
           the same launch) against MEASURED_PEAKS.json: algorithmic bytes / average launch duration over a graph of
           4 launches on 4 distinct cold buffer sets.
cpu_baseline / --impl reference: the CPU oracle port of the reference's torch code
           (oracle/hector_oracle.py, torch CPU, all host threads) on the same workload.
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
sys.path.insert(0, ROOT)

import torch  # noqa: E402

B_ENV_STEP = 16450          # algorithmic bytes per env-step (SURVEY.md §8d)
FRAME_OBS, STACK_OBS, FRAME_PRIV, STACK_PRIV = 41, 15, 70, 15
T_GAE = 24


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the measurement (NVML; the recipe's nvidia-smi fields)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.sm, self.sm_max, self.reasons = index, [], None, set()
        self.stop_flag = threading.Event()
        self.error = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
            while not self.stop_flag.is_set():
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = get_reasons(h)
                self.reasons |= {n for bit, n in names.items() if r & bit}
                self.stop_flag.wait(0.005)
        except Exception as e:          # no NVML: report it instead of inventing clocks
            self.error = repr(e)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=2)
        sm = sorted(self.sm)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
               "samples": len(sm)}
        if self.error:
            out["error"] = self.error
        return out


def bind_to_gpu_cpus(index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `index` (its NUMA node): pinned host buffers and the
    copy engines' DMA then stay on that socket (e2e leg at N > 1)."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        words = nv.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:
        return None


def make_workload(n, frames, seed):
    from isaac_b200.synthetic import make_tape
    return make_tape(n, frames, seed=seed, fall_prob=0.005, randomize_gains=True)


def fill_storage_cpu(st, seed):
    g = torch.Generator().manual_seed(seed)
    T, N = st["rewards"].shape[:2]
    st["observations"].copy_(torch.randn(T, N, 615, generator=g))
    st["privileged_observations"].copy_(torch.randn(T, N, 1050, generator=g))
    st["actions"].copy_(torch.randn(T, N, 10, generator=g))
    st["mu"].copy_(st["actions"] + 0.3 * torch.randn(T, N, 10, generator=g))
    st["sigma"].fill_(1.0)
    st["rewards"].copy_(torch.rand(T, N, 1, generator=g) * 0.05)
    st["values"].copy_(torch.randn(T, N, 1, generator=g) * 0.5)
    st["dones"].copy_((torch.rand(T, N, 1, generator=g) < 0.005).to(torch.uint8))
    st["actions_log_prob"].copy_(-0.5 * ((st["actions"] - st["mu"]) ** 2).sum(-1, keepdim=True) - 9.19)


def workload_name(n):
    """config.workload, identical on both arms."""
    return f"hector task, {n} envs per GPU, env.step with stubbed physics (BASELINE configs[1])"


DUMP_LIMIT_BYTES = 64_000_000          # 64 MB in all


def dump_outputs(path, out):
    """--dump-outputs: what env.step() returned in the last timed step, one float32 .npy per array - obs,
    privileged_obs, rewards, resets, time_outs ([N, ...] rows per env) and episode_<name> (the scalars of
    extras["episode"]).  Above 64 MB in all, the per-env arrays keep a fixed sample of env rows (seed 0, ascending
    ids, the same rows in every array), so that runs with the same arguments write comparable files."""
    import numpy as np
    obs, priv, rew, reset, extras = out
    per_env = {"obs": obs, "privileged_obs": priv, "rewards": rew, "resets": reset}
    if "time_outs" in extras:
        per_env["time_outs"] = extras["time_outs"]
    n = obs.shape[0]
    row_bytes = sum(4 * t[0].numel() for t in per_env.values())
    if n * row_bytes > DUMP_LIMIT_BYTES:          # (one row less leaves room for the .npy headers and the episode scalars)
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes - 1, replace=False))
        ids = torch.from_numpy(rows).to(obs.device)
        per_env = {k: t.index_select(0, ids) for k, t in per_env.items()}
    arrays = {k: t.detach().float().cpu().numpy() for k, t in per_env.items()}
    arrays.update({"episode_" + k: np.float32(float(v)) for k, v in extras.get("episode", {}).items()})
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.asarray(a, dtype=np.float32))


# ------------------------------------------------------------------------------------ reference arm
def reference_env(n, frames, seed):
    """The reference's CPU implementation of env.step on the workload's tape: the UNMODIFIED reference
    (found by oracle/ref_harness.py) when it is there
    (kind "reference"), else the oracle port (kind "port").  Returns (step(i), kind, description)."""
    from isaac_b200.envs.hector_config import HectorCfg
    tape = make_workload(n, frames, seed)
    from oracle import ref_harness
    if ref_harness.reference_root() is not None:
        ref = ref_harness.ReferenceEnv(tape.statics, tape.physics[0], tape.noise[0])
        return (lambda i: ref.step(tape.physics[i % frames], tape.noise[i % frames]), "reference",
                f"unmodified reference HectorFreeEnv.step ({ref_harness.reference_root()}), isaacgym stubbed")
    print("bench.py: the unmodified reference is not found (set ISAAC_REFERENCE to a checkout of DRCL-USC/isaac); "
          "the CPU arm times the oracle port instead (cpu_baseline.kind = \"port\")", file=sys.stderr, flush=True)
    from oracle.hector_oracle import OracleHectorEnv
    env = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    return (lambda i: env.step(tape.physics[i % frames], tape.noise[i % frames]), "port", "torch CPU oracle port")


def run_reference(args, rank):
    """--impl reference: the reference's own torch CPU code on the box's host cores, all threads (rank 0 only; at N > 1
    it still steps ONE shard of args.envs envs - the CPU has no second socket per GPU - so per-N ratios compare a CPU
    shard with N GPU shards)."""
    if rank != 0:
        return
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):      # the reference prints its networks on construction; stdout = one JSON line
        line = _reference_line(args)
    print(json.dumps(line), flush=True)


def _reference_line(args):
    from oracle.ppo_oracle import gae_returns
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = args.envs
    step, kind, what = reference_env(n, 4, 1234)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        out = step(args.warmup + i)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    value = n * args.steps / dt
    g = torch.Generator().manual_seed(0)
    r, v = torch.rand(T_GAE, n, 1, generator=g), torch.randn(T_GAE, n, 1, generator=g)
    d, lv = (torch.rand(T_GAE, n, 1, generator=g) < 0.005).byte(), torch.randn(n, 1, generator=g)
    # PPO: GAE + update on the CPU, a bounded sample (1 epoch x 4 minibatches of the same [24, n] rollout)
    from oracle import ref_harness
    from oracle.ppo_oracle import OraclePPO, init_actor_critic_params
    cfg1 = dict(PPO_CFG, num_learning_epochs=1)
    perm = torch.randperm(n * T_GAE, generator=g)
    if kind == "reference":
        policy = dict(init_noise_std=1.0, actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128])
        ref = ref_harness.ReferencePPO(init_actor_critic_params(seed=5), n, T_GAE, cfg1, policy)
        st = ref.alg.storage
        fill_storage_cpu(dict(observations=st.observations, privileged_observations=st.privileged_observations,
                              actions=st.actions, mu=st.mu, sigma=st.sigma, rewards=st.rewards, values=st.values,
                              dones=st.dones, actions_log_prob=st.actions_log_prob), 100)
        st.step = T_GAE
        t0 = time.perf_counter()
        ref.compute_returns(torch.randn(n, 1050, generator=g))
        gae_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        ref.update(perm)
        ppo_s = time.perf_counter() - t0
    else:
        gae_returns(r, v, d, lv, 0.994, 0.9)
        t0 = time.perf_counter()
        for _ in range(5):
            gae_returns(r, v, d, lv, 0.994, 0.9)
        gae_s = (time.perf_counter() - t0) / 5
        ora = OraclePPO(init_actor_critic_params(seed=5), n, T_GAE, **cfg1)
        fill_storage_cpu(ora.st, 100)
        ora.compute_returns(torch.randn(n, 1050, generator=g))
        t0 = time.perf_counter()
        ora.update(perm)
        ppo_s = time.perf_counter() - t0
    sample = f"{args.steps} steps of {n} envs after {args.warmup} warm-up, {what}, torch CPU {torch.__version__}, {cores} threads"
    line = {"impl": "reference", "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(n), "envs_per_gpu": n, "decimation": 10,
                       "note": "the CPU arm steps one shard of envs_per_gpu envs at every --gpus N"},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
            "gae": {"value": T_GAE * n / gae_s, "unit": "samples/s", "T": T_GAE,
                    "what": "PPO.compute_returns (critic forward + GAE)" if kind == "reference" else "GAE scan"},
            "gpu_launches": 0,
            "ppo": {"value": T_GAE * n / (ppo_s * 5), "unit": "samples/s", "sample_passes_per_s": T_GAE * n / ppo_s,
                    "sample": f"1 epoch x 4 minibatches of [{T_GAE},{n}] timed ({ppo_s:.1f} s), x5 epochs extrapolated"},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    return line


# ------------------------------------------------------------------------------------ B200 arm
def cpu_baseline(n, budget_s=10.0):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind, what = reference_env(n, 3, 1234)
    for i in range(2):
        step(i)
    steps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s and steps < 5000:
        step(steps)
        steps += 1
    dt = time.perf_counter() - t0
    return {"value": n * steps / dt, "unit": "env-steps/s", "cores": cores, "kind": kind,
            "sample": f"{steps} steps of {n} envs ({dt:.1f} s), {what}, {cores} threads"}


def measure_tf32_peak(dev, seconds=1.5):
    """Dense TF32 tensor-core peak of this GPU, the way MEASURED_PEAKS.json measures bf16: torch.matmul (cuBLAS) on
    8192^3 fp32 operands with TF32 math allowed - best of 10 (burst) and back to back for `seconds` (sustained)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a, b = torch.randn(n, n, device=dev), torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize(dev)
        flop = 2.0 * n ** 3
        best = 0.0
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            e1.synchronize()
            best = max(best, flop / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        reps = max(10, int(seconds / (flop / (best * 1e12))))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b, out=c)
        e1.record()
        e1.synchronize()
        sustained = reps * flop / (e0.elapsed_time(e1) * 1e-3) / 1e12
        return {"burst_tflops": best, "sustained_tflops": sustained,
                "how": f"torch.matmul fp32 {n}^3 with allow_tf32 (cuBLAS): best of 10; {reps} back to back"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


PPO_FLOP_PER_SAMPLE_PASS = 6.853e6        # fwd 3.032 + bwd 3.821 MFLOP (SURVEY.md §8d)
PPO_CFG = dict(num_learning_epochs=5, num_mini_batches=4, clip_param=0.2, gamma=0.994, lam=0.9, value_loss_coef=1.0,
               entropy_coef=0.001, learning_rate=1e-5, max_grad_norm=1.0, use_clipped_value_loss=True,
               schedule="adaptive", desired_kl=0.01)


def fill_storage(st, gen_seed, device):
    """PPO sweep inputs (SURVEY.md §8d): N(0,1) observations, dones ~ Bernoulli(0.005)."""
    g = torch.Generator(device=device).manual_seed(gen_seed)
    T, N = st.num_transitions_per_env, st.num_envs
    st.observations.copy_(torch.randn(T, N, 615, device=device, generator=g))
    st.privileged_observations.copy_(torch.randn(T, N, 1050, device=device, generator=g))
    st.actions.copy_(torch.randn(T, N, 10, device=device, generator=g))
    st.mu.copy_(st.actions + 0.3 * torch.randn(T, N, 10, device=device, generator=g))
    st.sigma.fill_(1.0)
    st.rewards.copy_(torch.rand(T, N, 1, device=device, generator=g) * 0.05)
    st.values.copy_(torch.randn(T, N, 1, device=device, generator=g) * 0.5)
    st.dones.copy_((torch.rand(T, N, 1, device=device, generator=g) < 0.005).to(torch.uint8))
    st.actions_log_prob.copy_(-0.5 * ((st.actions - st.mu) ** 2).sum(-1, keepdim=True) - 9.19)


def bench_iteration(env, phys, phys_frames, alg, dev, n, iters=2):
    """One learning iteration the way OnPolicyRunner.learn drives it (on_policy_runner.py:124-170): T x (act, env.step,
    process_env_step), compute_returns, update - the reference's own `Perf/total_fps` = T * N / (collection + learning)
    (on_policy_runner.py:199-213), wall clock, physics stubbed."""
    frames = len(phys_frames)
    alg.attach_env(env)          # step() writes its observations straight into the rollout slots (SURVEY.md §8f rank 1)
    obs, priv = env.get_observations(), env.get_privileged_observations()
    out = None
    for it in range(iters + 1):
        alg.storage.clear()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for t in range(T_GAE):
            actions = alg.act(obs, priv)
            phys.load_frame(phys_frames[t % frames])
            obs, priv, rew, dones, infos = env.step(actions)
            alg.process_env_step(rew, dones, infos)
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        alg.compute_returns(priv)
        alg.update()
        torch.cuda.synchronize(dev)
        t2 = time.perf_counter()
        out = {"total_fps": T_GAE * n / (t2 - t0), "collection_ms": 1e3 * (t1 - t0), "learning_ms": 1e3 * (t2 - t1),
               "unit": "env-steps/s per GPU, wall clock, T=24 rollout + 5 epochs x 4 minibatches",
               "definition": "Perf/total_fps of on_policy_runner.py:199-213 (physics stubbed)",
               "observations": "written by env.step() into the rollout slots (PPO.attach_env)"}
    alg.attach_env(None)
    return out


def time_updates(alg, args, dev, n, world, rank, last, reps):
    """Mean device time (ms, max over ranks) of compute_returns + update() over `reps` timed updates after one warm-up
    (the second update also captures the per-minibatch graphs: two warm-ups on a single GPU)."""
    import torch.distributed as dist
    stream = torch.cuda.current_stream(dev)
    times = []
    warm = 2 if (world == 1 or alg._peer is not None) else 1      # graph capture happens in the second update
    for r in range(reps + warm):
        fill_storage(alg.storage, 100 + rank, dev)
        alg.storage.step = T_GAE
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        alg.compute_returns(last)
        alg.update()
        b.record(stream)
        b.synchronize()
        if r >= warm:
            times.append(a.elapsed_time(b))
    t = torch.tensor([sum(times) / len(times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def bench_ppo(args, dev, n, world, rank, env=None, phys=None, phys_frames=None):
    """compute_returns + update() on [T=24, n] rollouts: PPO samples/s (BASELINE configs[1]/[4])."""
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    torch.manual_seed(5)
    ac = ActorCritic(615, 1050, 10, actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128], device=dev)
    alg = PPO(ac, device=dev, **PPO_CFG)
    alg.init_storage(n, T_GAE, [615], [1050], [10])
    if world > 1:
        from isaac_b200.parallel import attach_data_parallel
        # default: ONE kernel per rank over NVLink peer memory (reduce + clip + Adam + broadcast); HB_DP_FUSED=0 = NCCL
        attach_data_parallel(alg, env=env, fused=os.environ.get("HB_DP_FUSED", "1") != "0",
                             use_multicast=os.environ.get("HB_DP_MULTICAST", "1") != "0")
    last = torch.randn(n, 1050, device=dev)
    stream = torch.cuda.current_stream(dev)
    # rollout side (SURVEY.md §8f rank 1): PPO.act + process_env_step per env step, T steps; the observations are
    # already in the slot, as after PPO.attach_env(env)
    alg.storage.observations.normal_(), alg.storage.privileged_observations.normal_()
    rew_, done_ = torch.rand(n, device=dev), torch.rand(n, device=dev) < 0.005
    infos_ = {"time_outs": torch.rand(n, device=dev) < 0.0004}
    roll_ms = None
    for r in range(2):
        alg.storage.clear()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for k in range(T_GAE):
            alg.act(*alg.storage.observation_slot(k))
            alg.process_env_step(rew_, done_, infos_)
        b.record(stream)
        b.synchronize()
        roll_ms = a.elapsed_time(b) / T_GAE
    reps = max(2, args.ppo_updates)
    upd_sampler = ClockSampler(dev.index or 0)          # SM clock under the update's GEMM load (the power cap acts here)
    upd_sampler.start()
    ms = time_updates(alg, args, dev, n, world, rank, last, reps)
    update_clocks = upd_sampler.summary()
    samples = n * T_GAE * world
    passes = samples * PPO_CFG["num_learning_epochs"]
    tflops = passes * PPO_FLOP_PER_SAMPLE_PASS / (ms * 1e-3) / 1e12
    mean_kl, lr_after = alg.last_mean_kl, alg.learning_rate
    iteration = bench_iteration(env, phys, phys_frames, alg, dev, n) if env is not None else None
    # the fp32-grade mode (3xTF32: hi/lo split operands, three partial products per GEMM), same update
    fp32_grade = None
    if world == 1 and not args.skip_3xtf32:
        torch.manual_seed(5)
        ac3 = ActorCritic(615, 1050, 10, actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128], device=dev,
                          precision="3xtf32")
        alg3 = PPO(ac3, device=dev, **PPO_CFG)
        alg3.init_storage(n, T_GAE, [615], [1050], [10])
        ms3 = time_updates(alg3, args, dev, n, world, rank, last, 2)
        fp32_grade = {"value": samples / (ms3 * 1e-3), "unit": "samples/s", "ms_per_update": ms3,
                      "dtype": "3xTF32 (hi/lo split operands, f32 accumulate): fp32-grade results"}
        del alg3, ac3
    peak = measure_tf32_peak(dev) if rank == 0 or world == 1 else None
    out = {"value": samples / (ms * 1e-3), "unit": "samples/s", "sample_passes_per_s": passes / (ms * 1e-3),
           "iteration": iteration,
           "ms_per_update": ms, "T": T_GAE, "epochs": 5, "mini_batches": 4, "dtype": "tf32 operands, f32 accumulate",
           "tensor_tflops": tflops, "fp32_grade": fp32_grade,
           "gradient_exchange": ("single GPU" if world == 1 else
                                 ("hb_dp_optimizer_step over peer memory" + (" (NVLS multimem)" if alg._peer.multicast else " (peer loads / stores)")
                                  if alg._peer is not None else "NCCL all-reduce of the flat gradient + local optimizer step")),
           "mean_kl": mean_kl, "learning_rate": lr_after,
           "rollout_act_and_record_ms_per_step": roll_ms, "update_clocks": update_clocks}
    if peak is not None:
        # a whole update is a seconds-scale loop under the power cap: the sustained figure is the denominator
        out.update({"tensor_peak_tflops": peak["sustained_tflops"] * world, "tensor_frac": tflops / (peak["sustained_tflops"] * world),
                    "tensor_peak_burst_tflops": peak["burst_tflops"] * world,
                    "tensor_peak_source": "measured in this run: " + peak["how"] + " (sustained)"})
    return out


def run_b200(args, rank, world):
    import torch.distributed as dist
    from isaac_b200 import _lib
    from isaac_b200.algo.rollout_storage import gae_compute_returns
    from isaac_b200.envs.hector_config import HectorCfg
    from isaac_b200.envs.hector_env import HectorFreeEnvB200
    from isaac_b200.physics import SyntheticPhysics

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:                    # (the single-GPU run keeps every core: it also times the CPU baseline)
        bind_to_gpu_cpus(local)      # before any pinned allocation: first touch lands on the GPU's NUMA node
    lib = _lib.load(check_device=True)
    for kv in args.opt:
        k, v = kv.split("=")
        _lib.check(lib.hb_set_option(k.encode(), int(v)), f"hb_set_option({kv})")
    n = args.envs
    frames = 4
    tape = make_workload(n, frames, 1234 + rank)
    phys_frames = [f.to(dev) for f in tape.physics]
    noise_frames = [f.to(dev) for f in tape.noise]
    phys = SyntheticPhysics(n, device=dev)
    phys.load_frame(phys_frames[0])
    env = HectorFreeEnvB200(HectorCfg(), sim_device=str(dev), physics=phys, statics=tape.statics,
                            dense_rows=bool(os.environ.get("HB_DENSE_ROWS")),
                            initial_noise=noise_frames[0])
    env.episode_length_buf.copy_(tape.statics.episode_length0)
    if not args.no_graph:
        for i in range(3):          # eager warm-up (lazy module load, cudaFuncSetAttribute) before capture
            env.step(noise_frames[0].actions)
        env.enable_cuda_graph()
        env.prepare_action_buffers(*[f.actions for f in noise_frames])      # no graph capture inside a timed step
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)     # > 126 MB L2
    flush_sink = torch.zeros(1, device=dev)
    stream = torch.cuda.current_stream(dev)

    def flush_l2(i):
        """Outside every timed region: a 256 MiB write evicts the step's data, then a 256 MiB read leaves L2
        full of CLEAN lines - after a write-only flush the next kernel would pay for writing ~126 MB of dirty
        flush lines back to HBM inside its own timed region."""
        flush.fill_(float(i))
        flush_sink.copy_(flush.sum())

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    last_out = [None]

    def one_step(i, timed):
        f = i % frames
        phys.load_frame(phys_frames[f])
        flush_l2(i)
        if args.no_graph:
            env.inject_noise(noise_frames[f])   # eager path: noise tensors already resident in HBM
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        last_out[0] = env.step(noise_frames[f].actions)
        if timed:
            e1.record(stream)
            return e0, e1

    sampler = ClockSampler(local)       # samples through warm-up, the timed steps and the per-kernel timings
    sampler.start()
    for i in range(args.warmup):
        one_step(i, False)
    barrier()
    lib.hb_launch_count_reset()
    t0 = time.perf_counter()
    evs = [one_step(args.warmup + i, True) for i in range(args.steps)]
    barrier()
    wall = time.perf_counter() - t0
    launches = lib.hb_launch_count() + (0 if args.no_graph else args.steps * env.graph_launches_per_step)
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    if args.dump_outputs and rank == 0:          # before the kernel timings below reuse the env's buffers
        dump_outputs(args.dump_outputs, last_out[0])

    # ---- per-kernel timings for the roofline (each launch alone, L2 flushed before it) ----
    def time_launch(fn, reps=10):
        """One launch, replayed from a single-node CUDA graph so that the host-side launch path (ctypes,
        argument marshalling) stays out of the event interval; L2 flushed before every replay."""
        def body(st_):
            rc = fn(st_)
            if rc not in (0, None):
                _lib.check(rc, "time_launch")
        g = _lib.LaunchGraph(dev).record(body)
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
        return tot / reps

    def time_chain(fns, reps=10):
        """Average duration of len(fns) back-to-back launches replayed from one CUDA graph, each launch on its own
        (cold) buffers: the graph-launch latency in front of the first kernel is amortised over the chain."""
        def body(st_):
            for fn in fns:
                rc = fn(st_)
                if rc not in (0, None):
                    _lib.check(rc, "time_chain")
        g = _lib.LaunchGraph(dev).record(body)
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
        return tot / reps / len(fns)

    (o_prev, p_prev), (o_cur, p_cur) = env._own[0][:2], env._own[1][:2]      # the env's own pair; rows at the 640 / 1056-float pitch
    P, B = env._pp, env._pb
    rb = None            # unconditional shift (reset envs are zeroed by hb_env_reset_finalize)
    dense = [torch.randn(n, w, device=dev) for w in (STACK_PRIV * FRAME_PRIV, STACK_PRIV * FRAME_PRIV,
                                                     STACK_OBS * FRAME_OBS, STACK_OBS * FRAME_OBS)]
    k_priv = time_launch(lambda st: lib.hb_stack_shift(dense[0].data_ptr(), dense[1].data_ptr(), rb, n,
                                                    STACK_PRIV * FRAME_PRIV, FRAME_PRIV, st))
    k_obs = time_launch(lambda st: lib.hb_stack_shift(dense[2].data_ptr(), dense[3].data_ptr(), rb, n,
                                                   STACK_OBS * FRAME_OBS, FRAME_OBS, st))
    del dense
    # short kernels: chains (CUDA events tick in ~2 us steps), per-launch time = chain / length
    k_pd = time_chain([lambda st: lib.hb_env_compute_torques(P, B, st)] * 8)
    env._draw_noise(False)              # device generator, like the replayed step
    k_post = time_chain([lambda st: lib.hb_env_post_physics(P, B, env._pn, o_cur.data_ptr(), p_cur.data_ptr(),
                                                         _lib.HB_STAGE_STEP, st)] * 4)
    k_fin = time_chain([lambda st: lib.hb_env_reset_finalize(P, B, o_cur.data_ptr(), p_cur.data_ptr(),
                                                          env._host_count.data_ptr(), None, st)] * 4)
    k_stack_single = time_launch(lambda st: lib.hb_env_stack_observations(P, B, o_prev.data_ptr(), p_prev.data_ptr(),
                                                                       o_cur.data_ptr(), p_cur.data_ptr(), st))
    # the roofline kernel: 4 launches per timed replay, each on its own cold set of history buffers
    CHAIN = 4
    ld_o, ld_p = env._p.obs_ld, env._p.priv_ld
    sets = [(torch.randn(n, ld_o, device=dev), torch.randn(n, ld_p, device=dev), torch.empty(n, ld_o, device=dev),
             torch.empty(n, ld_p, device=dev)) for _ in range(CHAIN)]
    k_stack = time_chain([(lambda st, s_=s_: lib.hb_env_stack_finalize(P, B, s_[0].data_ptr(), s_[1].data_ptr(),
                                                                      s_[2].data_ptr(), s_[3].data_ptr(),
                                                                      env._host_count.data_ptr(), None, st)) for s_ in sets])
    del sets
    # GAE: CUDA events tick in ~2 us steps on this driver, so one short launch cannot be timed alone - a graph of 8
    # launches on 8 distinct (cold) buffer sets, / 8
    g = torch.Generator().manual_seed(rank)
    gsets = []
    for _ in range(8):
        r_, v_ = torch.rand(T_GAE, n, 1, generator=g).to(dev), torch.randn(T_GAE, n, 1, generator=g).to(dev)
        d_, lv_ = (torch.rand(T_GAE, n, 1, generator=g) < 0.005).byte().to(dev), torch.randn(n, 1, generator=g).to(dev)
        gsets.append((r_, v_, d_, lv_, torch.empty_like(r_), torch.empty_like(r_)))
    gae_compute_returns(*gsets[0], 0.994, 0.9)          # allocates the launch's scratch before capture
    gae_stats = torch.zeros(2, dtype=torch.float64, device=dev)

    def gae_chain(**kw):
        return time_chain([(lambda st, s_=s_: gae_compute_returns(*s_, 0.994, 0.9, **kw) and 0) for s_ in gsets])

    k_gae = gae_chain()                                  # hb_gae_fused: one launch
    lib.hb_set_option(b"coop_launch", 1)
    k_gae_coop = gae_chain()
    lib.hb_set_option(b"coop_launch", 0)
    k_gae_two = gae_chain(stats=gae_stats)               # memset + scan + normalise
    del gsets
    clocks = sampler.summary()          # the env-stage measurement (the headline value and its roofline) ends here
    ppo_sampler = ClockSampler(local)   # the GEMM-heavy PPO legs draw more power: their clocks are reported with them
    ppo_sampler.start()
    ppo = None if args.skip_ppo else bench_ppo(args, dev, n, world, rank, env, phys, phys_frames)
    ppo_clocks = ppo_sampler.summary()
    if ppo is not None:
        ppo["clocks"] = ppo_clocks

    # ---- e2e: host buffers in, host buffers out, env's own noise ----
    # Pipelined like a host consumer would run it: the two big results of step k (obs, privileged obs: 27 MB at 4096
    # envs) leave on a copy stream into one of two pinned buffer sets while step k+1 already runs; the host only waits
    # for the buffer set it is about to read (step k-1's), and a step may not start overwriting an observation buffer
    # whose copy is still in flight.  Rewards and resets are single device buffers that the next step overwrites: they
    # are copied in stream order behind the step (20 KB).  Every step's inputs come from pinned host memory.
    host_frames = [type(f)(*(t.cpu().pin_memory() for t in (f.root_states, f.dof_state, f.contact_forces, f.rigid_state)))
                   for f in tape.physics]
    host_actions = [f.actions.pin_memory() for f in tape.noise]
    # dense host images; each observation tensor (rows at the device's 128-byte pitch) leaves as ONE 2-D DMA copy (hb_copy_rows)
    out_host = [[torch.empty(n, env.num_obs).pin_memory(), torch.empty(n, env.num_privileged_obs).pin_memory(),
                 torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.bool).pin_memory()] for _ in range(2)]
    act_dev = torch.empty(n, 10, device=dev)
    copy_stream = torch.cuda.Stream(dev)
    ev_step = [torch.cuda.Event() for _ in range(2)]
    ev_copied = [torch.cuda.Event() for _ in range(2)]
    checksum = [0.0]

    def copy_rows(dst, src, st):          # [n, width] view of pitched device rows -> dense pinned host rows
        _lib.check(lib.hb_copy_rows(dst.data_ptr(), dst.stride(0) * 4, src.data_ptr(), src.stride(0) * 4, src.shape[1] * 4,
                                    src.shape[0], st.cuda_stream), "hb_copy_rows")

    def consume(slot):          # the caller's read of a finished step: waits for that buffer set only
        ev_copied[slot].synchronize()
        checksum[0] += float(out_host[slot][2][0])

    def e2e_step(i):
        f, slot = i % frames, i & 1
        if i >= 2:
            stream.wait_event(ev_copied[slot])       # step i reuses the observation buffers step i-2's copies read
        phys.load_frame(host_frames[f])
        act_dev.copy_(host_actions[f], non_blocking=True)
        out = env.step(act_dev)
        out_host[slot][2].copy_(out[2], non_blocking=True)
        out_host[slot][3].copy_(out[3], non_blocking=True)
        ev_step[slot].record(stream)
        copy_stream.wait_event(ev_step[slot])
        with torch.cuda.stream(copy_stream):
            copy_rows(out_host[slot][0], out[0], copy_stream)
            copy_rows(out_host[slot][1], out[1], copy_stream)
            ev_copied[slot].record(copy_stream)
        if i >= 1:
            consume(slot ^ 1)                        # hand step i-1's results to the caller

    def e2e_run(k, step_fn=None, last=None):
        step_fn = step_fn or e2e_step
        for i in range(k):
            step_fn(i)
        (last or consume)((k - 1) & 1)               # the last step's results
        torch.cuda.synchronize(dev)

    e2e_run(max(4, args.warmup))
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    barrier()
    e2e_full_wall = time.perf_counter() - t0

    # ---- e2e through the host mirror (isaac_b200.envs.host_mirror): the same host-visible results - obs / privileged obs
    # as [N, 615] / [N, 1050] host tensors, rewards, resets - but only the NEWEST frames cross PCIe: a step's stack is the
    # previous one shifted by a frame, so the GPU appends the new frames to per-env rings in pinned memory and the
    # stacked observations are strided views of those rings.  Same pipeline: step k+1 and its frame copies are enqueued
    # before the caller reads step k (the GPU never rewrites slots that an earlier step's views still show).
    from isaac_b200.envs.host_mirror import HostObservationMirror
    mirror = HostObservationMirror(env, spare=int(os.environ.get("HB_MIRROR_SPARE", "17")), use_dma=os.environ.get("HB_MIRROR_DMA", "1") != "0")
    small_host = [[torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.bool).pin_memory()] for _ in range(2)]
    reset_snap = [torch.empty(n, dtype=torch.bool, device=dev) for _ in range(2)]
    tickets = [None, None]
    last_views = [None]

    def consume_mirror(slot):          # the caller's read of a finished step: waits for that step's frames only
        ho, hp = last_views[0] = mirror.views(tickets[slot])
        checksum[0] += float(small_host[slot][0][0]) + float(ho[0, -1]) + float(hp[n - 1, 0])

    trace = [0.0] * 6 if os.environ.get("HB_E2E_TRACE") else None

    def e2e_mirror_step(i):
        f, slot = i % frames, i & 1
        t_0 = time.perf_counter()
        if i >= 2:
            stream.wait_event(ev_copied[slot])       # step i reuses the observation buffers update i-2 read
        phys.load_frame(host_frames[f])
        act_dev.copy_(host_actions[f], non_blocking=True)
        t_1 = time.perf_counter()
        out = env.step(act_dev)
        t_2 = time.perf_counter()
        small_host[slot][0].copy_(out[2], non_blocking=True)
        small_host[slot][1].copy_(out[3], non_blocking=True)
        reset_snap[slot].copy_(out[3], non_blocking=True)      # the next step overwrites reset_buf while the copy stream still reads it
        ev_step[slot].record(stream)
        t_3 = time.perf_counter()
        copy_stream.wait_event(ev_step[slot])
        torch.cuda.set_stream(copy_stream)
        tickets[slot] = mirror.update(out[0], out[1], reset_snap[slot])
        ev_copied[slot].record(copy_stream)
        torch.cuda.set_stream(stream)
        t_4 = time.perf_counter()
        if i >= 1:
            consume_mirror(slot ^ 1)                 # the caller reads step i-1 while step i's frames are on their way
        if trace is not None:
            t_5 = time.perf_counter()
            for q, (a_, b_) in enumerate(((t_0, t_1), (t_1, t_2), (t_2, t_3), (t_3, t_4), (t_4, t_5))):
                trace[q] += b_ - a_
            trace[5] += 1

    torch.cuda.synchronize(dev)
    mirror.resync(env.get_observations(), env.get_privileged_observations())
    e2e_run(max(4, args.warmup), e2e_mirror_step, consume_mirror)
    # the mirrored views equal the device tensors (checked here on the last warm-up step, and step by step in tests/test_host_mirror.py)
    assert torch.equal(last_views[0][0], env.get_observations().cpu()), "host mirror differs from the device stack"
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps, e2e_mirror_step, consume_mirror)
    barrier()
    e2e_wall = time.perf_counter() - t0
    if trace is not None and rank == 0:
        print("e2e host time per step (us): inputs %.1f | env.step %.1f | small copies %.1f | mirror.update %.1f | consume (wait) %.1f" %
              tuple(1e6 * v / trace[5] for v in trace[:5]), file=sys.stderr, flush=True)
    h2d = sum(t.numel() * t.element_size() for t in (host_frames[0].root_states, host_frames[0].dof_state,
                                                      host_frames[0].contact_forces, host_frames[0].rigid_state,
                                                      host_actions[0]))
    d2h_full = sum(t.numel() * t.element_size() for t in out_host[0])
    d2h = mirror.bytes_per_update + sum(t.numel() * t.element_size() for t in small_host[0])

    t = torch.tensor([dev_ms, wall, e2e_wall, k_priv, k_obs, k_pd, k_gae, k_post, k_stack, k_fin, k_stack_single, e2e_full_wall],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall, e2e_wall, k_priv, k_obs, k_pd, k_gae, k_post, k_stack, k_fin, k_stack_single, e2e_full_wall = t.tolist()
    if rank != 0:
        return
    peak, peak_src = peaks()
    total_envs = n * world
    value = total_envs * args.steps / (dev_ms * 1e-3)
    hist_priv = n * 2 * (STACK_PRIV - 1) * FRAME_PRIV * 4          # read + write of the carried frames
    hist_obs = n * 2 * (STACK_OBS - 1) * FRAME_OBS * 4
    ach = (hist_priv + hist_obs) / (k_stack * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):           # dram bytes of one launch from the committed ncu --set full captures, per shard size
        traffic = json.load(open(tpath)).get("bytes_per_launch", {}).get(str(n))      # null when this size was not captured
    line = {
        "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(n),
                   "envs_per_gpu": n, "decimation": 10, "frame_stack": 15,
                   "launch": "eager, noise tensors resident in HBM" if args.no_graph else
                             "CUDA-graph replay (2 graphs/step around the reset-count hand-off), noise drawn in-kernel (Philox)",
                   "timing": "per-step CUDA events, L2 flushed between steps (256 MiB write then 256 MiB read, outside the events)",
                   "wall_ms_per_step_incl_flush": 1e3 * wall / args.steps},
        "clocks": clocks,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm",
                     "kernel": "stack_finalize_kernel (frame stacking: 14 carried frames of 41 + 70 floats, read + write; the "
                               "shard-wide reset results ride in the last blocks of the same launch)",
                     "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": hist_priv + hist_obs,
                     "launch_ms": k_stack,
                     "timing": "CUDA events around a graph of 4 launches on 4 distinct cold buffer sets (L2 flushed before), / 4",
                     "single_launch_ms_incl_graph_launch_latency": k_stack_single},
        "roofline_step": {"bytes_per_env_step": B_ENV_STEP, "achieved": value / world * B_ENV_STEP / 1e9,
                          "peak": peak, "unit": "GB/s", "frac": value / world * B_ENV_STEP / 1e9 / peak},
        "kernels": {"post_physics_ms": k_post, "reset_finalize_ms": k_fin, "stack_pair_ms": k_stack,
                    "stack_pair_gbs": (hist_obs + hist_priv) / (k_stack * 1e-3) / 1e9,
                    "stack_priv_ms": k_priv, "stack_obs_ms": k_obs,
                    "stack_obs_gbs": hist_obs / (k_obs * 1e-3) / 1e9, "pd_ms": k_pd,
                    "pd_gbs": n * 240 / (k_pd * 1e-3) / 1e9, "gae_ms": k_gae, "gae_cooperative_launch_ms": k_gae_coop, "gae_two_kernel_form_ms": k_gae_two,
                    "gae_gbs": n * T_GAE * 25 / (k_gae * 1e-3) / 1e9},
        "gae": {"value": total_envs * T_GAE / (k_gae * 1e-3), "unit": "samples/s", "T": T_GAE},
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(n)
    # the last keys of the line (a truncated tail still carries them): PPO samples/s and the end-to-end number
    line["ppo"] = ppo
    line["e2e"] = {"value": total_envs * args.steps / e2e_wall, "unit": "env-steps/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_wall / args.steps,
                   "d2h_gbs_per_gpu": d2h * args.steps / e2e_wall / 1e9,
                   "pipeline": "HostObservationMirror (isaac_b200/envs/host_mirror.py): every step's inputs come from pinned host "
                               "memory, its results are host tensors - rewards / resets copied, obs [N,615] / privileged obs "
                               "[N,1050] as strided views of pinned per-env frame rings to which the GPU appends only the step's "
                               "NEWEST frames (hb_env_mirror_frames, 2-D DMA copies: a stack is the previous one shifted by a frame); bit-equal to "
                               "the device tensors (asserted in this run, tests/test_host_mirror.py); step k+1 and its frame copies are "
                               "enqueued before the caller reads step k; CPU affinity = the GPU's NUMA node",
                   "full_stack_copy": {"value": total_envs * args.steps / e2e_full_wall, "unit": "env-steps/s",
                                       "d2h_bytes_per_step": d2h_full, "ms_per_step": 1e3 * e2e_full_wall / args.steps,
                                       "d2h_gbs_per_gpu": d2h_full * args.steps / e2e_full_wall / 1e9,
                                       "pipeline": "the whole obs / privileged-obs stacks of step k leave by DMA (hb_copy_rows) into "
                                                   "double-buffered dense pinned tensors while step k+1 runs (what the reference's "
                                                   "obs.to(rl_device) moves, on_policy_runner.py:136)"}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--envs", type=int, default=4096, help="envs per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly from Python")
    ap.add_argument("--opt", action="append", default=[], help="library tuning switch name=value (hb_set_option)")
    ap.add_argument("--skip-ppo", action="store_true", help="env stage only (tuning sweeps)")
    ap.add_argument("--ppo-updates", type=int, default=3, help="timed PPO updates (after one warm-up)")
    ap.add_argument("--skip-3xtf32", action="store_true", help="do not time the fp32-grade (3xTF32) update as well")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what env.step() returned in the last timed step as "
                                                          "DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        # stdout carries exactly one JSON line: NCCL's banner ("NCCL version ...", printed to stdout when
        # NCCL_DEBUG=VERSION/INFO) is sent to stderr while the communicator comes up
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    try:
        run_b200(args, rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
