"""Device time of one PPO update and of one PPO.act per action count: hector's observation widths (615 / 1050) and
networks (actor 512-256-128, critic 768-256-128), ELU, for counts on the fused heads (7, 10, 15) and on the generic path
(19, 23, 29).  10 runs the kernels compiled for hector's count, so its update time is the one bench.py's `ppo` line
reports; the other counts run the runtime-count instantiations.

    python scripts/bench_num_actions.py [--rounds R] [--reps K] [--envs N]

One update = compute_returns + update() on a [24, N] rollout (default N = 4096), 5 epochs x 4 minibatches, TF32, with
bench.py's PPO settings; the fused counts replay the per-minibatch graphs.  One act = PPO.act + process_env_step for a
rollout step whose observations are already in the storage slot, averaged over the 24 steps of a rollout (the fused counts
replay the slot's act graph).  The counts are timed in turn, R rounds (default 3) of K updates (default 5) and one
rollout each after warm-up, so that drift of the clock under the power cap spreads over all of them; the median over
rounds is printed.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import torch

import bench
from bench_policy_config import HECTOR, card
from isaac_b200 import _lib
from isaac_b200.algo.actor_critic import ActorCritic
from isaac_b200.algo.ppo import PPO

COUNTS = [7, 10, 15, 19, 23, 29]


def fill_storage(st, seed, dev):
    """bench.fill_storage for any action count."""
    g = torch.Generator(device=dev).manual_seed(seed)
    T, N, A = st.num_transitions_per_env, st.num_envs, st.actions.shape[-1]
    st.observations.copy_(torch.randn(T, N, 615, device=dev, generator=g))
    st.privileged_observations.copy_(torch.randn(T, N, 1050, device=dev, generator=g))
    st.actions.copy_(torch.randn(T, N, A, device=dev, generator=g))
    st.mu.copy_(st.actions + 0.3 * torch.randn(T, N, A, device=dev, generator=g))
    st.sigma.fill_(1.0)
    st.rewards.copy_(torch.rand(T, N, 1, device=dev, generator=g) * 0.05)
    st.values.copy_(torch.randn(T, N, 1, device=dev, generator=g) * 0.5)
    st.dones.copy_((torch.rand(T, N, 1, device=dev, generator=g) < 0.005).to(torch.uint8))
    st.actions_log_prob.copy_(-0.5 * ((st.actions - st.mu) ** 2).sum(-1, keepdim=True) - 0.919 * A)


def time_updates(alg, dev, last, reps):
    """Mean device time (ms) of compute_returns + update() over `reps` updates."""
    stream = torch.cuda.current_stream(dev)
    times = []
    for _ in range(reps):
        fill_storage(alg.storage, 100, dev)
        alg.storage.step = bench.T_GAE
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        alg.compute_returns(last)
        alg.update()
        b.record(stream)
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sum(times) / len(times)


def time_act(alg, dev, rew, done, infos):
    """Mean device time (us) of PPO.act + process_env_step over the steps of one rollout."""
    stream = torch.cuda.current_stream(dev)
    alg.storage.clear()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for k in range(bench.T_GAE):
        alg.act(*alg.storage.observation_slot(k))
        alg.process_env_step(rew, done, infos)
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / bench.T_GAE


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--envs", type=int, default=4096)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    _lib.load(check_device=True)
    n, T = args.envs, bench.T_GAE
    last = torch.randn(n, 1050, device=dev)
    rew, done = torch.rand(n, device=dev), torch.rand(n, device=dev) < 0.005
    infos = {"time_outs": torch.rand(n, device=dev) < 0.0004}
    algs = {}
    for na in COUNTS:
        torch.manual_seed(5)
        ac = ActorCritic(615, 1050, na, **HECTOR, device=dev)
        alg = PPO(ac, device=dev, **bench.PPO_CFG)
        alg.init_storage(n, T, [615], [1050], [na])
        alg.storage.observations.normal_(), alg.storage.privileged_observations.normal_()
        time_act(alg, dev, rew, done, infos)            # warm-up: modules, the act graph of every slot
        time_updates(alg, dev, last, 2)                  # warm-up: the second update captures the minibatch graphs
        algs[na] = alg
    upd, act = {na: [] for na in COUNTS}, {na: [] for na in COUNTS}
    for _ in range(args.rounds):
        for na, alg in algs.items():
            act[na].append(time_act(alg, dev, rew, done, infos))
            upd[na].append(time_updates(alg, dev, last, args.reps))
    name, limit = card(dev)
    print(f"{name}, power limit {limit if limit is None else f'{limit:.0f} W'}; {n} envs x {T} steps, "
          f"{bench.PPO_CFG['num_learning_epochs']} epochs x {bench.PPO_CFG['num_mini_batches']} minibatches, TF32")
    print(f"{'actions':>8}{'path':>9}{'ms / update':>13}{'us / act':>10}   per round (ms / update; us / act)")
    rows = []
    for na, alg in algs.items():
        path = "fused" if alg.actor_critic.fused_head else "generic"
        mu, ma = statistics.median(upd[na]), statistics.median(act[na])
        print(f"{na:>8}{path:>9}{mu:>13.2f}{ma:>10.1f}   " + " ".join(f"{t:.2f}" for t in upd[na]) + "; "
              + " ".join(f"{t:.1f}" for t in act[na]))
        rows.append(dict(num_actions=na, path=path, ms_per_update=mu, us_per_act=ma, update_rounds=upd[na], act_rounds=act[na]))
    print(json.dumps({"device": name, "power_limit_w": limit, "envs": n, "steps": T, "results": rows}))


if __name__ == "__main__":
    main()
