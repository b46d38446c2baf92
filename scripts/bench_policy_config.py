"""Device time of one PPO update per policy configuration: hector's networks (actor 512-256-128, critic 768-256-128) with
each activation of get_activation, and one deeper pair (four hidden layers each), next to the ELU default.

    python scripts/bench_policy_config.py [--rounds R] [--reps K] [--envs N]

One update = compute_returns + update() on a [24, N] rollout (default N = 4096), 5 epochs x 4 minibatches, TF32, the
per-minibatch graphs replayed - the update bench.py times.  The configurations are timed in turn, R rounds (default 3)
of K updates each (default 5) after warm-up, so that slow drift of the clock under the power cap spreads over all of
them; each round's mean is printed, and the median over rounds is compared with ELU.  The card's name and power limit
are read in the same run, since the numbers depend on both."""
import argparse
import json
import os
import statistics
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import torch

import bench
from isaac_b200 import _lib
from isaac_b200.algo.actor_critic import ActorCritic
from isaac_b200.algo.ppo import PPO

HECTOR = dict(actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128])
DEEP = dict(actor_hidden_dims=[512, 256, 256, 128], critic_hidden_dims=[768, 256, 256, 128])
CONFIGS = [("elu", HECTOR, "elu"), ("selu", HECTOR, "selu"), ("relu", HECTOR, "relu"), ("lrelu", HECTOR, "lrelu"),
           ("tanh", HECTOR, "tanh"), ("sigmoid", HECTOR, "sigmoid"), ("elu, 4+4 hidden layers", DEEP, "elu")]


def card(dev):
    """Name and enforced power limit (W) of the device."""
    name, limit = torch.cuda.get_device_name(dev), None
    try:
        import pynvml as nv
        nv.nvmlInit()
        limit = nv.nvmlDeviceGetEnforcedPowerLimit(nv.nvmlDeviceGetHandleByIndex(dev.index or 0)) / 1000.0
    except Exception:
        pass
    return name, limit


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
    algs = []
    for label, net, act in CONFIGS:
        torch.manual_seed(5)
        ac = ActorCritic(615, 1050, 10, **net, activation=act, device=dev)
        alg = PPO(ac, device=dev, **bench.PPO_CFG)
        alg.init_storage(n, T, [615], [1050], [10])
        bench.time_updates(alg, args, dev, n, 1, 0, last, 1)          # warm-up: modules, graphs of every minibatch
        algs.append(alg)
    times = {label: [] for label, _, _ in CONFIGS}
    for _ in range(args.rounds):
        for (label, _, _), alg in zip(CONFIGS, algs):
            times[label].append(bench.time_updates(alg, args, dev, n, 1, 0, last, args.reps))
    name, limit = card(dev)
    base = statistics.median(times["elu"])
    print(f"{name}, power limit {limit if limit is None else f'{limit:.0f} W'}; {n} envs x {T} steps, "
          f"{bench.PPO_CFG['num_learning_epochs']} epochs x {bench.PPO_CFG['num_mini_batches']} minibatches, TF32")
    print(f"{'configuration':<26}{'ms / update (median)':>22}{'vs elu':>9}   per round")
    rows = []
    for label, net, act in CONFIGS:
        med = statistics.median(times[label])
        print(f"{label:<26}{med:>22.2f}{med / base:>9.3f}   " + " ".join(f"{t:.2f}" for t in times[label]))
        rows.append(dict(config=label, activation=act, **net, ms_per_update=med, rounds=times[label], vs_elu=med / base))
    print(json.dumps({"device": name, "power_limit_w": limit, "envs": n, "steps": T, "results": rows}))


if __name__ == "__main__":
    main()
