"""TEST INFRASTRUCTURE — the CPU oracle of oracle/ppo_oracle.py for any depth and activation.

`oracle/ppo_oracle.py` is the pinned restatement of the reference (tests/test_oracle_pinning.py) and states hector's
networks: three hidden layers, ELU.  The reference's ActorCritic (actor_critic.py:36-128) takes any `actor_hidden_dims` /
`critic_hidden_dims` and an `activation` resolved by get_activation.  This module extends the oracle to that space
without restating it: `mlp` walks the layers present in `params`, and `PolicyOraclePPO` runs OraclePPO's own methods
with its network (`mlp` and `PARAM_ORDER` of oracle.ppo_oracle bound to this net for the duration of each call), so the
PPO arithmetic compared against is the pinned one.  With the defaults both compute exactly what oracle.ppo_oracle does.
"""
from __future__ import annotations

from contextlib import contextmanager
from typing import List

import torch
import torch.nn.functional as F

import oracle.ppo_oracle as po

# get_activation (actor_critic.py): the module each name builds, as the function it applies ("crelu" is nn.ReLU there)
ACTIVATIONS = {"elu": F.elu, "selu": F.selu, "relu": F.relu, "crelu": F.relu, "lrelu": F.leaky_relu, "tanh": torch.tanh,
               "sigmoid": torch.sigmoid}


def depth(params, net: str) -> int:
    """Number of nn.Linear layers of `net` in `params` (hidden layers + the output layer)."""
    return sum(1 for k in params if k.startswith(net + ".") and k.endswith(".weight"))


def param_order(params) -> List[str]:
    """The reference module's parameters() order for the networks in `params`: std, then the actor's and the critic's
    layers, weight before bias (oracle.ppo_oracle.PARAM_ORDER for three hidden layers each)."""
    return ["std"] + [f"{net}.{2 * i}.{w}" for net in ("actor", "critic") for i in range(depth(params, net))
                      for w in ("weight", "bias")]


def mlp(params, net: str, x: torch.Tensor, activation: str = "elu") -> torch.Tensor:
    """(Linear, activation) per hidden layer, then the output Linear (actor_critic.py:54-77), over the layers in `params`."""
    act, n = ACTIVATIONS[activation], depth(params, net)
    for i in range(0, 2 * (n - 1), 2):
        x = act(F.linear(x, params[f"{net}.{i}.weight"], params[f"{net}.{i}.bias"]))
    return F.linear(x, params[f"{net}.{2 * (n - 1)}.weight"], params[f"{net}.{2 * (n - 1)}.bias"])


class PolicyOraclePPO(po.OraclePPO):
    """OraclePPO for the networks in `params` and `activation` (same constructor otherwise)."""

    def __init__(self, params, *args, activation: str = "elu", **kwargs):
        self.order, self.activation = param_order(params), activation
        with self._network():
            super().__init__(params, *args, **kwargs)

    @contextmanager
    def _network(self):
        saved = po.mlp, po.PARAM_ORDER
        po.mlp = lambda p, net, x: mlp(p, net, x, self.activation)
        po.PARAM_ORDER = self.order
        try:
            yield
        finally:
            po.mlp, po.PARAM_ORDER = saved

    def act(self, *args, **kwargs):
        with self._network():
            return super().act(*args, **kwargs)

    def compute_returns(self, *args, **kwargs):
        with self._network():
            return super().compute_returns(*args, **kwargs)

    def update(self, *args, **kwargs):
        with self._network():
            return super().update(*args, **kwargs)
