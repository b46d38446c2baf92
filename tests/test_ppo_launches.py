"""Which library calls PPO makes, in what order and with which GEMM shapes: the launch counts and the grouped actor /
critic pairs that the timings of DESIGN.md §4 rest on.  A recorder stands in for the library handle of PPO and its
ActorCritic: it forwards every hb_* call and logs its name and, for the GEMM entry points, each descriptor.  The
expected descriptors are derived from ActorCritic.layers and the 128-byte row pitch of the activation buffers."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DESC_FIELDS = ("M", "N", "K", "lda", "ldb", "ldd", "a_mn_major", "b_mn_major", "epilogue", "split_k", "precision")


class Recorder:
    def __init__(self, lib):
        self.lib, self.calls, self.capturing = lib, [], []

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if not name.startswith("hb_") or name == "hb_gemm_workspace_floats":      # the latter only sizes 3xTF32 scratch
            return fn

        def call(*args):
            descs = [a._obj for a in args[:-1]] if name in ("hb_gemm_tf32", "hb_gemm_tf32_grouped") else []
            self.calls.append((name, *(tuple(getattr(d, f) for f in DESC_FIELDS) for d in descs)))
            self.capturing.append(torch.cuda.is_current_stream_capturing())
            return fn(*args)
        return call


def record(alg, fn):
    rec = Recorder(alg._lib)
    alg._lib = alg.actor_critic._lib = rec
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        alg._lib = alg.actor_critic._lib = rec.lib
    return rec


def make_alg(dev, task, precision="tf32", n=64, t=4):
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    from isaac_b200.envs import TASKS
    _, cfg_cls, ppo_cls = TASKS[task]
    ec, pc = cfg_cls().env, ppo_cls().policy
    ac = ActorCritic(ec.num_observations, ec.num_privileged_obs, ec.num_actions, actor_hidden_dims=pc.actor_hidden_dims,
                     critic_hidden_dims=pc.critic_hidden_dims, device=dev, precision=precision)
    assert ac.fused_head == (task == "hector")
    alg = PPO(ac, device=dev, num_learning_epochs=1, num_mini_batches=2, schedule="fixed")
    alg.init_storage(n, t, [ec.num_observations], [ec.num_privileged_obs], [ec.num_actions])
    return alg


def observations(alg, g):
    """Observation views at the rollout storage's row pitch, so that the GEMMs read them in place."""
    from isaac_b200.algo.actor_critic import pitch
    ac, n = alg.actor_critic, alg.storage.num_envs
    views = []
    for width in (ac.num_actor_obs, ac.num_critic_obs):
        buf = torch.zeros(n, pitch(width + 1))
        buf[:, :width] = torch.randn(n, width, generator=g)
        views.append(buf.to(alg.device)[:, :width])
    return views


# ---- expected descriptors: (M, N, K, lda, ldb, ldd, a_mn_major, b_mn_major, epilogue, split_k, precision) of layer i
def _layer(ac, net, i):
    return [L for L in ac.layers if L.net == net][i]


def _d_ld(L):
    """Row pitch of the gradient w.r.t. layer L's output: d_out [m, rows] for an output layer, else dz [m, pitch(width)]."""
    from isaac_b200.algo.actor_critic import pitch
    return L.rows if L.last else pitch(L.fan_out)


def fwd(ac, net, i, m, prec):
    from isaac_b200._lib import HB_EPI_BIAS, HB_EPI_BIAS_ELU
    from isaac_b200.algo.actor_critic import pitch
    L = _layer(ac, net, i)
    # inputs and hidden activations: rows of fan_in + the ones column at a 128-byte pitch
    return (m, L.rows if L.last else L.fan_out, L.fan_in, pitch(L.fan_in + 1), L.ld,
            L.rows if L.last else pitch(L.fan_out + 1), 0, 0, HB_EPI_BIAS if L.last else HB_EPI_BIAS_ELU, 0, prec)


def wgrad(ac, net, i, m, prec):
    from isaac_b200._lib import HB_EPI_ATOMIC_ADD
    from isaac_b200.algo.actor_critic import pitch
    L = _layer(ac, net, i)
    return (L.rows, L.fan_in + 1, m, _d_ld(L), pitch(L.fan_in + 1), L.ld, 1, 1, HB_EPI_ATOMIC_ADD, 0, prec)


def dgrad(ac, net, i, m, prec):
    from isaac_b200._lib import HB_EPI_ELU_BWD
    from isaac_b200.algo.actor_critic import pitch
    L = _layer(ac, net, i)
    return (m, L.fan_in, L.rows, _d_ld(L), L.ld, pitch(L.fan_in), 0, 1, HB_EPI_ELU_BWD, 0, prec)


def grouped(desc, ac, i, m, prec):
    return ("hb_gemm_tf32_grouped", desc(ac, "critic", i, m, prec), desc(ac, "actor", i, m, prec))       # critic first


def grouped_forward(ac, m, prec):
    return [grouped(fwd, ac, i, m, prec) for i in range(3)]


def grouped_backward(ac, m, prec):
    """Layers 2, 1, 0: data gradient, then weight gradient (layer 0: weight gradient only)."""
    return [g for i in (2, 1, 0) for g in ([grouped(dgrad, ac, i, m, prec)] if i else []) + [grouped(wgrad, ac, i, m, prec)]]


def one_net_forward(ac, net, m, prec):
    return [("hb_gemm_tf32", fwd(ac, net, i, m, prec)) for i in range(4)]


def one_net_backward(ac, net, m, prec):
    """Layers 3, 2, 1, 0: weight gradient, then data gradient (layer 0: weight gradient only)."""
    return [("hb_gemm_tf32", d(ac, net, i, m, prec)) for i in (3, 2, 1, 0) for d in ((wgrad, dgrad) if i else (wgrad,))]


@pytest.mark.parametrize("task,graph", [("hector", False), ("hector", True), ("hector_full", False)],
                         ids=["hector-eager", "hector-graph", "hector_full-generic"])
def test_act_launches(lib, cuda_device, task, graph):
    """PPO.act on its own draw.  Fused head: the draw, three grouped hidden-layer launches, hb_ppo_act_fused - issued
    eagerly, or recorded once into the slot's graph.  Generic path: the draw, four GEMMs per network, hb_ppo_act_head."""
    from isaac_b200._lib import HB_GEMM_TF32
    alg = make_alg(cuda_device, task)
    alg.graph_rollout = graph
    ac, n = alg.actor_critic, alg.storage.num_envs
    obs, cobs = observations(alg, torch.Generator().manual_seed(0))
    rec = record(alg, lambda: alg.act(obs, cobs))
    if ac.fused_head:
        body = [*grouped_forward(ac, n, HB_GEMM_TF32), ("hb_ppo_act_fused",)]
    else:
        body = [*one_net_forward(ac, "actor", n, HB_GEMM_TF32), *one_net_forward(ac, "critic", n, HB_GEMM_TF32),
                ("hb_ppo_act_head",)]
    assert rec.calls == [("hb_ppo_draw_normal",), *body]
    assert rec.capturing == [graph] * len(rec.calls)
    assert len(alg._act_graphs) == int(graph)


@pytest.mark.parametrize("task,precision", [("hector", "tf32"), ("hector", "3xtf32"), ("hector_full", "tf32")],
                         ids=["hector", "hector-3xtf32", "hector_full-generic"])
def test_minibatch_step_launches(lib, cuda_device, task, precision):
    """minibatch_gradients + optimizer_step after prepare_minibatches.  Fused head: three grouped forward launches,
    hb_ppo_head_fused, five grouped backward launches.  Generic path: four forward GEMMs per network, hb_ppo_loss_head,
    seven backward GEMMs of the actor, then seven of the critic.  Then hb_optimizer_step."""
    from isaac_b200._lib import HB_GEMM_3XTF32, HB_GEMM_TF32
    dev = cuda_device
    alg = make_alg(dev, task, precision)
    ac, s = alg.actor_critic, alg.storage
    g = torch.Generator().manual_seed(1)
    for _ in range(s.num_transitions_per_env):
        obs, cobs = observations(alg, g)
        alg.act(obs, cobs)
        alg.process_env_step(torch.rand(s.num_envs, generator=g).to(dev), (torch.rand(s.num_envs, generator=g) < 0.1).to(dev),
                             {"time_outs": torch.zeros(s.num_envs, dtype=torch.bool, device=dev)})
    alg.compute_returns(cobs)
    alg.prepare_minibatches()
    rec = record(alg, lambda: (alg.minibatch_gradients(0), alg.optimizer_step(0)))
    m, prec = alg._mb, HB_GEMM_3XTF32 if precision == "3xtf32" else HB_GEMM_TF32
    if ac.fused_head:
        want = [*grouped_forward(ac, m, prec), ("hb_ppo_head_fused",), *grouped_backward(ac, m, prec)]
    else:
        want = [*one_net_forward(ac, "actor", m, prec), *one_net_forward(ac, "critic", m, prec), ("hb_ppo_loss_head",),
                *one_net_backward(ac, "actor", m, prec), *one_net_backward(ac, "critic", m, prec)]
    assert rec.calls == [*want, ("hb_optimizer_step",)]
    assert not any(rec.capturing)
