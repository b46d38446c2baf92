"""ActorCritic configured like the reference's (algo/ppo/actor_critic.py:36-128): `activation` from get_activation's set and
any number of hidden layers per network, with the activation evaluated in the GEMM epilogues (HB_EPI_BIAS_ACT /
HB_EPI_ACT_BWD, hb_gemm_desc.activation) and in the fused loss head (hb_ppo_loss_params.activation).

CPU: the any-depth oracle (tests/_policy_oracle.py) against the pinned one and against nn.Sequential built the
reference's way; the constructor's argument checks; the library's rejection of bad activation descriptors.  GPU: each
epilogue against torch fp64 forward / autograd, the fused head per activation, each activation's minibatch gradients and
PPO end to end against the oracle, the reference-style module's state_dict and initialisation, checkpoints through
OnPolicyRunner, and the launch sequence of an unequal-depth pair."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from _util import assert_close
from oracle import make_golden as mg
from _policy_oracle import ACTIVATIONS as TORCH_ACTS, PolicyOraclePPO, mlp, param_order
from oracle import ppo_oracle
from oracle.ppo_oracle import OraclePPO, PARAM_ORDER, init_actor_critic_params
from isaac_b200.algo.actor_critic import ACTIVATIONS as HB_CODES

# the distinct kernels: "crelu" is nn.ReLU in get_activation, so it is "relu" here
ACTS = ["elu", "selu", "relu", "lrelu", "tanh", "sigmoid"]
HB_ERR_BAD_ARG, HB_ERR_UNSUPPORTED = -1, -3

# hector's networks, an unequal-depth pair that still takes the fused head (both last hidden widths 128), and a pair
# whose last hidden widths are not 128 (output layers as GEMMs + hb_ppo_loss_head)
HECTOR = dict(actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128])
UNEQUAL = dict(actor_hidden_dims=[256, 128], critic_hidden_dims=[512, 256, 256, 256, 128])
GENERIC = dict(actor_hidden_dims=[256, 256], critic_hidden_dims=[384, 192, 160])


def reference_modules(num_obs, num_critic_obs, num_actions, actor_hidden_dims, critic_hidden_dims, activation,
                      init_noise_std=1.0):
    """The reference's ActorCritic layout (actor_critic.py:36-83, get_activation): actor, critic, std, built in that
    order from the global torch generator."""
    nn = torch.nn
    act = {"elu": nn.ELU(), "selu": nn.SELU(), "relu": nn.ReLU(), "crelu": nn.ReLU(), "lrelu": nn.LeakyReLU(),
           "tanh": nn.Tanh(), "sigmoid": nn.Sigmoid()}[activation]

    def sequential(n_in, hidden, n_out):
        layers = [nn.Linear(n_in, hidden[0]), act]
        for i in range(len(hidden)):
            if i == len(hidden) - 1:
                layers.append(nn.Linear(hidden[i], n_out))
            else:
                layers += [nn.Linear(hidden[i], hidden[i + 1]), act]
        return nn.Sequential(*layers)

    m = nn.Module()
    m.actor = sequential(num_obs, actor_hidden_dims, num_actions)
    m.critic = sequential(num_critic_obs, critic_hidden_dims, 1)
    m.std = nn.Parameter(init_noise_std * torch.ones(num_actions))
    return m


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------- CPU: oracle
def test_oracle_defaults_equal_the_pinned_oracle():
    """Hector's networks and ELU: the any-depth mlp and PolicyOraclePPO compute bit for bit what oracle.ppo_oracle does
    (act, compute_returns, a two-epoch update), and leave the pinned module as they found it."""
    params = init_actor_critic_params(seed=5)
    assert param_order(params) == PARAM_ORDER
    g = torch.Generator().manual_seed(0)
    obs, cobs = torch.randn(64, 615, generator=g), torch.randn(64, 1050, generator=g)
    assert torch.equal(mlp(params, "actor", obs), ppo_oracle.mlp(params, "actor", obs))
    assert torch.equal(mlp(params, "critic", cobs), ppo_oracle.mlp(params, "critic", cobs))
    cfg = dict(mg.PPO_ALG, schedule="adaptive", num_learning_epochs=2, num_mini_batches=2)
    n, t = 16, 4
    pinned, general = OraclePPO(params, n, t, **cfg), PolicyOraclePPO(params, n, t, **cfg)
    for _ in range(t):
        step = (torch.randn(n, 615, generator=g), torch.randn(n, 1050, generator=g), torch.randn(n, 10, generator=g))
        env = (torch.rand(n, generator=g), torch.rand(n, generator=g) < 0.1, {"time_outs": torch.rand(n, generator=g) < 0.1})
        assert torch.equal(pinned.act(*step), general.act(*step))
        pinned.process_env_step(*env), general.process_env_step(*env)
    last = torch.randn(n, 1050, generator=g)
    pinned.compute_returns(last), general.compute_returns(last)
    perm = torch.randperm(n * t, generator=g)
    assert pinned.update(perm) == general.update(perm) and pinned.lr_trace == general.lr_trace
    for k in PARAM_ORDER:
        assert torch.equal(pinned.params[k], general.params[k]), k
    assert ppo_oracle.mlp.__name__ == "mlp" and ppo_oracle.PARAM_ORDER == PARAM_ORDER


@pytest.mark.parametrize("activation", ACTS + ["crelu"])
@pytest.mark.parametrize("dims", [([300], [200]), ([256, 128], [512, 256, 256, 128]), ([160, 96, 128], [128])],
                         ids=["1-1", "2-4", "3-1"])
def test_oracle_equals_reference_sequential(activation, dims):
    ah, ch = dims
    params = init_actor_critic_params(48, 70, 10, ah, ch, seed=2)
    ref = reference_modules(48, 70, 10, ah, ch, activation)
    ref.load_state_dict(params, strict=True)
    assert param_order(params) == [k for k, _ in ref.named_parameters()]
    g = torch.Generator().manual_seed(1)
    obs, cobs = torch.randn(33, 48, generator=g), torch.randn(33, 70, generator=g)
    with torch.no_grad():
        assert torch.equal(mlp(params, "actor", obs, activation), ref.actor(obs))
        assert torch.equal(mlp(params, "critic", cobs, activation), ref.critic(cobs))


# ---------------------------------------------------------------------------------------------------- CPU: argument checks
@pytest.mark.parametrize("kwargs,match", [
    (dict(activation="swish"), "unknown activation"),
    (dict(actor_hidden_dims=[]), "actor_hidden_dims is empty"),
    (dict(critic_hidden_dims=[]), "critic_hidden_dims is empty"),
    (dict(actor_hidden_dims=[256, 64]), "MN-major B operand needs N > 64"),
    (dict(critic_hidden_dims=[32]), "MN-major B operand needs N > 64"),
], ids=["activation", "empty-actor", "empty-critic", "actor-64", "critic-32"])
def test_constructor_rejects(kwargs, match):
    from isaac_b200.algo.actor_critic import ActorCritic
    with pytest.raises(ValueError, match=match):
        ActorCritic(615, 1050, 10, **dict(HECTOR, **kwargs), device="cpu")


def test_gemm_rejects_bad_activation_descriptors(lib):
    """Caught before any launch: an unknown activation, two grouped problems with different activations, and a non-ELU
    activation in a layout its epilogue is not built for."""
    from isaac_b200 import _lib
    fake = 1 << 20          # 16-byte aligned, never dereferenced

    def desc(**kw):
        d = _lib.GemmDesc(A=fake, B=fake, D=fake, M=256, N=128, K=64, lda=64, ldb=128, ldd=128, bias=fake, bias_stride=1,
                          H=fake, ldh=128, epilogue=_lib.HB_EPI_BIAS_ACT)
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    for precision in (_lib.HB_GEMM_TF32, _lib.HB_GEMM_3XTF32):
        for act in (-1, 6):
            assert lib.hb_gemm_tf32(C.byref(desc(activation=act, precision=precision)), None) == HB_ERR_BAD_ARG
            assert b"unknown activation" in lib.hb_last_error()
    rc = lib.hb_gemm_tf32_grouped(C.byref(desc(activation=_lib.HB_ACT_TANH)), C.byref(desc(activation=_lib.HB_ACT_RELU)), None)
    assert rc == HB_ERR_BAD_ARG and b"share epilogue" in lib.hb_last_error()
    for epi, a_mn, b_mn in ((_lib.HB_EPI_BIAS_ACT, 0, 1), (_lib.HB_EPI_BIAS_ACT, 1, 1), (_lib.HB_EPI_ACT_BWD, 0, 0),
                            (_lib.HB_EPI_ACT_BWD, 1, 1)):
        d = desc(epilogue=epi, a_mn_major=a_mn, b_mn_major=b_mn, activation=_lib.HB_ACT_SIGMOID)
        assert lib.hb_gemm_tf32(C.byref(d), None) == HB_ERR_UNSUPPORTED, (epi, a_mn, b_mn)


# ---------------------------------------------------------------------------------------------------- GPU: GEMM epilogues
def _padded(rows, cols, dev, g, extra=0):
    t = torch.zeros(rows, (cols + extra + 3) // 4 * 4, device=dev)
    t[:, :cols] = torch.randn(rows, cols, generator=g).to(dev)
    return t


def _tf32(x, mode):
    i = x.view(torch.int32)
    return ((i if mode == "trunc" else i + 0x1000) & ~0x1FFF).view(torch.float32)


def _epilogue_case(dev, name, kind, seed):
    """Operands of one ragged GEMM and its fp64 reference.  fwd: D = f(A B^T + b) (M, N, K = 300, 200, 615); dgrad:
    D = (dZ W) * f'(z) with H = f(z) stored in fp32 (M, N, K = 300, 200, 136).  Returns the descriptor kwargs, the output,
    the reference for each TF32 operand rounding and for fp32 operands, and |a|.|b|."""
    from isaac_b200 import _lib
    g = torch.Generator().manual_seed(seed)
    f = TORCH_ACTS[name]
    M, N = 300, 200
    if kind == "fwd":
        K = 615
        A, B = _padded(M, K, dev, g, extra=1), _padded(N, K, dev, g, extra=1)
        A[:, :K] *= 0.1
        bias = torch.randn(N, generator=g).to(dev)
        D = torch.zeros(M, N + 4, device=dev)
        kw = dict(A=A.data_ptr(), B=B.data_ptr(), D=D.data_ptr(), M=M, N=N, K=K, lda=A.stride(0), ldb=B.stride(0), ldd=D.stride(0),
                  epilogue=_lib.HB_EPI_BIAS_ACT, bias=bias.data_ptr(), bias_stride=1, activation=HB_CODES[name])
        a, b = A[:, :K].cpu(), B[:, :K].cpu()
        want = {m: f(fa(a).double() @ fa(b).double().T + bias.cpu().double()) for m, fa in
                (("trunc", lambda x: _tf32(x, "trunc")), ("round", lambda x: _tf32(x, "round")), ("fp32", lambda x: x))}
        keep = (A, B, bias)
    else:
        K = 136
        dZ, W = _padded(M, K, dev, g), _padded(K, N, dev, g, extra=1)
        z = torch.randn(M, N, generator=g, dtype=torch.float64)
        H = torch.zeros(M, N + 4, device=dev)
        H[:, :N] = f(z).float().to(dev)
        zl = z.clone().requires_grad_(True)
        fprime = torch.autograd.grad(f(zl).sum(), zl)[0]          # f'(z) by autograd
        D = torch.zeros(M, N, device=dev)
        kw = dict(A=dZ.data_ptr(), B=W.data_ptr(), D=D.data_ptr(), M=M, N=N, K=K, lda=dZ.stride(0), ldb=W.stride(0), ldd=D.stride(0),
                  b_mn_major=1, epilogue=_lib.HB_EPI_ACT_BWD, H=H.data_ptr(), ldh=H.stride(0), activation=HB_CODES[name])
        a, b = dZ[:, :K].cpu(), W[:K, :N].T.contiguous().cpu()
        want = {m: (fa(a).double() @ fa(b).double().T) * fprime for m, fa in
                (("trunc", lambda x: _tf32(x, "trunc")), ("round", lambda x: _tf32(x, "round")), ("fp32", lambda x: x))}
        keep = (dZ, W, H)
    scale = a.double().abs() @ b.double().abs().T
    return kw, D[:, :N], want, scale, keep


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "dgrad"])
@pytest.mark.parametrize("name", ACTS)
def test_activation_epilogues_tf32_and_3xtf32(lib, cuda_device, name, kind):
    """TF32: the result of the tensor core's TF32 operands (truncated or rounded) followed by f / f', to the tolerances of
    test_mlp_gemm.py.  3xTF32: the fp64 result of the fp32 operands, fp32-grade (2e-6 of |a|.|b|)."""
    from isaac_b200 import _lib
    from isaac_b200.algo.actor_critic import gemm
    dev = cuda_device
    st = torch.cuda.current_stream(dev).cuda_stream
    kw, got, want, scale, keep = _epilogue_case(dev, name, kind, seed=ACTS.index(name) + 10 * (kind == "fwd"))
    gemm(lib, st, None, **kw)
    torch.cuda.synchronize()
    if kind == "fwd":          # test_forward_bias_elu_epilogue's bound
        err = min((got.cpu().double() - want[m]).abs().max().item() for m in ("trunc", "round"))
        assert err < 1e-4, (name, err)
    else:                      # test_dgrad_b_mn_major_with_elu_backward's bound
        err = min(((got.cpu().double() - want[m]).abs() / scale.clamp_min(1e-30)).max().item() for m in ("trunc", "round"))
        assert err < 2e-5, (name, err)
    got.zero_()
    gemm(lib, st, [None, dev], **kw)
    torch.cuda.synchronize()
    err = ((got.cpu().double() - want["fp32"]).abs() / (scale + want["fp32"].abs()).clamp_min(1e-30)).max().item()
    print(f"{name} {kind}: 3xTF32 error relative to |a|.|b| {err:.2e}")
    assert err < 2e-6, (name, err)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ACTS)
def test_activation_grouped_launch_equals_two_launches(lib, cuda_device, name):
    """hb_gemm_tf32_grouped with a non-ELU activation: bit-equal to the two single launches, forward and data gradient."""
    from isaac_b200.algo.actor_critic import gemm, gemm2
    dev = cuda_device
    st = torch.cuda.current_stream(dev).cuda_stream
    for kind in ("fwd", "dgrad"):
        cases = [_epilogue_case(dev, name, kind, seed=s) for s in (1, 2)]
        for kw, _, _, _, _ in cases:
            gemm(lib, st, None, **kw)
        torch.cuda.synchronize()
        single = [c[1].clone() for c in cases]
        for c in cases:
            c[1].zero_()
        gemm2(lib, st, None, cases[0][0], None, cases[1][0])
        torch.cuda.synchronize()
        for c, s in zip(cases, single):
            assert torch.equal(c[1], s), (name, kind)
            assert float(s.abs().max()) > 0


# ---------------------------------------------------------------------------------------------------- GPU: fused head
@pytest.mark.gpu
@pytest.mark.parametrize("name", ACTS)
def test_fused_head_matches_autograd_per_activation(lib, cuda_device, name):
    """hb_ppo_head_fused with hb_ppo_loss_params.activation: from given last hidden activations h = f(z) everything is
    fp32 arithmetic, so the gradients agree with torch autograd in fp64 (through f at z) to fp32 accuracy."""
    from isaac_b200 import _lib
    dev = cuda_device
    NA, mb, HID = 10, 1000, 128
    f = TORCH_ACTS[name]
    g = torch.Generator().manual_seed(23)
    f64 = torch.float64
    r32 = lambda x: x.float().double()
    z3a, z3c = r32(torch.randn(mb, HID, generator=g, dtype=f64)), r32(torch.randn(mb, HID, generator=g, dtype=f64))
    w4a, b4a = r32(0.2 * torch.randn(NA, HID, generator=g, dtype=f64)), r32(0.1 * torch.randn(NA, generator=g, dtype=f64))
    w4c, b4c = r32(0.2 * torch.randn(1, HID, generator=g, dtype=f64)), r32(0.1 * torch.randn(1, generator=g, dtype=f64))
    std = r32(0.5 + torch.rand(NA, generator=g, dtype=f64))
    actions = r32(torch.randn(mb, NA, generator=g, dtype=f64))
    mu_old = r32(actions + 0.4 * torch.randn(mb, NA, generator=g, dtype=f64))
    sig_old = r32(0.5 + torch.rand(mb, NA, generator=g, dtype=f64))
    v_old, adv, ret = (r32(torch.randn(mb, generator=g, dtype=f64)) for _ in range(3))
    za, zc = z3a.clone().requires_grad_(True), z3c.clone().requires_grad_(True)
    # the kernel reads h rounded to fp32; the fp64 reference runs on those values, its f' at z
    ha, hc = f(za), f(zc)
    ha32, hc32 = r32(ha.detach()), r32(hc.detach())
    ha_in = ha + (ha32 - ha.detach())
    hc_in = hc + (hc32 - hc.detach())
    # (as in test_ppo_parity.py: ratios mostly far from the clip bounds, where fp32 and fp64 could choose different branches)
    lp_old = r32(-0.5 * ((actions - mu_old) ** 2).sum(-1) - 0.9 * NA + 0.3 * torch.randn(mb, generator=g, dtype=f64))
    W4a, B4a, W4c, B4c, S = (x.clone().requires_grad_(True) for x in (w4a, b4a, w4c, b4c, std))
    mu = ha_in @ W4a.T + B4a
    v = (hc_in @ W4c.T + B4c).squeeze(-1)
    sigma = mu * 0.0 + S
    lp = (-((actions - mu) ** 2) / (2 * sigma ** 2) - sigma.log() - 0.5 * np.log(2 * np.pi)).sum(-1)
    kl = (torch.log(sigma / sig_old + 1e-5) + (sig_old ** 2 + (mu_old - mu) ** 2) / (2 * sigma ** 2) - 0.5).sum(-1)
    ent = (0.5 + 0.5 * np.log(2 * np.pi) + sigma.log()).sum(-1)
    ratio = torch.exp(lp - lp_old)
    sur = torch.max(-adv * ratio, -adv * ratio.clamp(0.8, 1.2))
    vclip = v_old + (v - v_old).clamp(-0.2, 0.2)
    vl = torch.max((v - ret) ** 2, (vclip - ret) ** 2)
    (sur.mean() + 1.0 * vl.mean() - 0.001 * ent.mean()).backward()
    assert ((ratio < 0.8) | (ratio > 1.2)).float().mean() > 0.02

    ld = 132

    def packed(rows, w, b):
        P = torch.zeros(16, ld)
        P[:rows, :HID], P[:rows, HID] = w.float(), b.float()
        return P.to(dev)

    def act_buf(h):
        Hb = torch.zeros(mb, ld)
        Hb[:, :HID], Hb[:, HID] = h.float(), 1.0
        return Hb.to(dev)

    Ha, Hc, Pa, Pc = act_buf(ha32), act_buf(hc32), packed(NA, w4a, b4a), packed(1, w4c, b4c)
    rec = torch.zeros(mb, 3 * NA + 6)
    rec[:, 0:NA], rec[:, NA:2 * NA], rec[:, 2 * NA:3 * NA] = actions.float(), mu_old.float(), sig_old.float()
    rec[:, 3 * NA], rec[:, 3 * NA + 1], rec[:, 3 * NA + 2], rec[:, 3 * NA + 3] = v_old.float(), adv.float(), ret.float(), lp_old.float()
    rec = rec.to(dev)
    std_d = std.float().to(dev)
    dza, dzc = torch.empty(mb, HID, device=dev), torch.empty(mb, HID, device=dev)
    Ga, Gc = torch.zeros(16, ld, device=dev), torch.zeros(16, ld, device=dev)
    d_std, stats = torch.zeros(16, device=dev), torch.zeros(4, dtype=f64, device=dev)
    lpp = _lib.PpoLossParams(0.2, 1.0, 0.001, 1, NA, HB_CODES[name])
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.hb_ppo_head_fused(Ha.data_ptr(), ld, Hc.data_ptr(), ld, Pa.data_ptr(), Pc.data_ptr(), ld, std_d.data_ptr(),
                                     rec.data_ptr(), mb, mb, C.byref(lpp), dza.data_ptr(), dzc.data_ptr(), HID, Ga.data_ptr(),
                                     Gc.data_ptr(), d_std.data_ptr(), stats.data_ptr(), st), "hb_ppo_head_fused")
    torch.cuda.synchronize()
    tol = dict(rtol=2e-4, atol=2e-8)
    assert_close("dz_actor", dza.cpu().numpy(), za.grad.numpy(), **tol)
    assert_close("dz_critic", dzc.cpu().numpy(), zc.grad.numpy(), **tol)
    assert_close("dW_actor", Ga[:NA, :HID].cpu().numpy(), W4a.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert_close("db_actor", Ga[:NA, HID].cpu().numpy(), B4a.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert_close("dW_critic", Gc[:1, :HID].cpu().numpy(), W4c.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert_close("db_critic", Gc[:1, HID].cpu().numpy(), B4c.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert_close("d_std", d_std[:NA].cpu().numpy(), S.grad.numpy(), rtol=2e-4, atol=1e-7)
    np.testing.assert_allclose(stats.cpu().numpy(), [sur.sum().item(), vl.sum().item(), kl.sum().item(), ent.sum().item()],
                               rtol=2e-5)
    lpp.activation = 6
    assert lib.hb_ppo_head_fused(Ha.data_ptr(), ld, Hc.data_ptr(), ld, Pa.data_ptr(), Pc.data_ptr(), ld, std_d.data_ptr(),
                                 rec.data_ptr(), mb, mb, C.byref(lpp), dza.data_ptr(), dzc.data_ptr(), HID, Ga.data_ptr(),
                                 Gc.data_ptr(), d_std.data_ptr(), stats.data_ptr(), st) == HB_ERR_BAD_ARG


# ---------------------------------------------------------------------------------------------------- GPU: PPO end to end
def make_pair(dev, net, activation, precision, n, t, alg_cfg, seed=3):
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    params = init_actor_critic_params(615, 1050, 10, tuple(net["actor_hidden_dims"]), tuple(net["critic_hidden_dims"]), seed=seed)
    ac = ActorCritic(615, 1050, 10, **net, activation=activation, device=dev, precision=precision)
    ac.load_state_dict(params)
    alg = PPO(ac, device=dev, **alg_cfg)
    alg.init_storage(n, t, [615], [1050], [10])
    ora = PolicyOraclePPO(params, n, t, **alg_cfg, activation=activation)
    return alg, ora, params


def rollout(alg, ora, dev, g, n, t):
    """t steps of act (injected eps) / process_env_step and compute_returns on both sides, from the same random inputs."""
    for _ in range(t):
        o, co, eps = torch.randn(n, 615, generator=g), torch.randn(n, 1050, generator=g), torch.randn(n, 10, generator=g)
        rew, dones, tos = torch.rand(n, generator=g), torch.rand(n, generator=g) < 0.1, torch.rand(n, generator=g) < 0.05
        alg.injected_eps = eps.to(dev)
        alg.act(o.to(dev), co.to(dev))
        ora.act(o, co, eps)
        alg.process_env_step(rew.to(dev), dones.to(dev), {"time_outs": tos.to(dev)})
        ora.process_env_step(rew, dones, {"time_outs": tos})
    last = torch.randn(n, 1050, generator=g)
    alg.compute_returns(last.to(dev))
    ora.compute_returns(last)


def same_rollout_data(alg, ora):
    """Hand the update the oracle's rollout, so that only the update path is compared."""
    for k in ("actions", "values", "returns", "advantages", "actions_log_prob", "mu", "sigma", "rewards"):
        getattr(alg.storage, k).copy_(ora.st[k])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ACTS)
def test_minibatch_gradients_match_autograd_per_activation(lib, cuda_device, name):
    """One minibatch of the unequal-depth pair in 3xTF32 - grouped and single forward launches, the fused head, grouped
    and single backward launches - against torch autograd on the oracle's loss: every parameter's gradient to 1e-5."""
    from oracle.ppo_oracle import gaussian_entropy, gaussian_log_prob
    dev = cuda_device
    n, t = 64, 8
    cfg = dict(mg.PPO_ALG, schedule="fixed", num_learning_epochs=1, num_mini_batches=1)
    alg, ora, _ = make_pair(dev, UNEQUAL, name, "3xtf32", n, t, cfg)
    g = torch.Generator().manual_seed(0)
    rollout(alg, ora, dev, g, n, t)
    same_rollout_data(alg, ora)
    perm = torch.randperm(n * t, generator=g)
    alg.prepare_minibatches(perm)
    alg.minibatch_gradients(0)
    torch.cuda.synchronize()
    flat = {k: v.flatten(0, 1)[perm] for k, v in ora.st.items()}
    P = ora.params
    mu = mlp(P, "actor", flat["observations"], name)
    sigma = mu * 0.0 + P["std"]
    ratio = torch.exp(gaussian_log_prob(flat["actions"], mu, sigma) - flat["actions_log_prob"].squeeze())
    adv = flat["advantages"].squeeze()
    surrogate = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 0.8, 1.2)).mean()
    v = mlp(P, "critic", flat["privileged_observations"], name)
    v_old, ret = flat["values"], flat["returns"]
    v_clip = v_old + (v - v_old).clamp(-0.2, 0.2)
    value_loss = torch.max((v - ret).pow(2), (v_clip - ret).pow(2)).mean()
    (surrogate + 1.0 * value_loss - 0.001 * gaussian_entropy(sigma).mean()).backward()
    grads = dict(alg.actor_critic.named_gradients())
    errs = {k: rel_l2(grads[k].cpu(), P[k].grad) for k in ora.order}
    assert max(errs.values()) < 1e-5, errs


# End to end over 20 Adam steps.  PPO's objective is discontinuous (clipping, max), so two fp32 implementations drift
# apart wherever a sample sits at a branch point; with ReLU / LeakyReLU kinks or SELU's larger pre-activations that drift
# exceeds test_ppo_parity.py's tolerances on these trajectories, although each minibatch's gradients agree to 1e-5 (test
# above).  The trajectories compared here use the smooth activations.
E2E = [("hector-tanh", HECTOR, "tanh", "3xtf32"), ("unequal-tanh", UNEQUAL, "tanh", "3xtf32"),
       ("generic-sigmoid", GENERIC, "sigmoid", "3xtf32"), ("unequal-sigmoid-tf32", UNEQUAL, "sigmoid", "tf32")]


@pytest.mark.gpu
@pytest.mark.parametrize("net,activation,precision", [e[1:] for e in E2E], ids=[e[0] for e in E2E])
def test_ppo_matches_oracle(lib, cuda_device, net, activation, precision):
    """Forward, act with injected eps and one fixed-schedule update (the golden case's sizes: 64 envs x 24 steps, 5 epochs
    x 4 minibatches) against OraclePPO with the same activation and depths.  3xTF32 at test_ppo_parity.py's fp32-grade
    tolerances, TF32 at its TF32 tolerances."""
    dev = cuda_device
    n, t = mg.PPO_CASE["n"], mg.PPO_CASE["t"]          # the golden case's sizes and schedule: 20 Adam steps
    cfg = dict(mg.PPO_ALG, schedule="fixed")
    alg, ora, params = make_pair(dev, net, activation, precision, n, t, cfg)
    ac = alg.actor_critic
    assert ac.fused_head == (net is not GENERIC)
    fp32 = precision == "3xtf32"
    # forward
    g = torch.Generator().manual_seed(0)
    obs, cobs = torch.randn(200, 615, generator=g), torch.randn(200, 1050, generator=g)
    mu, v = ac.act_inference(obs.to(dev)).cpu(), ac.evaluate(cobs.to(dev)).cpu()
    with torch.no_grad():
        w_mu, w_v = mlp(params, "actor", obs, activation), mlp(params, "critic", cobs, activation)
    tol = 1e-5 if fp32 else 4e-3
    assert rel_l2(mu, w_mu) < tol and rel_l2(v, w_v) < tol, (rel_l2(mu, w_mu), rel_l2(v, w_v))
    if fp32:
        assert_close("mu", mu.numpy(), w_mu.numpy(), rtol=1e-5, atol=1e-5 * float(w_mu.abs().max()))
        assert_close("value", v.numpy(), w_v.numpy(), rtol=1e-5, atol=1e-5 * float(w_v.abs().max()))
    # act (injected eps), process_env_step, compute_returns
    rollout(alg, ora, dev, g, n, t)
    s = alg.storage
    for k in ("actions", "values", "mu", "actions_log_prob"):
        assert rel_l2(getattr(s, k).cpu(), ora.st[k]) < tol, (k, rel_l2(getattr(s, k).cpu(), ora.st[k]))
    # one update from identical rollout data
    same_rollout_data(alg, ora)
    perm = torch.randperm(n * t, generator=g)
    alg.injected_perm = perm
    v_loss, s_loss = alg.update()
    w_vl, w_sl = ora.update(perm)
    loss_tol = 2e-5 if fp32 else 5e-3
    assert abs(v_loss - w_vl) < loss_tol * max(1.0, abs(w_vl)) and abs(s_loss - w_sl) < loss_tol, (v_loss, w_vl, s_loss, w_sl)
    sd = ac.state_dict()
    assert list(sd) == ora.order
    lr, steps_taken = cfg["learning_rate"], cfg["num_learning_epochs"] * cfg["num_mini_batches"]
    for k in ora.order:
        got, want, init = sd[k].cpu().double(), ora.params[k].detach().double(), params[k].double()
        if fp32:       # test_update_matches_reference_golden's fp32-grade bounds
            err = (got - want).abs()
            off = err > (lr * 1e-2 + 1e-5 * want.abs())
            assert int(off.sum()) <= max(1, got.numel() // 10000), f"{k}: {int(off.sum())} of {got.numel()} beyond rtol 1e-5 / atol lr*1e-2"
            assert float(err.max()) <= 0.1 * lr, f"{k}: max error {float(err.max()):.3e}"
            assert float((got - want).norm() / (want - init).norm().clamp_min(1e-30)) < 1e-3, k
        else:          # its TF32 bounds: Adam's per-element bound and the update direction
            assert (got - want).abs().max().item() <= 2.0 * lr * steps_taken * 1.01 + 1e-9, k
            assert float((got - want).norm() / (want - init).norm().clamp_min(1e-30)) < 0.25, k


# ---------------------------------------------------------------------------------------------------- GPU: interface
@pytest.mark.gpu
@pytest.mark.parametrize("net,activation", [(UNEQUAL, "tanh"), (GENERIC, "crelu"), (HECTOR, None)],
                         ids=["unequal-tanh", "generic-crelu", "hector-default"])
def test_state_dict_and_initialisation_match_the_reference_module(lib, cuda_device, net, activation):
    from isaac_b200.algo.actor_critic import ActorCritic
    torch.manual_seed(12)
    ref = reference_modules(615, 1050, 10, net["actor_hidden_dims"], net["critic_hidden_dims"], activation or "elu")
    torch.manual_seed(12)
    ac = ActorCritic(615, 1050, 10, **net, activation=activation, device=cuda_device)
    sd = ac.state_dict()
    assert list(sd) == [k for k, _ in ref.named_parameters()]
    ref_sd = ref.state_dict()
    for k in sd:
        assert torch.equal(sd[k].cpu(), ref_sd[k]), k        # same seed, same initial parameters
    ref.load_state_dict({k: v.cpu() + 1.0 for k, v in sd.items()}, strict=True)
    ac.load_state_dict(ref.state_dict())
    for k, v in ac.state_dict().items():
        assert torch.equal(v.cpu(), ref.state_dict()[k]), k


@pytest.mark.gpu
def test_optimizer_state_round_trips_through_the_runner(lib, cuda_device, tmp_path):
    from isaac_b200.algo import OnPolicyRunner
    from test_runner import TRAIN_CFG, make_env
    cfg = dict(TRAIN_CFG, policy=dict(TRAIN_CFG["policy"], **UNEQUAL, activation="selu"))
    runner = OnPolicyRunner(make_env(cuda_device), cfg, log_dir=None, device=str(cuda_device))
    runner.learn(num_learning_iterations=1)
    ac = runner.alg.actor_critic
    n_layers = len(ac.layers)
    assert n_layers == 3 + 6
    osd = runner.alg.optimizer.state_dict()
    assert len(osd["state"]) == 1 + 2 * n_layers and osd["param_groups"][0]["params"] == list(range(1 + 2 * n_layers))
    path = os.path.join(tmp_path, "model.pt")
    runner.save(path)
    runner2 = OnPolicyRunner(make_env(cuda_device), cfg, log_dir=None, device=str(cuda_device))
    runner2.load(path)
    assert torch.equal(runner2.alg.actor_critic.flat, ac.flat) and runner2.alg._step == runner.alg._step
    assert torch.equal(runner2.alg._exp_avg, runner.alg._exp_avg) and torch.equal(runner2.alg._exp_avg_sq, runner.alg._exp_avg_sq)
    osd2 = runner2.alg.optimizer.state_dict()
    for i, e in osd["state"].items():
        assert torch.equal(osd2["state"][i]["exp_avg"], e["exp_avg"]) and torch.equal(osd2["state"][i]["exp_avg_sq"], e["exp_avg_sq"])


# ---------------------------------------------------------------------------------------------------- GPU: launches
@pytest.mark.gpu
def test_unequal_depth_launches(lib, cuda_device, monkeypatch):
    """UNEQUAL (actor 256-128, critic 512-256-256-256-128, fused head), in the style of test_ppo_launches.py.  act: the
    draw, grouped forward launches for hidden layers 0-1, the critic's hidden layers 2-4 alone, hb_ppo_act_fused.
    Minibatch step: the same forward, hb_ppo_head_fused, then top down the critic's layers 4, 3 and 2 alone (data
    gradient, weight gradient), grouped data and weight gradients of layer 1, the grouped weight gradient of layer 0,
    hb_optimizer_step.  Every descriptor carries the activation."""
    import test_ppo_launches as tpl
    from isaac_b200._lib import HB_GEMM_TF32
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    monkeypatch.setattr(tpl, "DESC_FIELDS", tpl.DESC_FIELDS + ("activation",))
    dev = cuda_device
    ac = ActorCritic(615, 1050, 10, **UNEQUAL, activation="tanh", device=dev)
    assert ac.fused_head
    alg = PPO(ac, device=dev, num_learning_epochs=1, num_mini_batches=2, schedule="fixed")
    alg.init_storage(64, 4, [615], [1050], [10])
    alg.graph_rollout = False
    act = ac.hb_activation

    def one(desc, net, i, m):
        return ("hb_gemm_tf32", desc(ac, net, i, m, HB_GEMM_TF32) + (act,))

    def both(desc, i, m):
        return ("hb_gemm_tf32_grouped", desc(ac, "critic", i, m, HB_GEMM_TF32) + (act,), desc(ac, "actor", i, m, HB_GEMM_TF32) + (act,))

    def forward(m):
        return [both(tpl.fwd, 0, m), both(tpl.fwd, 1, m), *[one(tpl.fwd, "critic", i, m) for i in (2, 3, 4)]]

    def backward(m):
        return [*[one(d, "critic", i, m) for i in (4, 3, 2) for d in (tpl.dgrad, tpl.wgrad)],
                both(tpl.dgrad, 1, m), both(tpl.wgrad, 1, m), both(tpl.wgrad, 0, m)]

    g = torch.Generator().manual_seed(2)
    obs, cobs = tpl.observations(alg, g)
    rec = tpl.record(alg, lambda: alg.act(obs, cobs))
    assert rec.calls == [("hb_ppo_draw_normal",), *forward(64), ("hb_ppo_act_fused",)]
    s = alg.storage
    alg.process_env_step(torch.rand(64, generator=g).to(dev), torch.zeros(64, dtype=torch.bool, device=dev), {})
    for _ in range(s.num_transitions_per_env - 1):
        obs, cobs = tpl.observations(alg, g)
        alg.act(obs, cobs)
        alg.process_env_step(torch.rand(64, generator=g).to(dev), torch.zeros(64, dtype=torch.bool, device=dev), {})
    alg.compute_returns(cobs)
    alg.prepare_minibatches()
    rec = tpl.record(alg, lambda: (alg.minibatch_gradients(0), alg.optimizer_step(0)))
    m = alg._mb
    assert rec.calls == [*forward(m), ("hb_ppo_head_fused",), *backward(m), ("hb_optimizer_step",)]
