"""Any number of actions from 1 to 64, as the reference's ActorCritic / PPO / RolloutStorage take whatever `num_actions` the
env reports.  10, 12 and 18 run kernels compiled for their count; every other count runs the runtime-count instantiation
of hb_ppo_pack_samples / hb_ppo_loss_head / hb_ppo_act_head, and up to 15 actions the fused output-layer heads
(hb_ppo_head_fused, hb_ppo_act_fused) take the count at run time too.

CPU: the constructor's range, and the library's refusal of counts outside each entry point's range before any launch.
GPU: each kernel against torch fp64 (forward values, autograd gradients), PPO end to end against the oracle for a fused
and a generic count, the launch sequence of both paths, and OnPolicyRunner over a small torch VecEnv with checkpoints."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from _util import assert_close
from _policy_oracle import ACTIVATIONS as TORCH_ACTS, PolicyOraclePPO, mlp
from oracle import make_golden as mg
from oracle.ppo_oracle import init_actor_critic_params

HB_ERR_BAD_ARG, HB_ERR_UNSUPPORTED = -1, -3
ACTS = ["elu", "selu", "relu", "lrelu", "tanh", "sigmoid"]
HECTOR = dict(actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128])
# small observation widths that the weight gradient of the first layer still takes: it reads [obs | 1] as an MN-major
# B operand, which needs more than 64 columns
OBS, PRIV = 72, 104
GENERIC_COUNTS = [1, 7, 13, 19, 23, 29, 64]
FUSED_COUNTS = [1, 5, 7, 13, 15]
HALF_LOG_2PI = 0.5 * np.log(2 * np.pi)


def pad16(n):
    return (n + 15) // 16 * 16


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("na", [1, 7, 15, 16, 23, 64])
def test_constructor_accepts_counts(lib, na):
    from isaac_b200.algo.actor_critic import ActorCritic
    ac = ActorCritic(OBS, PRIV, na, **HECTOR, device="cpu")
    assert ac.std.shape == (na,) and ac.output_layers[0].rows == pad16(na)
    assert ac.fused_head == (na <= 15)


@pytest.mark.parametrize("na", [0, 65])
def test_constructor_rejects_counts(na):
    from isaac_b200.algo.actor_critic import ActorCritic
    with pytest.raises(ValueError, match="1 to 64 actions"):
        ActorCritic(OBS, PRIV, na, **HECTOR, device="cpu")


def test_entry_points_reject_counts_outside_their_range(lib):
    """Below 1: HB_ERR_BAD_ARG, above the entry point's limit: HB_ERR_UNSUPPORTED, the range in hb_last_error(), and no
    launch (the pointers are never dereferenced)."""
    from isaac_b200 import _lib
    fake = 1 << 20
    lp = _lib.PpoLossParams(0.2, 1.0, 0.001, 1, 0, 0)

    def pack(na):
        return lib.hb_ppo_pack_samples(fake, 8, fake, fake, fake, fake, fake, fake, fake, na, fake, None)

    def loss(na):
        lp.num_actions = na
        return lib.hb_ppo_loss_head(fake, 128, fake, 16, fake, fake, 8, 8, C.byref(lp), fake, fake, fake, fake, None)

    def act(na):
        return lib.hb_ppo_act_head(fake, 128, fake, fake, 8, na, fake, fake, fake, fake, None)

    def head_fused(na):
        lp.num_actions = na
        return lib.hb_ppo_head_fused(fake, 132, fake, 132, fake, fake, 132, fake, fake, 8, 8, C.byref(lp), fake, fake, 128,
                                     fake, fake, fake, fake, None)

    def act_fused(na):
        return lib.hb_ppo_act_fused(fake, 132, fake, 132, fake, fake, 132, fake, fake, 8, na, fake, fake, fake, fake, fake, None)

    launches = lib.hb_launch_count()
    for fn, limit in ((pack, 64), (loss, 64), (act, 64), (head_fused, 15), (act_fused, 15)):
        for na in (-1, 0, limit + 1, 100):
            rc = fn(na)
            assert rc == (HB_ERR_BAD_ARG if na < 1 else HB_ERR_UNSUPPORTED), (fn.__name__, na, rc)
            msg = lib.hb_last_error().decode()
            assert f"num_actions = {na}" in msg and f"(1 to {limit}" in msg, msg
    for na in (16, 18, 23):
        assert head_fused(na) == HB_ERR_UNSUPPORTED and "(1 to 15;" in lib.hb_last_error().decode()
        assert act_fused(na) == HB_ERR_UNSUPPORTED and "(1 to 15;" in lib.hb_last_error().decode()
    assert lib.hb_launch_count() == launches


# ---------------------------------------------------------------------------------------------------- GPU: generic kernels
def _sample_set(na, n, g):
    """fp32-representable (as fp64) actions, old mu / sigma, values, advantages, returns and std; old log-probs a
    random distance from the new ones, so that some ratios are clipped but few sit near a clip bound."""
    f64 = torch.float64
    r32 = lambda x: x.float().double()
    s = dict(mu=r32(torch.randn(n, na, generator=g, dtype=f64)), std=r32(0.5 + torch.rand(na, generator=g, dtype=f64)))
    s["actions"] = r32(s["mu"] + 0.7 * torch.randn(n, na, generator=g, dtype=f64))
    s["mu_old"] = r32(s["actions"] + 0.4 * torch.randn(n, na, generator=g, dtype=f64))
    s["sig_old"] = r32(0.5 + torch.rand(n, na, generator=g, dtype=f64))
    s["v"], s["v_old"], s["adv"], s["ret"] = (r32(torch.randn(n, generator=g, dtype=f64)) for _ in range(4))
    lp_new = (-((s["actions"] - s["mu"]) ** 2) / (2 * s["std"] ** 2) - s["std"].log() - HALF_LOG_2PI).sum(-1)
    s["lp_old"] = r32(lp_new + 0.3 * torch.randn(n, generator=g, dtype=f64))
    return s


def _loss_reference(s, mu, v, std):
    """ppo.py:130-168 in fp64 on the given leaves; returns (loss, per-sample surrogate, value loss, kl, entropy, ratio)."""
    sigma = mu * 0.0 + std
    lp = (-((s["actions"] - mu) ** 2) / (2 * sigma ** 2) - sigma.log() - HALF_LOG_2PI).sum(-1)
    kl = (torch.log(sigma / s["sig_old"] + 1e-5) + (s["sig_old"] ** 2 + (s["mu_old"] - mu) ** 2) / (2 * sigma ** 2) - 0.5).sum(-1)
    ent = (0.5 + HALF_LOG_2PI + sigma.log()).sum(-1)
    ratio = torch.exp(lp - s["lp_old"])
    sur = torch.max(-s["adv"] * ratio, -s["adv"] * ratio.clamp(0.8, 1.2))
    vclip = s["v_old"] + (v - s["v_old"]).clamp(-0.2, 0.2)
    vl = torch.max((v - s["ret"]) ** 2, (vclip - s["ret"]) ** 2)
    return sur.mean() + 1.0 * vl.mean() - 0.001 * ent.mean(), sur, vl, kl, ent, ratio


@pytest.mark.gpu
@pytest.mark.parametrize("na", GENERIC_COUNTS)
def test_generic_kernels_match_fp64(lib, cuda_device, na):
    """hb_ppo_pack_samples (an exact gather), hb_ppo_act_head and hb_ppo_loss_head at rows padded to pad16(na), as the
    output-layer GEMMs leave them, against torch fp64 forward values and autograd gradients (test_ppo_parity.py's
    tolerances).  1000 samples: the last block is partly empty."""
    from isaac_b200 import _lib
    dev = cuda_device
    st = torch.cuda.current_stream(dev).cuda_stream
    g = torch.Generator().manual_seed(na)
    T, N = 4, 250
    B = T * N
    s = _sample_set(na, B, g)
    # ---- pack: storage-shaped [T, N, .] inputs, gathered by a permutation
    store = {k: s[k].float().view(T, N, -1).to(dev) for k in ("actions", "mu_old", "sig_old", "v_old", "adv", "ret", "lp_old")}
    perm = torch.randperm(B, generator=g)
    rec = torch.full((B, 3 * na + 6), float("nan"), device=dev)
    pd = perm.to(dev)
    _lib.check(lib.hb_ppo_pack_samples(pd.data_ptr(), B, *(store[k].data_ptr() for k in ("actions", "mu_old", "sig_old", "v_old",
                                                                                        "adv", "ret", "lp_old")),
                                       na, rec.data_ptr(), st), "hb_ppo_pack_samples")
    torch.cuda.synchronize()
    flat = {k: v.reshape(B, -1).cpu()[perm] for k, v in store.items()}
    want_rec = torch.cat([flat["actions"], flat["mu_old"], flat["sig_old"], flat["v_old"], flat["adv"], flat["ret"],
                          flat["lp_old"], torch.zeros(B, 2)], 1)
    assert torch.equal(rec.cpu(), want_rec)
    s = {k: (v[perm] if v.shape[0] == B else v) for k, v in s.items()}           # minibatch order, as the records

    # ---- act head: a = mu + sigma * eps, its log-prob, copies of mu and sigma
    ld = pad16(na)
    mu_pad = torch.randn(B, ld, generator=g)
    mu_pad[:, :na] = s["mu"].float()
    eps = torch.randn(B, na, generator=g)
    mu_d, std_d, eps_d = mu_pad.to(dev), s["std"].float().to(dev), eps.to(dev)
    acts, logp, mu_o, sig_o = (torch.empty(B, na, device=dev), torch.empty(B, device=dev), torch.empty(B, na, device=dev),
                               torch.empty(B, na, device=dev))
    _lib.check(lib.hb_ppo_act_head(mu_d.data_ptr(), ld, std_d.data_ptr(), eps_d.data_ptr(), B, na, acts.data_ptr(),
                                   logp.data_ptr(), mu_o.data_ptr(), sig_o.data_ptr(), st), "hb_ppo_act_head")
    torch.cuda.synchronize()
    a_w = s["mu"] + s["std"] * eps.double()
    lp_w = (-((a_w - s["mu"]) ** 2) / (2 * s["std"] ** 2) - s["std"].log() - HALF_LOG_2PI).sum(-1)
    assert_close("actions", acts.cpu().numpy(), a_w.numpy(), rtol=1e-5, atol=1e-6)
    assert_close("log_prob", logp.cpu().numpy(), lp_w.numpy(), rtol=1e-5, atol=1e-5)
    assert torch.equal(mu_o.cpu(), s["mu"].float()) and torch.equal(sig_o.cpu(), s["std"].float().expand(B, na))

    # ---- loss head and its gradients w.r.t. mu, value and std
    mb = B
    v_pad = torch.randn(mb, 16, generator=g)
    v_pad[:, 0] = s["v"].float()
    v_d = v_pad.to(dev)
    d_mu, d_v = torch.full((mb, ld), float("nan"), device=dev), torch.full((mb, 16), float("nan"), device=dev)
    d_std, stats = torch.zeros(na, device=dev), torch.zeros(4, dtype=torch.float64, device=dev)
    lpp = _lib.PpoLossParams(0.2, 1.0, 0.001, 1, na, 0)
    _lib.check(lib.hb_ppo_loss_head(mu_d.data_ptr(), ld, v_d.data_ptr(), 16, std_d.data_ptr(), rec.data_ptr(), mb, mb,
                                    C.byref(lpp), d_mu.data_ptr(), d_v.data_ptr(), d_std.data_ptr(), stats.data_ptr(), st),
               "hb_ppo_loss_head")
    torch.cuda.synchronize()
    mu_l, v_l, std_l = s["mu"].clone().requires_grad_(True), s["v"].clone().requires_grad_(True), s["std"].clone().requires_grad_(True)
    loss, sur, vl, kl, ent, ratio = _loss_reference(s, mu_l, v_l, std_l)
    loss.backward()
    assert ((ratio < 0.8) | (ratio > 1.2)).double().mean() > 0.02
    # the ratio's relative error is the fp32 rounding error of the log-prob sum, which grows with the number of terms:
    # test_ppo_parity.py's bounds up to 16 actions, in proportion beyond
    grow = max(1.0, na / 16)
    assert_close("d_mu", d_mu[:, :na].cpu().numpy(), mu_l.grad.numpy(), rtol=2e-5 * grow, atol=1e-9)
    assert_close("d_value", d_v[:, :1].cpu().numpy(), v_l.grad[:, None].numpy(), rtol=2e-5, atol=1e-9)
    assert_close("d_std", d_std.cpu().numpy(), std_l.grad.numpy(), rtol=1e-4 * grow, atol=1e-7)
    assert torch.all(d_mu[:, na:] == 0) and torch.all(d_v[:, 1:] == 0)
    want = [sur.sum().item(), vl.sum().item(), kl.sum().item(), ent.sum().item()]
    np.testing.assert_allclose(stats.cpu().numpy(), want, rtol=2e-5)


# ---------------------------------------------------------------------------------------------------- GPU: fused heads
HID, LD = 128, 132


def _fused_case(na, dev, g):
    """Last hidden pre-activations, output layers packed [W | b] into 16 rows, and a sample set."""
    f64 = torch.float64
    r32 = lambda x: x.float().double()
    c = dict(z3a=r32(torch.randn(1000, HID, generator=g, dtype=f64)), z3c=r32(torch.randn(1000, HID, generator=g, dtype=f64)),
             w4a=r32(0.2 * torch.randn(na, HID, generator=g, dtype=f64)), b4a=r32(0.1 * torch.randn(na, generator=g, dtype=f64)),
             w4c=r32(0.2 * torch.randn(1, HID, generator=g, dtype=f64)), b4c=r32(0.1 * torch.randn(1, generator=g, dtype=f64)))

    def packed(w, b):
        P = torch.zeros(16, LD)
        P[:w.shape[0], :HID], P[:w.shape[0], HID] = w.float(), b.float()
        return P.to(dev)

    c["Pa"], c["Pc"] = packed(c["w4a"], c["b4a"]), packed(c["w4c"], c["b4c"])
    return c


def _act_buf(h, dev):
    Hb = torch.zeros(h.shape[0], LD)
    Hb[:, :HID], Hb[:, HID] = h.float(), 1.0
    return Hb.to(dev)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ACTS)
@pytest.mark.parametrize("na", FUSED_COUNTS)
def test_head_fused_matches_autograd(lib, cuda_device, na, name):
    """hb_ppo_head_fused at a runtime count: from the last hidden activations h = f(z), the output layers, loss and all
    their gradients against fp64 autograd, as test_actor_critic_config.py checks 10 actions."""
    from isaac_b200 import _lib
    from isaac_b200.algo.actor_critic import ACTIVATIONS as HB_CODES
    dev = cuda_device
    f = TORCH_ACTS[name]
    g = torch.Generator().manual_seed(100 + na)
    c = _fused_case(na, dev, g)
    mb = c["z3a"].shape[0]
    za, zc = c["z3a"].clone().requires_grad_(True), c["z3c"].clone().requires_grad_(True)
    ha, hc = f(za), f(zc)
    ha32, hc32 = ha.detach().float().double(), hc.detach().float().double()
    ha_in, hc_in = ha + (ha32 - ha.detach()), hc + (hc32 - hc.detach())         # the kernel reads h rounded to fp32
    W4a, B4a, W4c, B4c = (c[k].clone().requires_grad_(True) for k in ("w4a", "b4a", "w4c", "b4c"))
    mu = ha_in @ W4a.T + B4a
    mu.retain_grad()
    v = (hc_in @ W4c.T + B4c).squeeze(-1)
    s = _sample_set(na, mb, g)
    # actions drawn from the policy, as in a rollout, and old log-probs around the new ones: the log-prob sums stay at
    # the size a rollout gives them, ~1.4 per action (their fp32 rounding is the ratio's relative error)
    with torch.no_grad():
        s["actions"] = (mu + s["std"] * torch.randn(mb, na, generator=g, dtype=torch.float64)).float().double()
        s["mu_old"] = (s["actions"] + 0.4 * torch.randn(mb, na, generator=g, dtype=torch.float64)).float().double()
        lp_new = (-((s["actions"] - mu) ** 2) / (2 * s["std"] ** 2) - s["std"].log() - HALF_LOG_2PI).sum(-1)
        s["lp_old"] = (lp_new + 0.3 * torch.randn(mb, generator=g, dtype=torch.float64)).float().double()
    S = s["std"].clone().requires_grad_(True)
    loss, sur, vl, kl, ent, ratio = _loss_reference(s, mu, v, S)
    loss.backward()
    assert ((ratio < 0.8) | (ratio > 1.2)).double().mean() > 0.02
    Ha, Hc = _act_buf(ha32, dev), _act_buf(hc32, dev)
    rec = torch.cat([s["actions"], s["mu_old"], s["sig_old"], s["v_old"][:, None], s["adv"][:, None], s["ret"][:, None],
                     s["lp_old"][:, None], torch.zeros(mb, 2, dtype=torch.float64)], 1).float().to(dev)
    std_d = s["std"].float().to(dev)
    dza, dzc = torch.empty(mb, HID, device=dev), torch.empty(mb, HID, device=dev)
    Ga, Gc = torch.zeros(16, LD, device=dev), torch.zeros(16, LD, device=dev)
    d_std, stats = torch.zeros(16, device=dev), torch.zeros(4, dtype=torch.float64, device=dev)
    lpp = _lib.PpoLossParams(0.2, 1.0, 0.001, 1, na, HB_CODES[name])
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.hb_ppo_head_fused(Ha.data_ptr(), LD, Hc.data_ptr(), LD, c["Pa"].data_ptr(), c["Pc"].data_ptr(), LD,
                                     std_d.data_ptr(), rec.data_ptr(), mb, mb, C.byref(lpp), dza.data_ptr(), dzc.data_ptr(), HID,
                                     Ga.data_ptr(), Gc.data_ptr(), d_std.data_ptr(), stats.data_ptr(), st), "hb_ppo_head_fused")
    torch.cuda.synchronize()
    tol = dict(rtol=2e-4, atol=2e-8)
    assert_close("dz_actor", dza.cpu().numpy(), za.grad.numpy(), **tol)
    assert_close("dz_critic", dzc.cpu().numpy(), zc.grad.numpy(), **tol)
    # each sample's ratio carries the fp32 rounding of its log-prob sum, and the actor's weight gradient sums the samples
    # with cancellation: besides test_actor_critic_config.py's bounds, an error of 5e-6 of the sum of the absolute
    # contributions (a plain fp32 evaluation of these formulas reaches 8.2e-7 on these cases)
    scale_w = (mu.grad.abs().T @ ha32.abs()).numpy()
    scale_b = mu.grad.abs().sum(0).numpy()
    assert_close("dW_actor", Ga[:na, :HID].cpu().numpy(), W4a.grad.numpy(), rtol=2e-4, atol=1e-7 + 5e-6 * scale_w)
    assert_close("db_actor", Ga[:na, HID].cpu().numpy(), B4a.grad.numpy(), rtol=2e-4, atol=1e-7 + 5e-6 * scale_b)
    assert_close("dW_critic", Gc[:1, :HID].cpu().numpy(), W4c.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert_close("db_critic", Gc[:1, HID].cpu().numpy(), B4c.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert_close("d_std", d_std[:na].cpu().numpy(), S.grad.numpy(), rtol=2e-4, atol=1e-7)
    assert torch.all(Ga[na:] == 0) and torch.all(Gc[1:] == 0) and torch.all(d_std[na:] == 0)      # nothing past the count
    np.testing.assert_allclose(stats.cpu().numpy(), [sur.sum().item(), vl.sum().item(), kl.sum().item(), ent.sum().item()],
                               rtol=2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("na", FUSED_COUNTS)
def test_act_fused_matches_fp64(lib, cuda_device, na):
    """hb_ppo_act_fused at a runtime count: both output layers, the sample, its log-prob, mu, sigma and the value."""
    from isaac_b200 import _lib
    dev = cuda_device
    g = torch.Generator().manual_seed(200 + na)
    c = _fused_case(na, dev, g)
    n = c["z3a"].shape[0]
    ha, hc = torch.nn.functional.elu(c["z3a"]).float().double(), torch.nn.functional.elu(c["z3c"]).float().double()
    std = (0.5 + torch.rand(na, generator=g)).double()
    eps = torch.randn(n, na, generator=g)
    Ha, Hc, std_d, eps_d = _act_buf(ha, dev), _act_buf(hc, dev), std.float().to(dev), eps.to(dev)
    acts, mu_o, sig_o = (torch.empty(n, na, device=dev) for _ in range(3))
    logp, vals = torch.empty(n, device=dev), torch.empty(n, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.hb_ppo_act_fused(Ha.data_ptr(), LD, Hc.data_ptr(), LD, c["Pa"].data_ptr(), c["Pc"].data_ptr(), LD,
                                    std_d.data_ptr(), eps_d.data_ptr(), n, na, acts.data_ptr(), logp.data_ptr(), mu_o.data_ptr(),
                                    sig_o.data_ptr(), vals.data_ptr(), st), "hb_ppo_act_fused")
    torch.cuda.synchronize()
    mu_w = ha @ c["w4a"].T + c["b4a"]
    v_w = (hc @ c["w4c"].T + c["b4c"]).squeeze(-1)
    a_w = mu_w + std * eps.double()
    lp_w = (-((a_w - mu_w) ** 2) / (2 * std ** 2) - std.log() - HALF_LOG_2PI).sum(-1)
    assert_close("mu", mu_o.cpu().numpy(), mu_w.numpy(), rtol=1e-5, atol=1e-6)
    assert_close("value", vals.cpu().numpy(), v_w.numpy(), rtol=1e-5, atol=1e-6)
    assert_close("actions", acts.cpu().numpy(), a_w.numpy(), rtol=1e-5, atol=1e-6)
    assert_close("log_prob", logp.cpu().numpy(), lp_w.numpy(), rtol=1e-5, atol=1e-5)
    assert torch.equal(sig_o.cpu(), std.float().expand(n, na))


# ---------------------------------------------------------------------------------------------------- GPU: PPO end to end
def make_pair(dev, na, n, t, cfg, precision="3xtf32", seed=3):
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    params = init_actor_critic_params(OBS, PRIV, na, tuple(HECTOR["actor_hidden_dims"]), tuple(HECTOR["critic_hidden_dims"]),
                                      seed=seed)
    ac = ActorCritic(OBS, PRIV, na, **HECTOR, device=dev, precision=precision)
    ac.load_state_dict(params)
    alg = PPO(ac, device=dev, **cfg)
    alg.init_storage(n, t, [OBS], [PRIV], [na])
    return alg, PolicyOraclePPO(params, n, t, **cfg), params


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("na", [7, 23], ids=["fused-7", "generic-23"])
def test_ppo_matches_oracle(lib, cuda_device, na):
    """Act with injected eps over the golden case's rollout (64 envs x 24 steps) and one fixed-schedule update of 5 epochs
    x 4 minibatches (20 Adam steps) in 3xTF32, against the oracle at test_ppo_parity.py's fp32-grade tolerances."""
    dev = cuda_device
    n, t = mg.PPO_CASE["n"], mg.PPO_CASE["t"]
    cfg = dict(mg.PPO_ALG, schedule="fixed")
    alg, ora, params = make_pair(dev, na, n, t, cfg)
    assert alg.actor_critic.fused_head == (na <= 15)
    g = torch.Generator().manual_seed(0)
    for _ in range(t):
        o, co, eps = torch.randn(n, OBS, generator=g), torch.randn(n, PRIV, generator=g), torch.randn(n, na, generator=g)
        rew, dones, tos = torch.rand(n, generator=g), torch.rand(n, generator=g) < 0.1, torch.rand(n, generator=g) < 0.05
        alg.injected_eps = eps.to(dev)
        alg.act(o.to(dev), co.to(dev))
        ora.act(o, co, eps)
        alg.process_env_step(rew.to(dev), dones.to(dev), {"time_outs": tos.to(dev)})
        ora.process_env_step(rew, dones, {"time_outs": tos})
    last = torch.randn(n, PRIV, generator=g)
    alg.compute_returns(last.to(dev))
    ora.compute_returns(last)
    s = alg.storage
    for k in ("actions", "values", "mu", "actions_log_prob"):
        assert rel_l2(getattr(s, k).cpu(), ora.st[k]) < 1e-5, (k, rel_l2(getattr(s, k).cpu(), ora.st[k]))
    for k in ("actions", "values", "returns", "advantages", "actions_log_prob", "mu", "sigma", "rewards"):
        getattr(s, k).copy_(ora.st[k])            # the update starts from identical rollout data
    perm = torch.randperm(n * t, generator=g)
    alg.injected_perm = perm
    v_loss, s_loss = alg.update()
    w_vl, w_sl = ora.update(perm)
    assert abs(v_loss - w_vl) < 2e-5 * max(1.0, abs(w_vl)) and abs(s_loss - w_sl) < 2e-5, (v_loss, w_vl, s_loss, w_sl)
    sd = alg.actor_critic.state_dict()
    assert list(sd) == ora.order
    lr = cfg["learning_rate"]
    for k in ora.order:
        got, want, init = sd[k].cpu().double(), ora.params[k].detach().double(), params[k].double()
        err = (got - want).abs()
        off = err > (lr * 1e-2 + 1e-5 * want.abs())
        assert int(off.sum()) <= max(1, got.numel() // 10000), f"{k}: {int(off.sum())} of {got.numel()} beyond rtol 1e-5 / atol lr*1e-2"
        assert float(err.max()) <= 0.1 * lr, f"{k}: max error {float(err.max()):.3e}"
        assert float((got - want).norm() / (want - init).norm().clamp_min(1e-30)) < 1e-3, k


# ---------------------------------------------------------------------------------------------------- GPU: launches
def _rollout(alg, g, tpl):
    dev, s = alg.device, alg.storage
    for _ in range(s.num_transitions_per_env):
        obs, cobs = tpl.observations(alg, g)
        alg.act(obs, cobs)
        alg.process_env_step(torch.rand(s.num_envs, generator=g).to(dev), torch.zeros(s.num_envs, dtype=torch.bool, device=dev), {})
    alg.compute_returns(cobs)


@pytest.mark.gpu
@pytest.mark.parametrize("na", [7, 23], ids=["fused-7", "generic-23"])
def test_launch_sequence(lib, cuda_device, na):
    """Recorded with test_ppo_launches.py's Recorder.  7 actions: act is the draw, three grouped forward launches and
    hb_ppo_act_fused, captured into the slot's graph; updates run hb_ppo_head_fused eagerly in the first update, capture
    it in the second and replay the captured graphs from then on.  23 actions: the draw, four GEMMs per network and
    hb_ppo_act_head; each update launches hb_ppo_loss_head eagerly."""
    import test_ppo_launches as tpl
    from isaac_b200._lib import HB_GEMM_TF32
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    dev = cuda_device
    ac = ActorCritic(OBS, PRIV, na, **HECTOR, device=dev)
    alg = PPO(ac, device=dev, num_learning_epochs=1, num_mini_batches=2, schedule="fixed")
    n = 64
    alg.init_storage(n, 4, [OBS], [PRIV], [na])
    fused = na <= 15
    g = torch.Generator().manual_seed(4)
    obs, cobs = tpl.observations(alg, g)
    rec = tpl.record(alg, lambda: alg.act(obs, cobs))
    if fused:
        body = [*tpl.grouped_forward(ac, n, HB_GEMM_TF32), ("hb_ppo_act_fused",)]
    else:
        body = [*tpl.one_net_forward(ac, "actor", n, HB_GEMM_TF32), *tpl.one_net_forward(ac, "critic", n, HB_GEMM_TF32),
                ("hb_ppo_act_head",)]
    assert rec.calls == [("hb_ppo_draw_normal",), *body]
    assert rec.capturing == [fused] * len(rec.calls) and len(alg._act_graphs) == int(fused)
    alg.process_env_step(torch.rand(n, generator=g).to(dev), torch.zeros(n, dtype=torch.bool, device=dev), {})
    alg.storage.clear()
    head = "hb_ppo_head_fused" if fused else "hb_ppo_loss_head"
    for update in range(3):
        _rollout(alg, g, tpl)
        rec = tpl.record(alg, alg.update)
        heads = [cap for (name, *_), cap in zip(rec.calls, rec.capturing) if name == head]
        other = "hb_ppo_loss_head" if fused else "hb_ppo_head_fused"
        assert not any(c[0] == other for c in rec.calls)
        if not fused or update == 0:            # eager: one launch per minibatch
            assert heads == [False, False], (update, heads)
        elif update == 1:                       # captured into the minibatch graphs
            assert heads == [True, True], (update, heads)
        else:                                   # replayed: the recorder sees no call
            assert heads == [], (update, heads)
    assert len(alg._update_graphs) == (2 if fused else 0)


# ---------------------------------------------------------------------------------------------------- GPU: runner
class StubVecEnv:
    """The VecEnv surface OnPolicyRunner uses, in torch: observations are fixed random projections of the last actions
    plus noise, the reward favours small actions, and episodes time out after `max_episode_length` steps."""

    def __init__(self, num_envs, num_actions, device, seed=0):
        self.num_envs, self.num_obs, self.num_privileged_obs, self.num_actions = num_envs, OBS, PRIV, num_actions
        self.max_episode_length, self.device = 6, device
        self.g = torch.Generator(device=device).manual_seed(seed)
        self.proj_obs = torch.randn(num_actions, OBS, generator=self.g, device=device) / num_actions ** 0.5
        self.proj_priv = torch.randn(num_actions, PRIV, generator=self.g, device=device) / num_actions ** 0.5
        self.episode_length_buf = torch.zeros(num_envs, dtype=torch.long, device=device)
        self.reset()

    def _observe(self, actions):
        self.obs = torch.tanh(actions @ self.proj_obs) + 0.1 * torch.randn(self.num_envs, OBS, generator=self.g, device=self.device)
        self.priv = torch.tanh(actions @ self.proj_priv)

    def reset(self):
        self.episode_length_buf.zero_()
        self._observe(torch.zeros(self.num_envs, self.num_actions, device=self.device))
        return self.obs, self.priv

    def get_observations(self):
        return self.obs

    def get_privileged_observations(self):
        return self.priv

    def step(self, actions):
        self.episode_length_buf += 1
        dones = self.episode_length_buf >= self.max_episode_length
        self.episode_length_buf[dones] = 0
        self._observe(actions.clamp(-5.0, 5.0))
        rewards = -(actions ** 2).mean(-1)
        return self.obs, self.priv, rewards, dones, {"time_outs": dones.clone()}


@pytest.mark.gpu
@pytest.mark.parametrize("na", [23, 7], ids=["generic-23", "fused-7"])
def test_runner_learns_and_round_trips_checkpoints(lib, cuda_device, tmp_path, na):
    """OnPolicyRunner.learn over the stub env for three iterations, with logging and checkpoints; the checkpoint's
    state_dict has the reference module's keys and std shape, and loads back into a new runner.  7 actions take the
    fused act graphs and, from the second update on, the update graphs; 23 actions take neither."""
    from isaac_b200.algo import OnPolicyRunner
    from test_actor_critic_config import reference_modules
    from test_runner import TRAIN_CFG
    dev = cuda_device
    cfg = dict(TRAIN_CFG, runner=dict(TRAIN_CFG["runner"], num_steps_per_env=8, save_interval=1))
    runner = OnPolicyRunner(StubVecEnv(128, na, dev), cfg, log_dir=str(tmp_path), device=str(dev))
    w0 = runner.alg.actor_critic.flat.clone()
    runner.learn(num_learning_iterations=3)
    torch.cuda.synchronize()
    alg = runner.alg
    assert runner.current_learning_iteration == 3 and not torch.equal(w0, alg.actor_critic.flat)
    assert torch.isfinite(alg.actor_critic.flat).all() and np.isfinite(runner.last_log["Loss/surrogate"])
    assert (len(alg._act_graphs) > 0) == (na <= 15) and (len(alg._update_graphs) > 0) == (na <= 15)
    path = os.path.join(tmp_path, "model_3.pt")
    assert os.path.exists(path)
    sd = torch.load(path, map_location="cpu")["model_state_dict"]
    ref = reference_modules(OBS, PRIV, na, HECTOR["actor_hidden_dims"], HECTOR["critic_hidden_dims"], "elu")
    assert list(sd) == [k for k, _ in ref.named_parameters()]
    assert sd["std"].shape == ref.std.shape == (na,)
    ref.load_state_dict(sd, strict=True)
    runner2 = OnPolicyRunner(StubVecEnv(128, na, dev, seed=1), cfg, log_dir=None, device=str(dev))
    runner2.load(path)
    assert torch.equal(runner2.alg.actor_critic.flat, alg.actor_critic.flat) and runner2.alg._step == alg._step
    assert torch.equal(runner2.alg._exp_avg, alg._exp_avg) and torch.equal(runner2.alg._exp_avg_sq, alg._exp_avg_sq)
    runner2.learn(num_learning_iterations=1)
    assert runner2.current_learning_iteration == 4 and torch.isfinite(runner2.alg.actor_critic.flat).all()
