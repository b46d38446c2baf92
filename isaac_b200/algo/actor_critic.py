"""`ActorCritic` with the reference's interface (algo/ppo/actor_critic.py:36-128) on the tcgen05 GEMM path.

Parameters live in ONE flat fp32 buffer so that gradient all-reduce, clip_grad_norm_ and Adam are single
passes.  Each `nn.Linear` is a packed matrix `P[out_pad, ld]` = `[W | b | 0-pad]` with `ld = pitch(in + 1)` (whole 128-byte rows):
  * the forward GEMM reads `W` through a TMA tensor map with K extent `in` and takes the bias from column `in`;
  * the weight-gradient GEMM multiplies by the activations extended with a constant ones column, so the bias
    gradient is simply column `in` of the packed gradient — no separate reduction kernel;
  * rows are 16-byte aligned (615*4 and 1050*4 are not, SURVEY.md §7 hard part 2).
Like the reference, each network has one or more hidden layers of its own widths and the activation `get_activation`
names (ELU, SELU, ReLU, LeakyReLU, Tanh, Sigmoid), evaluated in the GEMM epilogues.  `state_dict()` / `load_state_dict()`
use the reference's `nn.Sequential` keys (`actor.{0,2,...,2d}.{weight,bias}` for d hidden layers, `critic.…`, `std`), so
checkpoints interchange.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import Dict, List, Optional

import torch

from .. import _lib
from .._lib import (GemmDesc, HB_ACT_ELU, HB_ACT_LRELU, HB_ACT_RELU, HB_ACT_SELU, HB_ACT_SIGMOID, HB_ACT_TANH, HB_EPI_ACT_BWD,
                    HB_EPI_ATOMIC_ADD, HB_EPI_BIAS, HB_EPI_BIAS_ACT, HB_GEMM_3XTF32, HB_GEMM_TF32, PPO_MAX_ACTIONS,
                    PPO_MAX_FUSED_ACTIONS)

# the names get_activation resolves (algo/ppo/actor_critic.py), "crelu" being nn.ReLU there too
ACTIVATIONS = {"elu": HB_ACT_ELU, "selu": HB_ACT_SELU, "relu": HB_ACT_RELU, "crelu": HB_ACT_RELU, "lrelu": HB_ACT_LRELU,
               "tanh": HB_ACT_TANH, "sigmoid": HB_ACT_SIGMOID}


def pitch(n: int) -> int:
    """Row pitch (floats) of the buffers the TMA reads and writes here: whole 128-byte lines.  A 16-byte-aligned pitch is
    all the TMA asks for, but every 128-byte box row then straddles two lines and five 32-byte sectors instead of four:
    measured on the layer-1 forward GEMM (K = 1050), 79.9 us at a pitch of 1052 floats against 68.2 us at 1056."""
    return (n + 31) // 32 * 32


def pad4(n: int) -> int:
    return (n + 3) // 4 * 4


class _Layer:
    __slots__ = ("net", "index", "fan_in", "fan_out", "rows", "ld", "offset", "last")

    def __init__(self, net, index, fan_in, fan_out, last, offset):
        self.net, self.index, self.fan_in, self.fan_out, self.last, self.offset = net, index, fan_in, fan_out, last, offset
        self.rows = (fan_out + 15) // 16 * 16 if last else fan_out          # output layers are padded to a multiple of the smallest UMMA N
        self.ld = pitch(fan_in + 1)

    @property
    def numel(self):
        return self.rows * self.ld


def _desc(lib, scratch, kw):
    d = GemmDesc()
    for k, v in kw.items():
        setattr(d, k, v)
    if scratch is not None:
        d.precision = HB_GEMM_3XTF32
        need = int(lib.hb_gemm_workspace_floats(C.byref(d)))
        if scratch[0] is None or scratch[0].numel() < need:
            scratch[0] = torch.empty(need, device=scratch[1])
        d.workspace, d.workspace_floats = scratch[0].data_ptr(), scratch[0].numel()
    return d


def gemm(lib, st, scratch=None, **kw):
    """One hb_gemm_tf32 call.  `scratch` (a one-element list holding a float tensor or None) switches the call to
    HB_GEMM_3XTF32 and supplies / grows the workspace of the split operands."""
    _lib.check(lib.hb_gemm_tf32(C.byref(_desc(lib, scratch, kw)), st), "hb_gemm_tf32")


def gemm2(lib, st, scratch0, kw0, scratch1, kw1):
    """The same GEMM of both networks in one launch (hb_gemm_tf32_grouped)."""
    _lib.check(lib.hb_gemm_tf32_grouped(C.byref(_desc(lib, scratch0, kw0)), C.byref(_desc(lib, scratch1, kw1)), st),
               "hb_gemm_tf32_grouped")


class ActorCritic:
    is_recurrent = False

    def __init__(self, num_actor_obs, num_critic_obs, num_actions, actor_hidden_dims=(256, 256, 256),
                 critic_hidden_dims=(256, 256, 256), init_noise_std=1.0, activation=None, device="cuda:0", **kwargs):
        precision = kwargs.pop("precision", "tf32")
        if precision not in ("tf32", "3xtf32"):
            raise ValueError("precision must be 'tf32' or '3xtf32'")
        if kwargs:
            print("ActorCritic.__init__ got unexpected arguments, which will be ignored: " + str(list(kwargs)))
        if not 1 <= num_actions <= PPO_MAX_ACTIONS:
            raise ValueError(f"num_actions = {num_actions}: the PPO head kernels take 1 to {PPO_MAX_ACTIONS} actions")
        activation = "elu" if activation is None else activation
        if activation not in ACTIVATIONS:
            raise ValueError(f"unknown activation {activation!r}: one of {sorted(ACTIVATIONS)}")
        for name, dims in (("actor_hidden_dims", actor_hidden_dims), ("critic_hidden_dims", critic_hidden_dims)):
            if len(dims) == 0:
                raise ValueError(f"{name} is empty: each network needs at least one hidden layer")
            if min(dims) <= 64:
                raise ValueError(f"{name} = {list(dims)}: hidden widths must exceed 64 - the data-gradient GEMM into a hidden "
                                 "layer reads the weights as an MN-major B operand with N = that layer's width, and an "
                                 "MN-major B operand needs N > 64")
        self._lib = _lib.load()
        self.activation = activation
        self.hb_activation = ACTIVATIONS[activation]        # hb_activation of every GEMM epilogue and of the fused head
        self.device = torch.device(device)
        self.num_actor_obs, self.num_critic_obs, self.num_actions = num_actor_obs, num_critic_obs, num_actions
        self.layers: List[_Layer] = []
        off = 0
        for net, dims in (("actor", (num_actor_obs, *actor_hidden_dims, num_actions)),
                          ("critic", (num_critic_obs, *critic_hidden_dims, 1))):
            for i in range(len(dims) - 1):
                L = _Layer(net, 2 * i, dims[i], dims[i + 1], i == len(dims) - 2, off)
                self.layers.append(L)
                off += L.numel
        self.net_layers = {net: tuple(L for L in self.layers if L.net == net) for net in ("actor", "critic")}
        self.output_layers = (self.net_layers["actor"][-1], self.net_layers["critic"][-1])
        self._std_offset = off
        off += (num_actions + 15) // 16 * 16
        self.flat = torch.zeros(off, device=self.device)
        # the gradient buffer carries 8 spare floats behind the parameters: a data-parallel replica parks its loss
        # statistics there so that ONE all-reduce per optimizer step covers both (isaac_b200/parallel.py)
        self._grad_wire = torch.zeros(off + 8, device=self.device)
        self.grad = self._grad_wire[:off]
        # default nn.Linear initialisation, drawn in the reference's module construction order
        # (actor layers, critic layers, then std: actor_critic.py:54-83) so the same torch seed gives the same net
        for L in self.layers:
            lin = torch.nn.Linear(L.fan_in, L.fan_out)
            self._matrix(self.flat, L)[:L.fan_out, :L.fan_in] = lin.weight.detach().to(self.device)
            self._matrix(self.flat, L)[:L.fan_out, L.fan_in] = lin.bias.detach().to(self.device)
        self.flat[self._std_offset:self._std_offset + num_actions] = init_noise_std
        self.distribution = None
        self._ws: Dict[int, dict] = {}
        self._last: Optional[dict] = None
        # "tf32": operands truncated to TF32 by the tensor core (fast path).  "3xtf32": hi/lo split operands, three
        # partial products in one fp32 accumulator - fp32-grade results like the reference's nn.Linear (parity mode)
        self.precision = precision
        # 3xTF32 workspaces, one per network: a grouped launch takes both networks' at once, so growing a shared buffer for
        # the second descriptor would free the first one's
        self._scratch = {"actor": [None, self.device], "critic": [None, self.device]}

    def rebind(self, flat: torch.Tensor, grad_wire: torch.Tensor) -> None:
        """Move the flat parameter / gradient buffers to caller-provided storage of the same size (symmetric memory for
        data-parallel replicas); contents are the caller's responsibility."""
        if flat.numel() != self.flat.numel() or grad_wire.numel() != self._grad_wire.numel():
            raise ValueError("rebind needs buffers of the same size")
        self.flat, self._grad_wire = flat, grad_wire
        self.grad = grad_wire[:flat.numel()]

    # ------------------------------------------------------------------ parameter views
    def _matrix(self, flat, L):
        return flat[L.offset:L.offset + L.numel].view(L.rows, L.ld)

    @property
    def std(self):
        return self.flat[self._std_offset:self._std_offset + self.num_actions]

    def named_views(self, buf):
        """Named views of any buffer with the flat layout (parameters, gradients, Adam moments), in the order of the
        reference module's `parameters()` (std first, then actor, critic)."""
        yield "std", buf[self._std_offset:self._std_offset + self.num_actions]
        for L in self.layers:
            P = self._matrix(buf, L)
            yield f"{L.net}.{L.index}.weight", P[:L.fan_out, :L.fan_in]
            yield f"{L.net}.{L.index}.bias", P[:L.fan_out, L.fan_in]

    def named_parameters(self):
        return self.named_views(self.flat)

    def named_gradients(self):
        return self.named_views(self.grad)

    def parameters(self):
        return [p for _, p in self.named_parameters()]

    def state_dict(self):
        return OrderedDict((k, v.detach().clone().contiguous()) for k, v in self.named_parameters())

    def load_state_dict(self, sd, strict=True):
        views = dict(self.named_parameters())
        if strict and set(sd) != set(views):
            raise KeyError(f"state_dict keys differ: {sorted(set(sd) ^ set(views))}")
        for k, v in sd.items():
            if k in views:
                views[k].copy_(v.to(self.device))

    def to(self, device):
        if torch.device(device) != self.device:
            raise ValueError("ActorCritic lives on the device it was created on")
        return self

    def train(self, mode=True):
        return self

    def eval(self):
        return self

    def reset(self, dones=None):
        pass

    def forward(self):
        raise NotImplementedError

    # ------------------------------------------------------------------ workspaces
    def workspace(self, m: int) -> dict:
        """Activation buffers for a batch of m rows; hidden activations carry the constant ones column at
        index `width` that feeds the bias gradients."""
        ws = self._ws.get(m)
        if ws is None:
            z = lambda r, c: torch.zeros(r, c, device=self.device)
            ws = {"m": m}
            for net, Ls in self.net_layers.items():
                hs = []
                for L in Ls[:-1]:
                    h = z(m, pitch(L.fan_out + 1))
                    h[:, L.fan_out] = 1.0
                    hs.append(h)
                ws[net] = {"h": hs, "out": z(m, Ls[-1].rows), "d_out": z(m, Ls[-1].rows),
                           "dz": [z(m, pitch(L.fan_out)) for L in Ls[:-1]]}
            self._ws[m] = ws
        return ws

    def _scratch_for(self, net: str):
        return self._scratch[net] if self.precision == "3xtf32" else None

    # ------------------------------------------------------------------ GEMM descriptors
    @property
    def fused_head(self) -> bool:
        """Both last hidden layers are 128 wide (and at most 15 actions): the update path evaluates the output layers inside
        the loss kernel (hb_ppo_head_fused) instead of as 128-row tensor-core tiles with 10 / 1 useful columns."""
        return all(L.fan_in == 128 for L in self.output_layers) and self.num_actions <= PPO_MAX_FUSED_ACTIONS

    def _fwd_desc(self, net: str, i: int, a: torch.Tensor, ws: dict):
        """Forward GEMM of layer i of `net` on a [m, ld] (ld % 4 == 0, only the first fan_in columns are read), bias and (hidden
        layers) the activation in the epilogue.  Returns the kwargs of gemm / gemm2 and the output the GEMM writes."""
        L = self.net_layers[net][i]
        P = self._matrix(self.flat, L)
        d = ws[net]["out"] if L.last else ws[net]["h"][i]
        return dict(A=a.data_ptr(), B=P.data_ptr(), D=d.data_ptr(), M=ws["m"], N=L.rows if L.last else L.fan_out, K=L.fan_in,
                    lda=a.stride(0), ldb=L.ld, ldd=d.stride(0), epilogue=HB_EPI_BIAS if L.last else HB_EPI_BIAS_ACT,
                    bias=P.data_ptr() + L.fan_in * 4, bias_stride=L.ld, activation=self.hb_activation), d

    def _wgrad_desc(self, net: str, i: int, d_cur: torch.Tensor, x: torch.Tensor, ws: dict):
        """Weight gradient of layer i from d_cur, the gradient w.r.t. the layer's pre-activation output (x: the network's
        input): G[rows, fan_in + 1] += d_cur^T [rows, m] * [act_in | 1] [m, fan_in + 1], split-K atomics into self.grad."""
        L = self.net_layers[net][i]
        act_in = x if i == 0 else ws[net]["h"][i - 1]      # [m, fan_in (+ ones column)]
        return dict(A=d_cur.data_ptr(), B=act_in.data_ptr(), D=self._matrix(self.grad, L).data_ptr(), M=L.rows, N=L.fan_in + 1,
                    K=ws["m"], lda=d_cur.stride(0), ldb=act_in.stride(0), ldd=L.ld, a_mn_major=1, b_mn_major=1,
                    epilogue=HB_EPI_ATOMIC_ADD, split_k=0, activation=self.hb_activation)

    def _dgrad_desc(self, net: str, i: int, d_cur: torch.Tensor, ws: dict):
        """Data gradient of layer i > 0 through the previous activation f: dz_prev = (d_cur * W) . f'(h_prev).  Returns the
        kwargs and dz_prev, the d_cur of layer i - 1."""
        L = self.net_layers[net][i]
        h_prev, dz = ws[net]["h"][i - 1], ws[net]["dz"][i - 1]
        return dict(A=d_cur.data_ptr(), B=self._matrix(self.flat, L).data_ptr(), D=dz.data_ptr(), M=ws["m"], N=L.fan_in, K=L.rows,
                    lda=d_cur.stride(0), ldb=L.ld, ldd=dz.stride(0), b_mn_major=1, epilogue=HB_EPI_ACT_BWD, H=h_prev.data_ptr(),
                    ldh=h_prev.stride(0), activation=self.hb_activation), dz

    # ------------------------------------------------------------------ one network at a time
    def _mlp_forward(self, net: str, x: torch.Tensor, ws: dict):
        """x: [m, ld] with ld % 4 == 0 (only the first fan_in columns are read).  Returns out [m,16]."""
        lib, st = self._lib, torch.cuda.current_stream(self.device).cuda_stream
        a = x
        for i in range(len(self.net_layers[net])):
            kw, a = self._fwd_desc(net, i, a, ws)
            gemm(lib, st, self._scratch_for(net), **kw)
        return a

    def _mlp_backward(self, net: str, x: torch.Tensor, ws: dict):
        """Gradients of every packed matrix of `net` from d_out (filled by the loss head); accumulates into
        self.grad with split-K atomics (the buffer is zero on entry: Adam zeroes it).  Per layer, top down: the weight
        gradient, then the data gradient that feeds the layer below."""
        lib, st = self._lib, torch.cuda.current_stream(self.device).cuda_stream
        d_cur = ws[net]["d_out"]
        for i in reversed(range(len(self.net_layers[net]))):
            gemm(lib, st, self._scratch_for(net), **self._wgrad_desc(net, i, d_cur, x, ws))
            if i > 0:
                kw, d_cur = self._dgrad_desc(net, i, d_cur, ws)
                gemm(lib, st, self._scratch_for(net), **kw)

    # ------------------------------------------------------------------ both networks, layer by layer, grouped launches
    def _hidden_depths(self):
        return len(self.net_layers["actor"]) - 1, len(self.net_layers["critic"]) - 1

    def _gemm_both(self, kwc, kwa):
        """Layer i's GEMM of both networks in one grouped launch (the critic's, the larger problem, first) when both have a
        hidden layer i; otherwise one launch of the network that has it (the other's kwargs are None)."""
        lib, st = self._lib, torch.cuda.current_stream(self.device).cuda_stream
        if kwc is not None and kwa is not None:
            gemm2(lib, st, self._scratch_for("critic"), kwc, self._scratch_for("actor"), kwa)
        elif kwc is not None:
            gemm(lib, st, self._scratch_for("critic"), **kwc)
        else:
            gemm(lib, st, self._scratch_for("actor"), **kwa)

    def forward_both(self, xa: torch.Tensor, xc: torch.Tensor, ws: dict):
        """The hidden layers of the actor (on xa) and the critic (on xc), input side first: one grouped launch per layer
        index both networks have, then single launches for the deeper network's remaining layers (hector: three grouped
        launches instead of six).  Returns the last hidden activations (h_actor, h_critic)."""
        na, nc = self._hidden_depths()
        a, c = xa, xc
        for i in range(max(na, nc)):
            kwa = kwc = None
            if i < na:
                kwa, a = self._fwd_desc("actor", i, a, ws)
            if i < nc:
                kwc, c = self._fwd_desc("critic", i, c, ws)
            self._gemm_both(kwc, kwa)
        return a, c

    def backward_both(self, xa: torch.Tensor, xc: torch.Tensor, ws: dict):
        """Gradients of the hidden layers of both networks from the gradients w.r.t. the last hidden pre-activations (left in
        ws by hb_ppo_head_fused), top layer index first: per layer index one data-gradient launch (critical path first) and
        one weight-gradient launch, grouped where both networks have that hidden layer (hector: five launches for ten
        GEMMs)."""
        na, nc = self._hidden_depths()
        da, dc = ws["actor"]["dz"][-1], ws["critic"]["dz"][-1]
        for i in reversed(range(max(na, nc))):
            wa = self._wgrad_desc("actor", i, da, xa, ws) if i < na else None
            wc = self._wgrad_desc("critic", i, dc, xc, ws) if i < nc else None
            if i > 0:
                kwa = kwc = None
                if i < na:
                    kwa, da = self._dgrad_desc("actor", i, da, ws)
                if i < nc:
                    kwc, dc = self._dgrad_desc("critic", i, dc, ws)
                self._gemm_both(kwc, kwa)
            self._gemm_both(wc, wa)

    def _as_operand(self, x: torch.Tensor, width: int) -> torch.Tensor:
        """TMA needs 16-byte aligned rows: use x in place when its row stride allows, else stage a padded copy."""
        if x.is_cuda and x.dtype == torch.float32 and x.stride(-1) == 1 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0:
            return x
        buf = torch.zeros(x.shape[0], pitch(width + 1), device=self.device)
        buf[:, :width] = x
        return buf

    # ------------------------------------------------------------------ reference-named API
    def act_inference(self, observations):
        ws = self.workspace(observations.shape[0])
        out = self._mlp_forward("actor", self._as_operand(observations, self.num_actor_obs), ws)
        return out[:, :self.num_actions].clone()

    def evaluate(self, critic_observations, **kwargs):
        ws = self.workspace(critic_observations.shape[0])
        out = self._mlp_forward("critic", self._as_operand(critic_observations, self.num_critic_obs), ws)
        return out[:, :1].clone()

    def update_distribution(self, observations):
        ws = self.workspace(observations.shape[0])
        out = self._mlp_forward("actor", self._as_operand(observations, self.num_actor_obs), ws)
        mean = out[:, :self.num_actions]
        self.distribution = torch.distributions.Normal(mean, mean * 0.0 + self.std, validate_args=False)

    def act(self, observations, **kwargs):
        self.update_distribution(observations)
        return self.distribution.sample()

    def get_actions_log_prob(self, actions):
        return self.distribution.log_prob(actions).sum(dim=-1)

    @property
    def action_mean(self):
        return self.distribution.mean

    @property
    def action_std(self):
        return self.distribution.stddev

    @property
    def entropy(self):
        return self.distribution.entropy().sum(dim=-1)
