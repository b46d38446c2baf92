"""CPU reference of the library's device generator (numpy): Philox4x32-10 and the draws the kernels take from it.

Two streams use it, both keyed by a 64-bit seed and indexed by a 64-bit counter that lives in device memory:

- the env step (isaac_b200/csrc/env_kernels.cu, make_rng / rng_uniform4 / rng_normal4): counter words
  (env, slot, step lo, step hi), key = the env's seed (`HectorFreeEnvB200._rng_state` = {step counter, key});
- PPO.act's action sample (ppo_kernels.cu, draw_normal_kernel): counter words
  (quad lo, PPO_TAG ^ quad hi, call lo, call hi), key = `PPO._eps_state[2]`.

Uniforms are the top 24 bits of a word times 2^-24 (exact in fp32, in [0, 1)).  Normals are Box-Muller on the four words
of one call: radii from words x and z (as (top 24 bits + 1) * 2^-24, in (0, 1]), angles from words y and w, in the order
(r0 cos, r0 sin, r1 cos, r1 sin).  The kernels evaluate them with __logf / __sincosf in fp32; here they are computed in
float64 and rounded once, so kernel and reference differ by the intrinsics' error only.

This module is the one place in Python that knows the env step's slot layout.
"""
from __future__ import annotations

import numpy as np
import torch

# slots of one env and step (env_kernels.cu): z_action[<=24] | z_obs[<=80] | u_reset[<=29] | u_cmd[3] | u_push[5] | u_delay
SLOT_Z_ACTION, SLOT_Z_OBS, SLOT_U_RESET, SLOT_U_CMD, SLOT_U_PUSH, SLOT_U_DELAY = 0, 6, 26, 34, 35, 37
PPO_TAG = 0x50504F00                 # second counter word of the action-sample stream ("PPO\0")

_M32 = np.uint64(0xFFFFFFFF)
_MUL0, _MUL1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_BUMP0, _BUMP1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def split64(v: int):
    """(lo, hi) 32-bit words of a 64-bit value; a signed int64 (as the device stores a seed >= 2^63) wraps the same way."""
    v = int(v) & 0xFFFFFFFFFFFFFFFF
    return v & 0xFFFFFFFF, v >> 32


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (hb_common.cuh): 10 rounds, the key bumped after each.  Arguments broadcast (uint32 values);
    returns the four output words as uint32 arrays."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(x, dtype=np.uint64) & _M32 for x in np.broadcast_arrays(c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0, p1 = _MUL0 * c0, _MUL1 * c2              # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + _BUMP0) & _M32, (k1 + _BUMP1) & _M32
    return tuple(w.astype(np.uint32) for w in (c0, c1, c2, c3))


def uniforms(w) -> np.ndarray:
    """float32(w >> 8) * 2^-24: exact, in [0, 1)."""
    return (np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)


def normals4(x, y, z, w) -> np.ndarray:
    """Box-Muller on the four words of one call, in float64, rounded to fp32: [..., 4] = (r0 cos, r0 sin, r1 cos, r1 sin)."""
    top = lambda v: (np.asarray(v, dtype=np.uint32) >> np.uint32(8)).astype(np.float64)
    r0 = np.sqrt(-2.0 * np.log((top(x) + 1.0) * 2.0 ** -24))
    r1 = np.sqrt(-2.0 * np.log((top(z) + 1.0) * 2.0 ** -24))
    a0, a1 = 2.0 * np.pi * top(y) * 2.0 ** -24, 2.0 * np.pi * top(w) * 2.0 ** -24
    return np.stack((r0 * np.cos(a0), r0 * np.sin(a0), r1 * np.cos(a1), r1 * np.sin(a1)), axis=-1).astype(np.float32)


def _env_words(key: int, step: int, n: int, slot: int, count: int):
    """The Philox calls slot, slot+1, ... that hold `count` values of every env: four [n, calls] word arrays."""
    k0, k1 = split64(key)
    s0, s1 = split64(step)
    calls = (count + 3) // 4
    env = np.arange(n, dtype=np.uint64)[:, None]
    slots = slot + np.arange(calls, dtype=np.uint64)[None, :]
    return philox4x32_10(env, slots, s0, s1, k0, k1)


def env_uniforms(key: int, step: int, n: int, slot: int, count: int) -> np.ndarray:
    """[n, count] uniforms of a per-env vector that starts at `slot` (rng_uniforms: value i is word i % 4 of call
    slot + i // 4, so a sub-vector starting at `first` is columns first .. of this array)."""
    w = _env_words(key, step, n, slot, count)
    return uniforms(np.stack(w, axis=-1)).reshape(n, -1)[:, :count]


def env_normals(key: int, step: int, n: int, slot: int, count: int) -> np.ndarray:
    """[n, count] normals of a per-env vector that starts at `slot` (value i is element i % 4 of call slot + i // 4)."""
    return normals4(*_env_words(key, step, n, slot, count)).reshape(n, -1)[:, :count]


def env_draws(key: int, step: int, n: int, ndof: int, nobs: int, actions=None):
    """Every draw the env kernels take from the device generator at step counter `step`, as the
    isaac_b200.synthetic.NoiseFrame the oracle consumes (CPU, fp32).  `actions` ([n, ndof], default zeros) is passed
    through: it is the policy output, not a draw."""
    from isaac_b200.synthetic import NoiseFrame
    if not (0 < ndof <= 24 and 0 < nobs <= 80):
        raise ValueError("the slot layout holds at most 24 action and 80 observation columns")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    if actions is None:
        actions = torch.zeros(n, ndof)
    return NoiseFrame(actions=torch.as_tensor(actions, dtype=torch.float32).cpu(),
                      u_delay=t(env_uniforms(key, step, n, SLOT_U_DELAY, 1)),
                      z_action=t(env_normals(key, step, n, SLOT_Z_ACTION, ndof)),
                      u_cmd=t(env_uniforms(key, step, n, SLOT_U_CMD, 3)),
                      u_push=t(env_uniforms(key, step, n, SLOT_U_PUSH, 5)),
                      u_reset=t(env_uniforms(key, step, n, SLOT_U_RESET, ndof + 5)),     # dof jitter, root xy, command
                      z_obs=t(env_normals(key, step, n, SLOT_Z_OBS, nobs)))


def ppo_normals(key: int, call: int, count: int) -> np.ndarray:
    """The `count` N(0,1) values hb_ppo_draw_normal writes at call counter `call` (element i is element i % 4 of the
    Philox call for quad i // 4)."""
    k0, k1 = split64(key)
    c0, c1 = split64(call)
    q = np.arange((count + 3) // 4, dtype=np.uint64)
    w = philox4x32_10(q & _M32, np.uint64(PPO_TAG) ^ (q >> np.uint64(32)), c0, c1, k0, k1)
    return normals4(*w).reshape(-1)[:count]
