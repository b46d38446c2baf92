"""The frame-stack shift, next[:, :row-frame] = prev[:, frame:row] (hector_env.py:246-261), through its three entry
points: hb_stack_shift, hb_env_stack_observations and hb_env_stack_finalize (the last against the two separate calls
hb_env_stack_observations + hb_env_reset_finalize).  Each case checks the carried frames against torch, zero for the
reset envs where the call zeroes them, and that nothing else is written: the outputs sit inside sentinel guards, and the
newest-frame slot and the row padding keep their fill.

Shapes: the three built robots' stacks (compiled kernels), dense and at the 128-byte pitch; stacks with no compiled
kernel (the runtime-shape kernel) covering frame % 4 = 0..3 and rows that are not whole vectors; depth-1 stacks, which
carry nothing over.  Sizes 1, 37, 1003 and 4096 envs; buffers 16-byte aligned and 4 bytes off, the latter taking the
scalar shift.  A dispatch pin checks which kernel each case runs: equal outputs would hide a built shape that fell onto
the runtime-shape kernel (4.0-4.2 TB/s against 5.9 TB/s for the compiled kernel, DESIGN.md section 1)."""
import re

import pytest
import torch

from isaac_b200.synthetic import make_tape

pytestmark = pytest.mark.gpu

GUARD = 256          # sentinel floats on each side of every buffer
SENTINEL, FILL = -3.0, 7.0


def pitch(row):
    return (row + 1 + 31) // 32 * 32


# (obs frame, frame_stack, priv frame, c_frame_stack)
BUILT = {"hector": (41, 15, 70, 15), "hector_full": (65, 15, 94, 15), "xbot": (47, 15, 73, 3)}
RUNTIME = {
    "f0_f1": (44, 5, 73, 4),        # frame % 4 = 0 (obs), 1 (priv)
    "f2_f3": (38, 6, 51, 3),        # frame % 4 = 2, 3; the dense priv row (153) is not whole vectors
    "hector_s4": (41, 4, 70, 4),    # a built robot's frames at a depth with no compiled kernel
    "depth1": (41, 1, 70, 1),       # no shift blocks: finalisation only
    "depth1_obs": (41, 1, 70, 3),   # one history carries nothing over
}
SIZES = [1, 37, 1003, 4096]

_envs = {}


def _env(n, dev):
    if n not in _envs:
        from test_env_parity import make_cuda_env
        _envs[n] = make_cuda_env(make_tape(n, 1, seed=5 + n, fall_prob=0.0), dev)[0]
    return _envs[n]


def _guarded(n, ld, off, dev, src=None):
    """[n, ld] view `off` floats past a 16-byte boundary, inside sentinel guards; filled with FILL unless `src`."""
    raw = torch.full((n * ld + 2 * GUARD,), SENTINEL, device=dev)
    view = raw[GUARD + off:GUARD + off + n * ld].view(n, ld)
    view.copy_(src) if src is not None else view.fill_(FILL)
    assert (view.data_ptr() % 16 == 0) == (off == 0)
    return raw, view


def _check(raw, new, prev, row, frame, off, zero=None):
    n, ld = new.shape
    assert (raw[:GUARD + off] == SENTINEL).all() and (raw[GUARD + off + n * ld:] == SENTINEL).all(), "store outside the stack"
    want = prev[:, frame:row].clone()
    if zero is not None:
        want[zero] = 0.0
    assert torch.equal(new[:, :row - frame], want)
    assert (new[:, row - frame:] == FILL).all(), "the newest-frame slot and the row padding belong to post-physics"


def _set_shape(env, shape, pitched):
    fo, s, fp, cs = shape
    p = env._p
    p.num_single_obs, p.frame_stack, p.num_single_priv, p.c_frame_stack = fo, s, fp, cs
    p.obs_ld, p.priv_ld = (pitch(fo * s), pitch(fp * cs)) if pitched else (0, 0)
    return fo * s, fp * cs, (p.obs_ld or fo * s), (p.priv_ld or fp * cs)


def _arm_finalize(env, reset, dev, seed):
    """The state post-physics leaves for the finalisation: reset flags, one ballot per 32-env tile, reward sums."""
    from isaac_b200 import _lib
    n = reset.numel()
    g = torch.Generator(device=dev).manual_seed(seed)
    tiles = (n + 31) // 32
    pad = torch.zeros(tiles * 32, dtype=torch.bool, device=dev)
    pad[:n] = reset
    ballots = (pad.view(tiles, 32).long() * (2 ** torch.arange(32, device=dev, dtype=torch.int64))).sum(1)
    env.reset_buf.copy_(reset)
    env.time_out_buf.copy_(torch.rand(n, device=dev, generator=g) < 0.5)
    env._time_outs_latched.zero_()
    env._scratch_ballots.copy_(torch.where(ballots >= 2 ** 31, ballots - 2 ** 32, ballots).to(torch.int32))
    env._scratch_sums.copy_(torch.rand(_lib.HB_NUM_REWARDS, dtype=torch.float64, device=dev, generator=g))
    env.reset_env_ids.fill_(-1)
    means = torch.zeros(_lib.HB_NUM_REWARDS, device=dev)
    env._b.episode_means, env._b.episode_means_prev, env._b.episode_ring = means.data_ptr(), None, None
    return means


def _run_env_entry(lib, env, dev, shape, pitched, off, fused, seed):
    from isaac_b200 import _lib
    n = env.num_envs
    row_o, row_p, ld_o, ld_p = _set_shape(env, shape, pitched)
    g = torch.Generator(device=dev).manual_seed(seed)
    prev_o, prev_p = torch.randn(n, ld_o, device=dev, generator=g), torch.randn(n, ld_p, device=dev, generator=g)
    reset = torch.rand(n, device=dev, generator=g) < 0.3
    reset[-1] = True                                    # the last, possibly partial tile
    (rpo, po), (rpp, pp) = _guarded(n, ld_o, off, dev, prev_o), _guarded(n, ld_p, off, dev, prev_p)
    (ro, no), (rp, np_) = _guarded(n, ld_o, off, dev), _guarded(n, ld_p, off, dev)
    means = _arm_finalize(env, reset, dev, seed) if fused is not None else None
    P, B, st = env._pp, env._pb, torch.cuda.current_stream(dev).cuda_stream
    args = (P, B, po.data_ptr(), pp.data_ptr(), no.data_ptr(), np_.data_ptr())
    if fused:
        _lib.check(lib.hb_env_stack_finalize(*args, env._host_count.data_ptr(), None, st), "hb_env_stack_finalize")
    else:
        _lib.check(lib.hb_env_stack_observations(*args, st), "hb_env_stack_observations")
        if fused is not None:
            _lib.check(lib.hb_env_reset_finalize(P, B, no.data_ptr(), np_.data_ptr(), env._host_count.data_ptr(), None, st),
                       "hb_env_reset_finalize")
    torch.cuda.synchronize()
    zero = reset if fused is not None else None
    _check(ro, no, prev_o, row_o, shape[0], off, zero)
    _check(rp, np_, prev_p, row_p, shape[2], off, zero)
    if fused is None:
        return None
    cnt = int(env._reset_count.item())
    assert cnt == int(reset.sum()) == int(env._host_count[0])
    assert torch.equal(env.reset_env_ids[:cnt].long(), reset.nonzero().flatten())
    return no.clone(), np_.clone(), cnt, means.clone(), env._time_outs_latched.clone(), env._scratch_sums.clone()


SHAPE_CASES = [(k, v, False) for k, v in BUILT.items()] + [(k, v, True) for k, v in BUILT.items()] + \
              [(k, v, False) for k, v in RUNTIME.items()] + [("f2_f3", RUNTIME["f2_f3"], True)]
SHAPE_IDS = [f"{k}-{'pitched' if p else 'dense'}" for k, _, p in SHAPE_CASES]


@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset4"])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("case", SHAPE_CASES, ids=SHAPE_IDS)
def test_stack_observations_shifts_both_histories(lib, cuda_device, case, n, off):
    _, shape, pitched = case
    _run_env_entry(lib, _env(n, cuda_device), cuda_device, shape, pitched, off, None, seed=n + off)


@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset4"])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("case", SHAPE_CASES, ids=SHAPE_IDS)
def test_stack_finalize_equals_separate_calls(lib, cuda_device, case, n, off):
    _, shape, pitched = case
    env = _env(n, cuda_device)
    a = _run_env_entry(lib, env, cuda_device, shape, pitched, off, False, seed=n + off)
    b = _run_env_entry(lib, env, cuda_device, shape, pitched, off, True, seed=n + off)
    for x, y in zip(a, b):
        assert (x == y) if isinstance(x, int) else torch.equal(x, y)


# (row, frame) of hb_stack_shift: hector's two dense histories and two other shapes
SHIFT_SHAPES = {"hector_obs": (615, 41), "hector_priv": (1050, 70), "r220_f44": (220, 44), "r153_f51": (153, 51)}


@pytest.mark.parametrize("reset", [False, True], ids=["plain", "reset"])
@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset4"])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("shape", list(SHIFT_SHAPES.values()), ids=list(SHIFT_SHAPES))
def test_stack_shift(lib, cuda_device, shape, n, off, reset):
    from isaac_b200 import _lib
    dev = cuda_device
    row, frame = shape
    g = torch.Generator(device=dev).manual_seed(row + n)
    prev = torch.randn(n, row, device=dev, generator=g)
    flags = torch.rand(n, device=dev, generator=g) < 0.3
    (_, p), (raw, new) = _guarded(n, row, off, dev, prev), _guarded(n, row, off, dev)
    rb = flags.to(torch.uint8) if reset else None
    _lib.check(lib.hb_stack_shift(p.data_ptr(), new.data_ptr(), rb.data_ptr() if reset else None, n, row, frame,
                                  torch.cuda.current_stream(dev).cuda_stream), "hb_stack_shift")
    torch.cuda.synchronize()
    _check(raw, new, prev, row, frame, off, flags if reset else None)


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if re.search(r"stack_shift|stack_finalize|reset_finalize_kernel", e.name)]


def _fixed(row, ld, frame):
    arg = r"\s*(?:\(int\))?{}u?\s*"           # demanglers print 615, 615u or (int)615
    return re.compile("FixedShift<" + ",".join(arg.format(v) for v in (row, ld, frame)) + ">")


@pytest.mark.parametrize("fused", [False, True], ids=["observations", "finalize"])
@pytest.mark.parametrize("case", SHAPE_CASES, ids=SHAPE_IDS)
def test_dispatch(lib, cuda_device, case, fused):
    """Built shapes run the compiled kernel of their (ROW, LD, FRAME), other aligned shapes the runtime-shape kernel,
    unaligned buffers the scalar shift (and, finalising, reset_finalize_kernel behind it)."""
    name, shape, pitched = case
    env, dev = _env(1003, cuda_device), cuda_device
    row_o, row_p, ld_o, ld_p = _set_shape(env, shape, pitched)
    for off in (0, 1):
        got = _kernels(lambda: _run_env_entry(lib, env, dev, shape, pitched, off, True if fused else None, seed=off))
        shifts = row_o > shape[0] or row_p > shape[2]
        if off:
            assert sum("stack_shift_scalar_kernel" in k for k in got) == (row_o > shape[0]) + (row_p > shape[2])
            assert any("reset_finalize_kernel" in k for k in got) == fused
        elif name in BUILT:
            assert len(got) == 1 and "stack_shift_kernel" in got[0]
            assert _fixed(row_o, ld_o, shape[0]).search(got[0]) and _fixed(row_p, ld_p, shape[2]).search(got[0]), got
        elif shifts or fused:
            assert len(got) == 1 and "stack_shift_kernel" in got[0] and "ShiftShape" in got[0], got
        else:
            assert got == []


@pytest.mark.parametrize("reset", [False, True], ids=["plain", "reset"])
@pytest.mark.parametrize("shape", list(SHIFT_SHAPES.values()), ids=list(SHIFT_SHAPES))
def test_stack_shift_dispatch(lib, cuda_device, shape, reset):
    dev = cuda_device
    row, frame = shape
    n = 1003
    for off in (0, 1):
        (_, prev), (_, new) = _guarded(n, row, off, dev), _guarded(n, row, off, dev)
        rb = torch.zeros(n, dtype=torch.uint8, device=dev) if reset else None
        got = _kernels(lambda: lib.hb_stack_shift(prev.data_ptr(), new.data_ptr(), rb.data_ptr() if reset else None, n, row,
                                                  frame, torch.cuda.current_stream(dev).cuda_stream))
        assert len(got) == 1, got
        if off:
            assert "stack_shift_scalar_kernel" in got[0]
        elif shape in ((615, 41), (1050, 70)) and not reset:
            assert "stack_shift_kernel" in got[0] and _fixed(615, 615, 41).search(got[0]) and _fixed(1050, 1050, 70).search(got[0])
        else:
            assert "stack_shift_kernel" in got[0] and "ShiftShape" in got[0], got


def test_stack_shift_past_32_bit_indices(lib, cuda_device):
    """A history of exactly 2^32 floats: the 32-bit index paths do not apply and the count of their blocks wraps to 0;
    the scalar shift must still run over the whole buffer."""
    from isaac_b200 import _lib
    dev = cuda_device
    n, row, frame = 1 << 22, 1 << 10, 64
    if torch.cuda.mem_get_info(dev)[0] < 3 * n * row * 4:
        pytest.skip("needs 48 GiB free")
    prev = torch.arange(row, device=dev, dtype=torch.float32).repeat(n, 1)
    prev[:, 0] = torch.arange(n, device=dev, dtype=torch.float32)
    next_ = torch.full_like(prev, FILL)
    _lib.check(lib.hb_stack_shift(prev.data_ptr(), next_.data_ptr(), None, n, row, frame,
                                  torch.cuda.current_stream(dev).cuda_stream), "hb_stack_shift")
    torch.cuda.synchronize()
    assert torch.equal(next_[:, :row - frame], prev[:, frame:row]) and (next_[:, row - frame:] == FILL).all()
