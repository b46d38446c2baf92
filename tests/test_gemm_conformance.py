"""Conformance of every built tcgen05 GEMM kernel, gemm_tf32_kernel<BN, A_MN, B_MN, EPI, PAIR, ACT>, against an exact
reference.

Exact operands.  Every operand is a small integer times a power of two ({-2..2} * 2^-3, biases {-4..4} * 2^-3, atomic
prefills {-8..8} * 2^-6; {-1, 0, 1} at the large sizes).  TF32 holds such values exactly, every product is exact, and
every partial sum is a multiple of 2^-6 far below 2^24 * 2^-6, so fp32 accumulation is exact in any order: TMEM chains,
split-K, red.global.add, and 3xTF32 (whose lo parts are zero).  The result must therefore be BIT-EQUAL to the fp64
product (computed on the device: integer-valued fp64 sums are exact whatever the order), so a layout, swizzle, tile-edge,
split or tile-list mistake fails with zero tolerance, independently of TF32 rounding and of the truncating accumulator
(DESIGN.md section 4.1).  The fused activations f / f' are evaluated in fp64 on that exact accumulator and compared within
the documented error bounds of the fp32 operations the epilogue uses (the table above act_fwd_tolerance).

Poison and sentinels.  Every float outside the logical extent of A, B and H is NaN (the columns past K or past M / N up
to the leading dimension, and extra rows past the extent), so is every float between the entries of a strided bias; D
sits between sentinel rows and its columns between N and ldd keep a sentinel.  A read outside the problem turns the
result into NaN, a write outside it changes a sentinel.

Coverage.  One case per built instantiation: `expected_instantiations()` mirrors the dispatch of mlp_gemm.cu and a CPU
test checks it against the kernels listed in libhectorb200.so (cuobjdump + cu++filt), so a kernel added later without a
case fails the suite.  Each case runs under torch.profiler and asserts that exactly its kernel ran, over shapes at the
tile edges (M in {1, 127, 128, 129, 255, 256, 257, 300+}, N on both sides of the tile width, K in {1, 3, 4, 31, 32, 33,
615, 1050}, leading dimensions above the minimum).  Then: the grouped launch's branches, the launch options (pair mode,
tile_n, gemm_tile_snake, gemm_pdl), hector's dependent layer chain eagerly and from a CUDA graph, the training-size
forward (M = 393 216) and weight gradient (K = 393 216), 3xTF32, one Gaussian-operand case per (tile width, layout) at
test_mlp_gemm.check_product's bound, and the refusals."""
import ctypes as C
import os
import re
import shutil
import subprocess
import zlib
from contextlib import contextmanager

import pytest
import torch

HB_ERR_BAD_ARG, HB_ERR_UNSUPPORTED = -1, -3
STORE, BIAS, BIAS_ACT, ACT_BWD, ATOMIC = range(5)                 # hb_gemm_epilogue
ELU, SELU, RELU, LRELU, TANH, SIGMOID = range(6)                 # hb_activation
ACT_NAMES = ("elu", "selu", "relu", "lrelu", "tanh", "sigmoid")
LAYOUTS = ((False, False), (False, True), (True, True))           # (A MN-major, B MN-major); A MN-major with B K-major is refused
EPI_NAMES = ("store", "bias", "bias_act", "act_bwd", "atomic")
GRID = 2.0 ** -3                                                  # operand grid
SENTINEL = -7.0
GUARD_ROWS = 3


# ---------------------------------------------------------------------------------------------------- the instantiations
def expected_instantiations():
    """(BN, A_MN, B_MN, EPI, PAIR, ACT) of every kernel mlp_gemm.cu builds: every epilogue with ELU in every layout at every
    width (MN-major B only at 128 and 256: it needs N > 64), pair and non-pair at 256; the other activations in their MLP
    layouts only - bias + f forward (A, B K-major), f' data gradient (B MN-major)."""
    out = set()
    for a_mn, b_mn in LAYOUTS:
        for epi in range(5):
            for bn in ((128, 256) if b_mn else (16, 64, 128, 256)):
                for pair in ((False, True) if bn == 256 else (False,)):
                    out.add((bn, a_mn, b_mn, epi, pair, ELU))
    for act in (SELU, RELU, LRELU, TANH, SIGMOID):
        for bn in (16, 64, 128, 256):
            for pair in ((False, True) if bn == 256 else (False,)):
                out.add((bn, False, False, BIAS_ACT, pair, act))
                if bn >= 128:
                    out.add((bn, False, True, ACT_BWD, pair, act))
    return out


# Built instantiations that no descriptor can reach, with the reason.  Empty: dispatch_major resolves an MN-major B at
# BN < 128 to its refusal at compile time, so those kernels are not built.
UNREACHABLE = {}

CASES = sorted(expected_instantiations())


def inst_id(inst):
    bn, a_mn, b_mn, epi, pair, act = inst
    return (f"bn{bn}{'pair' if pair else ''}-{'m' if a_mn else 'k'}{'m' if b_mn else 'k'}-{EPI_NAMES[epi]}"
            + (f"-{ACT_NAMES[act]}" if epi in (BIAS_ACT, ACT_BWD) else ""))


_TARG = re.compile(r"gemm_tf32_kernel<([^>]*)>")


def parse_kernel(name):
    """The template arguments of a demangled gemm_tf32_kernel name; both demangler spellings ((int)128 / 128,
    (bool)0 / false) are accepted.  None for other kernels."""
    m = _TARG.search(name)
    if not m:
        return None
    toks = [re.sub(r"^\((?:int|bool)\)", "", t.strip()) for t in m.group(1).split(",")]
    bn, a_mn, b_mn, epi, pair, act = [{"true": 1, "false": 0}[t] if t in ("true", "false") else int(t.rstrip("u")) for t in toks]
    return bn, bool(a_mn), bool(b_mn), epi, bool(pair), act


def _cuda_tool(name):
    from isaac_b200 import build
    for cand in (shutil.which(name), os.path.join(os.path.dirname(build._nvcc()), name)):
        if cand and os.path.exists(cand):
            return cand
    return None


def built_instantiations():
    from isaac_b200 import _lib
    dump, filt = _cuda_tool("cuobjdump"), _cuda_tool("cu++filt")
    if dump is None or filt is None:
        pytest.skip("cuobjdump / cu++filt not found next to nvcc")
    syms = subprocess.run([dump, "-symbols", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"\b_Z\w*gemm_tf32_kernel\w*", syms)))
    names = subprocess.run([filt], input="\n".join(mangled) + "\n", capture_output=True, text=True, check=True).stdout
    insts = [parse_kernel(n) for n in names.splitlines() if n.strip()]
    assert len(insts) == len(mangled) and None not in insts, names
    return insts


def test_every_built_instantiation_has_a_case(lib):
    built = built_instantiations()
    assert len(built) == len(set(built))
    missing = set(built) - set(CASES) - set(UNREACHABLE)
    assert not missing, f"built kernels without a conformance case: {sorted(missing)}"
    stale = (set(CASES) | set(UNREACHABLE)) - set(built)
    assert not stale, f"cases for kernels that are not built: {sorted(stale)}"
    assert not set(CASES) & set(UNREACHABLE)


def test_case_shapes_reach_their_instantiation():
    """The shapes of every case satisfy the dispatch rules that select its kernel (checked on the GPU by the profiler)."""
    for inst in CASES:
        bn, a_mn, b_mn, epi, pair, act = inst
        for M, N, K, ld_extra in case_shapes(inst):
            assert bn == (16 if N <= 16 else 64 if N <= 64 else 128 if N <= 128 else case_tile_n(inst))
            assert not pair or M > 128
            assert not b_mn or N > 64


# Error bounds of the fused activations (hb::act_fwd / hb::act_grad, hb_common.cuh).  The accumulator z is exact, so the
# only errors are those of the fp32 evaluation of f(z) or f'(h) * acc:
#   every fp32 +, -, *, / rounds to within 2^-24 relative (round to nearest; ulp(y) <= 2^-23 |y|), and the fp32 constants
#   (SELU's scale and alpha, LReLU's 0.01) are within 2^-24 relative of their exact values;
#   __expf(x) (the TF32-mode tail): at most 2 + floor(|1.173 x|) ulp (CUDA Math API, intrinsic functions);
#   expf 2 ulp, expm1f 1 ulp, tanhf 2 ulp (CUDA Math API, single precision; the 3xTF32 pass and tanh in both modes).
# Forward, with E = the ulp bound of the exponential and e = its exact value:
#   ELU     z > 0: exact                  z <= 0: E ulp(e) + 1 rounding of the subtraction
#   SELU    z > 0: constant + 1 rounding  z <= 0: s*a (E ulp(e) + 1 rounding) + constant product + 1 rounding
#   ReLU    exact                         LReLU   z <= 0: constant + 1 rounding
#   tanh    2 ulp                         sigmoid E ulp(e) relative through 1 + e, + 2 roundings
# f'(h) * acc: at most three roundings and one constant (f' is written in h, which is exact on the grid used here).
U = 2.0 ** -23


def _exp_ulps(x, accurate):
    """E: expf's 2 ulp, or __expf's 2 + floor(|1.173 x|) ulp."""
    return torch.full_like(x, 2.0) if accurate else 2.0 + torch.floor((1.173 * x).abs())


def act_fwd_ref(act, z):
    s, a = 1.0507009873554804934193349852946, 1.6732632423543772848170429916717
    if act == ELU:
        return torch.where(z > 0, z, torch.expm1(z))
    if act == SELU:
        return s * torch.where(z > 0, z, a * torch.expm1(z))
    if act == RELU:
        return z.clamp_min(0.0)
    if act == LRELU:
        return torch.where(z > 0, z, 0.01 * z)
    if act == TANH:
        return torch.tanh(z)
    return torch.sigmoid(z)


def act_fwd_tolerance(act, z, f, accurate):
    """Largest |kernel - f(z)| the bounds above allow (z, f in fp64)."""
    zn = torch.minimum(z, torch.zeros_like(z))
    em1 = torch.expm1(zn)                                             # exp(z) - 1 for z <= 0
    # expm1f: 1 ulp of the result; __expf(z) - 1: E ulp of exp(z), then the subtraction's rounding
    em1_tol = U * em1.abs() if accurate else _exp_ulps(zn, False) * U * torch.exp(zn) + 0.5 * U * em1.abs()
    if act == ELU:
        t = torch.where(z > 0, 0.0, em1_tol)
    elif act == SELU:
        sa = 1.0507009873554804934193349852946 * 1.6732632423543772848170429916717
        t = torch.where(z > 0, U * f.abs(), sa * em1_tol + 2 * U * f.abs())
    elif act == RELU:
        t = torch.zeros_like(z)
    elif act == LRELU:
        t = torch.where(z > 0, 0.0, U * f.abs())
    elif act == TANH:
        t = 2 * U * f.abs()
    else:
        t = f.abs() * (_exp_ulps(-z, accurate) * U + 2 * U)
    return t + 1e-37


def act_grad_ref(act, h):
    s, a = 1.0507009873554804934193349852946, 1.6732632423543772848170429916717
    if act == ELU:
        return torch.where(h > 0, 1.0, h + 1.0)
    if act == SELU:
        return torch.where(h > 0, s, h + s * a)
    if act == RELU:
        return torch.where(h > 0, 1.0, 0.0)
    if act == LRELU:
        return torch.where(h > 0, 1.0, 0.01)
    if act == TANH:
        return 1.0 - h * h
    return (1.0 - h) * h


def act_grad_tolerance(acc, g, h):
    return 2 * U * acc.abs() * (g.abs() + h.abs() + 1.0) + 1e-37


def h_values(act, shape, gen, dev):
    """Forward activations h = f(z) on a 2^-4 grid inside f's range (exact through every f' formula)."""
    k = torch.randint(-15, 16, shape, generator=gen, device=dev).double()
    if act == RELU:
        k = k.clamp_min(0)
    elif act == SIGMOID:
        k = k.abs().clamp_min(1)
    return (k / 16).float()


# ---------------------------------------------------------------------------------------------------- shapes of a case
M_EDGES = (1, 127, 128, 129, 255, 256, 257, 300)
M_PAIR = (129, 255, 256, 257, 300, 513)
K_EDGES = (1, 3, 4, 31, 32, 33, 615, 1050)
N_EDGES = {16: (1, 5, 16), 64: (17, 33, 64), 128: (65, 127, 128, 129, 257), 256: (129, 255, 256, 257, 300)}


def case_tile_n(inst):
    return inst[0] if inst[0] >= 128 else 0


def case_shapes(inst):
    """Eight (M, N, K, extra leading-dimension floats): every M edge (the pair kernels: M > 128), every K edge, the N edges
    of the tile width cycled; the leading dimensions alternate between the minimum and 4 or 8 floats more."""
    bn, a_mn, b_mn, epi, pair, act = inst
    ms, ns = (M_PAIR if pair else M_EDGES), N_EDGES[bn]
    return [(ms[i % len(ms)], ns[(i + bn) % len(ns)], K_EDGES[(3 * i + bn // 16) % len(K_EDGES)], 4 * (i % 3)) for i in range(8)]


# ---------------------------------------------------------------------------------------------------- one problem
def pad4(n):
    return (n + 3) // 4 * 4


def grid_values(shape, gen, dev, lo=-2, hi=2, scale=GRID):
    return (torch.randint(lo, hi + 1, shape, generator=gen, device=dev).double() * scale).float()


def poisoned(rows, cols, ld, dev, values):
    """[rows + 2, ld] of NaN with values in [:rows, :cols]: the columns past cols and the two rows past rows are poison."""
    t = torch.full((rows + 2, ld), float("nan"), device=dev)
    t[:rows, :cols] = values
    return t


class Problem:
    """D (+)= A[M,K] B[N,K]^T with poisoned operands, sentinel-guarded output and an fp64 reference.  Layout of memory:
    A K-major [M, lda] / MN-major [K, lda]; B K-major [N, ldb] / MN-major [K, ldb].  bias_packed: the bias is column K of
    B (K-major B, the packed [W | b | 0] matrix of an nn.Linear: bias_stride = ldb); otherwise a NaN-filled vector read
    at bias_stride 1 or 3."""

    def __init__(self, dev, gen, M, N, K, a_mn=False, b_mn=False, epi=STORE, act=ELU, ld_extra=0, split_k=1, tile_n=0,
                 bias_packed=False, bias_stride=1, precision=0, ldd=None, lo=-2, hi=2, scale=GRID):
        from isaac_b200 import _lib
        self.M, self.N, self.K, self.epi, self.act, self.precision = M, N, K, epi, act, precision
        a = grid_values((M, K), gen, dev, lo, hi, scale)
        b = grid_values((N, K), gen, dev, lo, hi, scale)
        self.a64, self.b64 = a.double(), b.double()
        if a_mn:
            self.A = poisoned(K, M, pad4(M) + ld_extra, dev, a.T)
        else:
            self.A = poisoned(M, K, pad4(K) + ld_extra, dev, a)
        kb = K + 1 if bias_packed else K
        if b_mn:
            self.B = poisoned(K, N, pad4(N) + ld_extra, dev, b.T)
        else:
            self.B = poisoned(N, kb, pad4(kb) + ld_extra, dev, torch.cat([b, torch.zeros(N, kb - K, device=dev)], 1))
        d = _lib.GemmDesc()
        d.A, d.B, d.M, d.N, d.K = self.A.data_ptr(), self.B.data_ptr(), M, N, K
        d.lda, d.ldb = self.A.stride(0), self.B.stride(0)
        d.a_mn_major, d.b_mn_major, d.epilogue, d.activation = int(a_mn), int(b_mn), epi, act
        d.split_k, d.tile_n, d.precision = split_k, tile_n, precision
        self.bias64 = None
        if epi in (BIAS, BIAS_ACT):
            bias = grid_values((N,), gen, dev, -4, 4)
            self.bias64 = bias.double()
            if bias_packed:
                assert not b_mn
                self.B[:N, K] = bias
                d.bias, d.bias_stride = self.B.data_ptr() + 4 * K, self.B.stride(0)
            else:
                self.bias_buf = torch.full((N * bias_stride + 1,), float("nan"), device=dev)
                self.bias_buf[:N * bias_stride:bias_stride] = bias
                d.bias, d.bias_stride = self.bias_buf.data_ptr(), bias_stride
        if epi == ACT_BWD:
            h = h_values(act, (M, N), gen, dev)
            self.h64 = h.double()
            self.H = poisoned(M, N, pad4(N) + ld_extra, dev, h)
            d.H, d.ldh = self.H.data_ptr(), self.H.stride(0)
        # D: sentinel rows around it, sentinel columns between N and ldd (any ldd >= N for the atomic epilogue, which does
        # not store through a tensor map; a multiple of 4 otherwise)
        self.ldd = ldd or (pad4(N) + ld_extra)
        self.Dbuf = torch.full((M + 2 * GUARD_ROWS, self.ldd), SENTINEL, device=dev)
        self.D = self.Dbuf[GUARD_ROWS:GUARD_ROWS + M]
        self.prefill = None
        if epi == ATOMIC:
            self.prefill = grid_values((M, N), gen, dev, -8, 8, 2.0 ** -6)
            self.D[:, :N] = self.prefill
        d.D, d.ldd = self.D.data_ptr(), self.ldd
        if precision:
            self.ws = torch.empty(int(_lib.load().hb_gemm_workspace_floats(C.byref(d))), device=dev)
            d.workspace, d.workspace_floats = self.ws.data_ptr(), self.ws.numel()
        self.desc = d

    def run(self, lib, st):
        from isaac_b200 import _lib
        _lib.check(lib.hb_gemm_tf32(C.byref(self.desc), st), "hb_gemm_tf32")

    def accumulator(self):
        return self.a64 @ self.b64.T

    def check(self, what=""):
        """The output against the fp64 reference (bit-equal, or within ACT bounds), and the sentinels."""
        M, N = self.M, self.N
        what = f"{what} M={M} N={N} K={self.K} epi={EPI_NAMES[self.epi]} act={ACT_NAMES[self.act]}"
        assert (self.Dbuf[:GUARD_ROWS] == SENTINEL).all() and (self.Dbuf[GUARD_ROWS + M:] == SENTINEL).all(), \
            f"{what}: store outside the output rows"
        assert (self.D[:, N:] == SENTINEL).all(), f"{what}: store into the columns between N and ldd"
        got = self.D[:, :N].double()
        acc = self.accumulator()
        if self.epi == STORE:
            want = acc
        elif self.epi == BIAS:
            want = acc + self.bias64
        elif self.epi == ATOMIC:
            want = acc + self.prefill.double()
        elif self.epi == BIAS_ACT:
            z = acc + self.bias64
            want = act_fwd_ref(self.act, z)
            tol = act_fwd_tolerance(self.act, z, want, accurate=bool(self.precision))
            err = (got - want).abs()
            assert not got.isnan().any(), f"{what}: NaN in the output (a poisoned float was read)"
            bad = err > tol
            assert not bad.any(), f"{what}: {int(bad.sum())} outputs beyond the bound, worst {float((err / tol).max()):.3g} x bound"
            return
        else:
            g = act_grad_ref(self.act, self.h64)
            want = acc * g
            tol = act_grad_tolerance(acc, g, self.h64)
            assert not got.isnan().any(), f"{what}: NaN in the output (a poisoned float was read)"
            bad = (got - want).abs() > tol
            assert not bad.any(), f"{what}: {int(bad.sum())} outputs beyond the bound"
            return
        if not torch.equal(got, want):
            bad = (got != want) | got.isnan()
            r, c = bad.nonzero()[0].tolist()
            raise AssertionError(f"{what}: {int(bad.sum())} outputs differ from the exact product, first at ({r}, {c}): "
                                 f"{float(got[r, c])} != {float(want[r, c])}")


# ---------------------------------------------------------------------------------------------------- helpers
def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def gemm_kernels(fn):
    """The gemm_tf32_kernel instantiations `fn` launched, in order."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [k for k in (parse_kernel(e.name) for e in prof.events()) if k is not None]


@contextmanager
def gemm_options(lib, pair=1, snake=1, pdl=1):
    """Launch options for the block; every one is restored to its default (1) on the way out."""
    try:
        lib.hb_gemm_set_pair_mode(pair)
        assert lib.hb_set_option(b"gemm_tile_snake", snake) == 0
        assert lib.hb_set_option(b"gemm_pdl", pdl) == 0
        yield
    finally:
        lib.hb_gemm_set_pair_mode(1)
        lib.hb_set_option(b"gemm_tile_snake", 1)
        lib.hb_set_option(b"gemm_pdl", 1)


def case_problem(dev, gen, inst, M, N, K, ld_extra, i, precision=0):
    bn, a_mn, b_mn, epi, pair, act = inst
    kw = dict(a_mn=a_mn, b_mn=b_mn, epi=epi, act=act, ld_extra=ld_extra, tile_n=case_tile_n(inst), precision=precision)
    if epi in (BIAS, BIAS_ACT):          # the packed [W | b | 0] matrix (production), a dense and a strided bias vector
        kw.update(bias_packed=(i % 3 == 0) and not b_mn, bias_stride=1 + 2 * (i % 3 == 2))
    if epi == ATOMIC:
        kw.update(split_k=(1, 2, 7, 0, 1000)[i % 5], ldd=N + i % 3)
    return Problem(dev, gen, M, N, K, **kw)


# ---------------------------------------------------------------------------------------------------- GPU: exactness sanity
@pytest.mark.gpu
@pytest.mark.parametrize("K", [8, 4096])
def test_tensor_core_accumulates_grid_operands_exactly(lib, cuda_device, K):
    """The premise of this file: with grid operands the tensor core's fp32 accumulation is exact.  K = 8 is one MMA
    instruction; K = 4096 is 512 of them in one TMEM chain (no split)."""
    gen = torch.Generator(device=cuda_device).manual_seed(K)
    p = Problem(cuda_device, gen, 256, 256, K, tile_n=256)
    p.run(lib, _stream(cuda_device))
    torch.cuda.synchronize()
    p.check("sanity")


# ---------------------------------------------------------------------------------------------------- GPU: every instantiation
@pytest.mark.gpu
@pytest.mark.parametrize("inst", CASES, ids=[inst_id(c) for c in CASES])
def test_instantiation_is_exact_at_tile_edges(lib, cuda_device, inst):
    bn, a_mn, b_mn, epi, pair, act = inst
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(zlib.crc32(inst_id(inst).encode()))
    probs = [case_problem(dev, gen, inst, M, N, K, extra, i) for i, (M, N, K, extra) in enumerate(case_shapes(inst))]
    st = _stream(dev)
    with gemm_options(lib, pair=int(pair)):
        ran = gemm_kernels(lambda: [p.run(lib, st) for p in probs])
    assert ran == [inst] * len(probs), ran
    for p in probs:
        p.check(inst_id(inst))


# ---------------------------------------------------------------------------------------------------- GPU: TF32 rounding
GAUSS_CASES = [(bn, a, b) for a, b in LAYOUTS for bn in ((128, 256) if b else (16, 64, 128, 256))]


@pytest.mark.gpu
@pytest.mark.parametrize("bn,a_mn,b_mn", GAUSS_CASES)
def test_gaussian_operands_tf32_product(lib, cuda_device, bn, a_mn, b_mn):
    """Operands that TF32 does not hold: the result is a TF32 product of them (test_mlp_gemm.check_product's bound)."""
    from test_mlp_gemm import check_product
    dev = cuda_device
    N = {16: 13, 64: 61, 128: 125, 256: 383}[bn]
    M, K = 517, 333
    gen = torch.Generator(device=dev).manual_seed(bn + 2 * a_mn + b_mn)
    epi = ATOMIC if a_mn else STORE
    p = Problem(dev, gen, M, N, K, a_mn=a_mn, b_mn=b_mn, epi=epi, tile_n=bn if bn >= 128 else 0, split_k=0 if a_mn else 1)
    a, b = torch.randn(M, K, generator=gen, device=dev), torch.randn(N, K, generator=gen, device=dev)
    (p.A[:K, :M] if a_mn else p.A[:M, :K]).copy_(a.T if a_mn else a)
    (p.B[:K, :N] if b_mn else p.B[:N, :K]).copy_(b.T if b_mn else b)
    p.D[:, :N] = 0
    ran = gemm_kernels(lambda: p.run(lib, _stream(dev)))
    assert [k[0] for k in ran] == [bn], ran
    check_product(p.D[:, :N], a, b, f"bn {bn} a_mn {a_mn} b_mn {b_mn}")
    assert (p.D[:, N:] == SENTINEL).all()


# ---------------------------------------------------------------------------------------------------- GPU: grouped launches
def _grouped_case(dev, gen, kind, shapes, tile_n=(0, 0), precision=0):
    kinds = {"fwd": dict(epi=BIAS_ACT, act=RELU, bias_packed=True), "dgrad": dict(b_mn=True, epi=ACT_BWD, act=TANH),
             "wgrad": dict(a_mn=True, b_mn=True, epi=ATOMIC, split_k=0), "store": dict(epi=STORE)}
    return [Problem(dev, gen, M, N, K, tile_n=t, precision=precision, ld_extra=4 * i, **kinds[kind])
            for i, ((M, N, K), t) in enumerate(zip(shapes, tile_n))]


# (name, kind, ((M, N, K) x 2), tile_n x 2, pair mode, expected kernels as (BN, PAIR) per launch)
GROUPED = [
    ("both_wide", "fwd", ((513, 300, 615), (300, 257, 1050)), (256, 256), 1, [(256, True)]),
    ("both_wide_dgrad", "dgrad", ((513, 300, 128), (257, 512, 256)), (256, 256), 1, [(256, True)]),
    ("both_wide_wgrad", "wgrad", ((300, 513, 2000), (257, 616, 999)), (0, 0), 1, [(256, True)]),
    ("wide_and_n128", "fwd", ((513, 300, 615), (300, 100, 33)), (256, 0), 1, [(128, False)]),
    ("narrow_and_wide", "fwd", ((300, 40, 615), (300, 300, 31)), (0, 256), 1, [(64, False), (256, True)]),
    ("two_narrow_widths", "store", ((300, 10, 615), (129, 40, 31)), (0, 0), 1, [(16, False), (64, False)]),
    ("two_narrow_same", "store", ((300, 10, 615), (129, 12, 31)), (0, 0), 1, [(16, False)]),
    ("one_m_le_128", "fwd", ((128, 300, 615), (513, 257, 100)), (256, 256), 1, [(256, False)]),
    ("pair_off", "wgrad", ((300, 513, 2000), (257, 616, 999)), (0, 0), 0, [(256, False)]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", GROUPED, ids=[g[0] for g in GROUPED])
def test_grouped_launch_branches(lib, cuda_device, case):
    """Every branch of gemm_tf32_dispatch_grouped: both outputs against the reference, one or two launches as planned."""
    name, kind, shapes, tile_n, pair, expect = case
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(len(name))
    p0, p1 = _grouped_case(dev, gen, kind, shapes, tile_n)
    from isaac_b200 import _lib
    st = _stream(dev)
    with gemm_options(lib, pair=pair):
        ran = gemm_kernels(lambda: _lib.check(lib.hb_gemm_tf32_grouped(C.byref(p0.desc), C.byref(p1.desc), st), "grouped"))
    assert [(k[0], k[4]) for k in ran] == expect, ran
    p0.check(name + " problem 0")
    p1.check(name + " problem 1")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "dgrad", "wgrad"])
def test_grouped_3xtf32_runs_two_calls(lib, cuda_device, kind):
    from isaac_b200 import _lib
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(5)
    shapes = ((513, 300, 615), (257, 129, 33)) if kind != "dgrad" else ((513, 300, 129), (257, 129, 33))
    p0, p1 = _grouped_case(dev, gen, kind, shapes, precision=1)
    st = _stream(dev)
    ran = gemm_kernels(lambda: _lib.check(lib.hb_gemm_tf32_grouped(C.byref(p0.desc), C.byref(p1.desc), st), "grouped"))
    assert len(ran) == 2 and all(k[3] == ATOMIC for k in ran), ran
    p0.check("3xtf32 grouped 0")
    p1.check("3xtf32 grouped 1")


# ---------------------------------------------------------------------------------------------------- GPU: launch options
@pytest.mark.gpu
@pytest.mark.parametrize("pdl", [0, 1])
@pytest.mark.parametrize("snake", [0, 1])
@pytest.mark.parametrize("tile_n", [128, 256])
@pytest.mark.parametrize("pair", [0, 1])
def test_launch_options(lib, cuda_device, pair, tile_n, snake, pdl):
    """M = 24 576, N = 256: several rounds of tiles over the SMs at either width, so the snake order changes who computes
    what.  Forward with bias (K-major) and split-K weight gradient (MN-major), back to back on the stream."""
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(tile_n + 2 * snake + pdl + 4 * pair)
    fwd = Problem(dev, gen, 24576, 256, 96, epi=BIAS, tile_n=tile_n, bias_packed=True)
    wgr = Problem(dev, gen, 256, 252, 24576, a_mn=True, b_mn=True, epi=ATOMIC, tile_n=tile_n, split_k=0)
    st = _stream(dev)
    with gemm_options(lib, pair=pair, snake=snake, pdl=pdl):
        ran = gemm_kernels(lambda: (fwd.run(lib, st), wgr.run(lib, st)))
    want = (tile_n, bool(pair and tile_n == 256))
    assert [(k[0], k[4]) for k in ran] == [want, want], ran
    fwd.check("options fwd")
    wgr.check("options wgrad")


# ---------------------------------------------------------------------------------------------------- GPU: 3xTF32
X3_SHAPES = [(129, 257, 33), (1, 65, 1), (300, 131, 1050), (257, 17, 615), (127, 300, 3)]
X3_EPIS = [(STORE, ELU), (BIAS, ELU), (ATOMIC, ELU)] + [(e, a) for e in (BIAS_ACT, ACT_BWD) for a in range(6)]


@pytest.mark.gpu
@pytest.mark.parametrize("epi,act", X3_EPIS, ids=[f"{EPI_NAMES[e]}-{ACT_NAMES[a]}" for e, a in X3_EPIS])
@pytest.mark.parametrize("layout", LAYOUTS, ids=["kk", "km", "mm"])
def test_3xtf32_exact(lib, cuda_device, layout, epi, act):
    """HB_GEMM_3XTF32 on grid operands (lo parts zero): exact, K and MN-major widths that are not multiples of 4 included
    (the zero padding of split3_*).  The products run on the atomic kernel of the layout and the fused tails in the
    separate libm-accurate pass, so every activation is taken in every layout."""
    a_mn, b_mn = layout
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(epi * 8 + act)
    st = _stream(dev)
    for i, (M, N, K) in enumerate(X3_SHAPES):
        if b_mn and N <= 64:
            continue
        kw = dict(a_mn=a_mn, b_mn=b_mn, epi=epi, act=act, precision=1, ld_extra=4 * (i % 2))
        if epi in (BIAS, BIAS_ACT):
            kw.update(bias_packed=not b_mn and i % 2 == 0, bias_stride=1 + 2 * (i % 2))
        if epi == ATOMIC:
            kw.update(split_k=(1, 0, 7)[i % 3])
        p = Problem(dev, gen, M, N, K, **kw)
        p.run(lib, st)
        torch.cuda.synchronize()
        p.check("3xtf32")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS, ids=["kk", "km", "mm"])
def test_3xtf32_gaussian_is_fp32_grade(lib, cuda_device, layout):
    """Operands TF32 does not hold: within test_3xtf32_is_fp32_grade's 2e-6 of |a|.|b| of the fp64 product."""
    a_mn, b_mn = layout
    dev = cuda_device
    M, N, K = 301, 259, 1031
    gen = torch.Generator(device=dev).manual_seed(17 + a_mn + b_mn)
    p = Problem(dev, gen, M, N, K, a_mn=a_mn, b_mn=b_mn, epi=ATOMIC if a_mn else STORE, precision=1)
    a, b = torch.randn(M, K, generator=gen, device=dev), torch.randn(N, K, generator=gen, device=dev)
    (p.A[:K, :M] if a_mn else p.A[:M, :K]).copy_(a.T if a_mn else a)
    (p.B[:K, :N] if b_mn else p.B[:N, :K]).copy_(b.T if b_mn else b)
    p.D[:, :N] = 0
    p.run(lib, _stream(dev))
    torch.cuda.synchronize()
    want = a.double() @ b.double().T
    err = ((p.D[:, :N].double() - want).abs() / (a.double().abs() @ b.double().abs().T).clamp_min(1e-30)).max().item()
    assert err < 2e-6, err


# ---------------------------------------------------------------------------------------------------- GPU: hector's chain
HECTOR = {"critic": (1050, 768, 256, 128), "actor": (615, 512, 256, 128)}      # input and hidden widths
CHAIN_M = 24576                                                                 # 4096 envs x 24 steps / 4 minibatches


def _pitch(n):
    return (n + 31) // 32 * 32


class HectorChain:
    """hector's actor and critic hidden layers at M = 24 576 with ReLU (exact on grid values), laid out as ActorCritic
    lays them out (packed [W | b | 0] matrices, activations with a ones column, one flat gradient buffer): forward
    L1 -> L2 -> L3, data gradient L3 -> L2 -> L1, the weight and bias gradients of all six layers, every GEMM a grouped
    launch of both networks reading what the previous one wrote.  Inputs x in {-1, 0, 1}, weights, biases and the output
    gradient in {-1, 0, 1} * 2^-4; padding is NaN."""

    def __init__(self, dev, seed):
        from isaac_b200 import _lib
        M = CHAIN_M
        g = torch.Generator(device=dev).manual_seed(seed)
        q = lambda shape, s: (torch.randint(-1, 2, shape, generator=g, device=dev).double() * s).float()
        nan = lambda r, c: torch.full((r, c), float("nan"), device=dev)
        self.grad = torch.zeros(sum(d[i + 1] * _pitch(d[i] + 1) for d in HECTOR.values() for i in range(3)), device=dev)
        self.nets, off = {}, 0
        for net, d in HECTOR.items():
            x = nan(M, _pitch(d[0] + 1))
            x[:, :d[0]], x[:, d[0]] = q((M, d[0]), 1.0), 1.0
            W, h, G = [], [], []
            for i in range(3):
                P = torch.zeros(d[i + 1], _pitch(d[i] + 1), device=dev)
                P[:, :d[i] + 1] = q((d[i + 1], d[i] + 1), 2.0 ** -4)
                W.append(P)
                hh = nan(M, _pitch(d[i + 1] + 1))
                hh[:, d[i + 1]] = 1.0
                h.append(hh)
                G.append(self.grad[off:off + d[i + 1] * _pitch(d[i] + 1)].view(d[i + 1], _pitch(d[i] + 1)))
                off += G[-1].numel()
            dout = nan(M, _pitch(d[3]))
            dout[:, :d[3]] = q((M, d[3]), 2.0 ** -4)
            dz = [torch.zeros(M, _pitch(d[i + 1]), device=dev) for i in range(2)]
            self.nets[net] = dict(x=x, W=W, h=h, G=G, dout=dout, dz=dz)
        self.steps = []                                          # (what, descriptor of each network)
        for i in range(3):
            self.steps.append((f"forward layer {i}", [dict(
                A=(n["x"] if i == 0 else n["h"][i - 1]), B=n["W"][i], D=n["h"][i], M=M, N=d[i + 1], K=d[i], epilogue=BIAS_ACT,
                activation=RELU, bias=n["W"][i].data_ptr() + 4 * d[i], bias_stride=n["W"][i].stride(0))
                for n, d in self._both()]))
        for i in (2, 1):
            self.steps.append((f"data gradient into layer {i - 1}", [dict(
                A=(n["dout"] if i == 2 else n["dz"][i]), B=n["W"][i], D=n["dz"][i - 1], M=M, N=d[i], K=d[i + 1],
                b_mn_major=1, epilogue=ACT_BWD, H=n["h"][i - 1], activation=RELU) for n, d in self._both()]))
        for i in (2, 1, 0):
            self.steps.append((f"weight gradient layer {i}", [dict(
                A=(n["dout"] if i == 2 else n["dz"][i]), B=(n["x"] if i == 0 else n["h"][i - 1]), D=n["G"][i], M=d[i + 1],
                N=d[i] + 1, K=M, a_mn_major=1, b_mn_major=1, epilogue=ATOMIC, split_k=0) for n, d in self._both()]))
        self.descs = []
        for _, kws in self.steps:
            pair = []
            for kw in kws:
                t = {k: v for k, v in kw.items() if isinstance(v, torch.Tensor)}
                dd = _lib.GemmDesc(**{k: v for k, v in kw.items() if not isinstance(v, torch.Tensor)})
                dd.A, dd.B, dd.D = t["A"].data_ptr(), t["B"].data_ptr(), t["D"].data_ptr()
                dd.lda, dd.ldb, dd.ldd = t["A"].stride(0), t["B"].stride(0), t["D"].stride(0)
                if "H" in t:
                    dd.H, dd.ldh = t["H"].data_ptr(), t["H"].stride(0)
                pair.append(dd)
            self.descs.append(pair)

    def _both(self):
        return [(self.nets[net], d) for net, d in HECTOR.items()]

    def issue(self, lib, st):
        from isaac_b200 import _lib
        for (what, _), (d0, d1) in zip(self.steps, self.descs):
            _lib.check(lib.hb_gemm_tf32_grouped(C.byref(d0), C.byref(d1), st), what)

    def reset(self):
        self.grad.zero_()
        for n, d in self._both():
            for i in range(3):
                n["h"][i][:, :d[i + 1]] = float("nan")
            for t in n["dz"]:
                t.zero_()

    def outputs(self):
        out = {"grad": self.grad.clone()}
        for net, (n, d) in zip(HECTOR, self._both()):
            for i in range(3):
                out[f"{net} h{i}"] = n["h"][i][:, :d[i + 1]].clone()
            for i in range(2):
                out[f"{net} dz{i}"] = n["dz"][i][:, :d[i + 1]].clone()
        return out

    def reference(self):
        """fp64 outputs, and for every GEMM the largest sum of |products| over the grid of its result: below 2^24, every
        fp32 partial sum of that GEMM is exact."""
        out, ratios = {"grad": torch.zeros_like(self.grad, dtype=torch.float64)}, []
        off = 0
        for net, (n, d) in zip(HECTOR, self._both()):
            a = n["x"][:, :d[0] + 1].double()                    # with the ones column
            grid = 1.0
            acts = [a]
            for i in range(3):
                P = n["W"][i][:, :d[i] + 1].double()
                grid *= 2.0 ** -4
                ratios.append(float((a.abs() @ P.abs().T).max()) / grid)
                h = (a @ P.T).clamp_min(0)
                out[f"{net} h{i}"] = h
                a = torch.cat([h, torch.ones_like(h[:, :1])], 1)
                acts.append(a)
            dcur, gd = n["dout"][:, :d[3]].double(), 2.0 ** -4
            for i in (2, 1, 0):
                inp = acts[i]                                    # [x | 1] or [h_{i-1} | 1]
                gw = gd * (1.0 if i == 0 else 2.0 ** (-4 * i))
                ratios.append(float((dcur.abs().T @ inp.abs()).max()) / gw)
                G = out["grad"][off + sum(d[j + 1] * _pitch(d[j] + 1) for j in range(i)):][:d[i + 1] * _pitch(d[i] + 1)]
                G.view(d[i + 1], _pitch(d[i] + 1))[:, :d[i] + 1] = dcur.T @ inp
                if i > 0:
                    W = n["W"][i][:, :d[i]].double()
                    gd *= 2.0 ** -4
                    ratios.append(float((dcur.abs() @ W.abs()).max()) / gd)
                    dcur = (dcur @ W) * (out[f"{net} h{i - 1}"] > 0)
                    out[f"{net} dz{i - 1}"] = dcur
            off += sum(d[j + 1] * _pitch(d[j] + 1) for j in range(3))
        return out, max(ratios)


@pytest.mark.gpu
def test_hector_chain_eager_and_graph_replay(lib, cuda_device):
    """The dependent chain overlaps every GEMM's set-up with its predecessor (programmatic dependent launch: each GEMM
    triggers its dependents at entry and waits before reading).  The eager run equals the fp64 reference exactly, and the
    replay of the captured graph equals it too."""
    from isaac_b200 import _lib
    dev = cuda_device
    chain = HectorChain(dev, seed=2024)
    want, ratio = chain.reference()
    assert ratio < 2.0 ** 24, f"test data: some fp32 partial sums would round ({ratio:.3g})"
    st = _stream(dev)
    chain.reset()
    chain.issue(lib, st)
    torch.cuda.synchronize()
    for k, v in chain.outputs().items():
        assert torch.equal(v.double(), want[k]), f"eager chain: {k}"
    graph = _lib.LaunchGraph(dev).record(lambda s: chain.issue(lib, s))
    chain.reset()
    torch.cuda.synchronize()
    graph.replay(st)
    torch.cuda.synchronize()
    for k, v in chain.outputs().items():
        assert torch.equal(v.double(), want[k]), f"graph replay: {k}"


# ---------------------------------------------------------------------------------------------------- GPU: training size
@pytest.mark.gpu
def test_training_size_layer1(lib, cuda_device):
    """The benchmark's minibatch: 65 536 envs x 24 steps / 4 = 393 216 rows.  hector's actor layer 1 forward (bias + ELU
    from the packed matrix) at M = 393 216, and its weight gradient with K = 393 216 and automatic split-K; operands in
    {-1, 0, 1} (every sum below 2^19), fp64 reference in row chunks."""
    dev = cuda_device
    M, N, K = 393216, 512, 615
    if torch.cuda.mem_get_info(dev)[0] < 16 << 30:
        pytest.skip("needs 16 GiB free")
    gen = torch.Generator(device=dev).manual_seed(393216)
    st = _stream(dev)
    fwd = Problem(dev, gen, M, N, K, epi=BIAS_ACT, act=ELU, bias_packed=True, lo=-1, hi=1, scale=1.0, ld_extra=24)
    ran = gemm_kernels(lambda: fwd.run(lib, st))
    assert len(ran) == 1 and ran[0][3] == BIAS_ACT, ran
    got = fwd.D[:, :N]
    for r in range(0, M, 32768):
        z = fwd.a64[r:r + 32768] @ fwd.b64.T + fwd.bias64
        want = act_fwd_ref(ELU, z)
        tol = act_fwd_tolerance(ELU, z, want, accurate=False)
        assert ((got[r:r + 32768].double() - want).abs() <= tol).all(), f"forward rows {r}.."
    assert (fwd.Dbuf[:GUARD_ROWS] == SENTINEL).all() and (fwd.Dbuf[GUARD_ROWS + M:] == SENTINEL).all()
    del fwd, got
    wgr = Problem(dev, gen, N, K + 1, M, a_mn=True, b_mn=True, epi=ATOMIC, split_k=0, lo=-1, hi=1, scale=1.0)
    ran = gemm_kernels(lambda: wgr.run(lib, st))
    assert len(ran) == 1 and ran[0][3] == ATOMIC, ran
    acc = torch.zeros(N, K + 1, dtype=torch.float64, device=dev)
    for r in range(0, M, 32768):
        acc += wgr.a64[:, r:r + 32768] @ wgr.b64[:, r:r + 32768].T
    assert torch.equal(wgr.D[:, :K + 1].double(), acc + wgr.prefill.double()), "weight gradient"
    assert (wgr.D[:, K + 1:] == SENTINEL).all()


# ---------------------------------------------------------------------------------------------------- refusals
def _fake_desc(**kw):
    from isaac_b200 import _lib
    fake = 1 << 20          # 16-byte aligned, never dereferenced: refused before any launch
    d = _lib.GemmDesc(A=fake, B=fake, D=fake, M=256, N=128, K=64, lda=64, ldb=128, ldd=128)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


@pytest.mark.parametrize("kw,rc,msg", [
    (dict(a_mn_major=1, b_mn_major=0), HB_ERR_UNSUPPORTED, b"A MN-major with B K-major"),
    (dict(a_mn_major=1, b_mn_major=0, epilogue=ATOMIC), HB_ERR_UNSUPPORTED, b"A MN-major with B K-major"),
    (dict(b_mn_major=1, N=64), HB_ERR_BAD_ARG, b"N > 64"),
    (dict(b_mn_major=1, a_mn_major=1, N=16, epilogue=ATOMIC), HB_ERR_BAD_ARG, b"N > 64"),
    (dict(split_k=2), HB_ERR_BAD_ARG, b"split-K needs the atomic epilogue"),
    (dict(split_k=4, epilogue=BIAS, bias=1 << 20, bias_stride=1), HB_ERR_BAD_ARG, b"split-K needs the atomic epilogue"),
], ids=["a_mn_b_k", "a_mn_b_k_atomic", "b_mn_n64", "b_mn_n16", "split_store", "split_bias"])
def test_descriptor_refusals(lib, kw, rc, msg):
    """Refused with a status and a message before anything touches the device."""
    assert lib.hb_gemm_tf32(C.byref(_fake_desc(**kw)), None) == rc
    assert msg in lib.hb_last_error(), lib.hb_last_error()
    assert lib.hb_gemm_tf32_grouped(C.byref(_fake_desc(**kw)), C.byref(_fake_desc(**kw)), None) == rc


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["lda", "ldb", "ldd", "ldh", "A", "B", "D", "H"])
def test_tma_operand_refusals(lib, cuda_device, what):
    """A leading dimension that is not a multiple of 4 floats, or a base that is not 16-byte aligned, on any operand the
    TMA moves: HB_ERR_BAD_ARG with a message, and D untouched."""
    dev = cuda_device
    gen = torch.Generator(device=dev).manual_seed(1)
    p = Problem(dev, gen, 200, 130, 40, b_mn=True, epi=ACT_BWD)
    d = p.desc
    if what.startswith("ld"):
        setattr(d, what, getattr(d, what) - 1)
    else:
        setattr(d, what, getattr(d, what) + 4)
    before = p.Dbuf.clone()
    assert lib.hb_gemm_tf32(C.byref(d), _stream(dev)) == HB_ERR_BAD_ARG
    assert b"16-byte aligned base" in lib.hb_last_error()
    torch.cuda.synchronize()
    assert torch.equal(p.Dbuf, before)
