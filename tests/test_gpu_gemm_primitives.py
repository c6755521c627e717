"""The small primitives every gradient of a mixed-precision training step passes through, called directly and compared
with float64 references computed from the exact values each kernel was given:
  dab_gemm_bf16 / dab_linear_bf16 (K-major tcgen05 GEMM, every epilogue), dab_gemm_bf16_tn / _acc (MN-major split-K
  weight-gradient GEMM), dab_colsum_f32 / dab_bias_grad (column sums, ReLU mask, bf16 copy), dab_cast_f32_to_bf16,
  dab_sum_bf16, dab_relu_bwd_colsum, dab_pair_zero_masked;
and the to_out gradients of the bf16 IPA training layer, which are plain products and sums of what the layer holds.

Most operands are small integers (bf16 values in {-2, ..., 2}): every product and partial sum is then exact in fp32, so
the result cannot depend on the summation order, the split over K or the tensor core's internal accumulation, and the
tests require equality - one lost element, row, column, K step or split fails.  One random-normal case per kernel bounds
the error per element by 2^-16 (|A|^T |B|)_ij: far above fp32 accumulation noise, far below one missing 16-wide K step."""
import ctypes

import pytest
import torch

from diffab_pytorch_b200 import _lib
from diffab_pytorch_b200._lib import ptr

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF, F32, F64 = torch.bfloat16, torch.float32, torch.float64
NAN = float("nan")
N_SM = 148          # the launchers size their grid caps from the B200's SM count


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _ints(shape, seed, lo=-2, hi=2, dtype=BF):
    return torch.randint(lo, hi + 1, shape, device=DEV, generator=_gen(seed), dtype=dtype)


def _normal(shape, seed, dtype=BF):
    return torch.randn(shape, device=DEV, generator=_gen(seed)).to(dtype)


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _bf16_from_bits(bits):
    return torch.tensor([b - 0x10000 if b >= 0x8000 else b for b in bits], dtype=torch.int16, device=DEV).view(BF)


def _f32_from_bits(bits):
    return torch.tensor([b - 0x100000000 if b >= 0x80000000 else b for b in bits], dtype=torch.int32, device=DEV).view(F32)


# ReLU outputs for the mask operand: +-0, +- the smallest and the largest subnormal, +- the smallest normal, +-1,
# +- the largest finite value, +-inf.  `y > 0` keeps exactly the positive ones.
_RELU_OUT_BITS = [0x0000, 0x8000, 0x0001, 0x8001, 0x007F, 0x807F, 0x0080, 0x8080, 0x3F80, 0xBF80, 0x7F7F, 0xFF7F,
                  0x7F80, 0xFF80]


def _relu_outputs(shape, seed):
    table = _bf16_from_bits(_RELU_OUT_BITS)
    return table[torch.randint(0, table.numel(), shape, device=DEV, generator=_gen(seed), dtype=torch.int32)]


def _within_product_bound(got, ref, bound):
    err = (got.double() - ref).abs()
    worst = float((err / bound.clamp_min(1e-300)).max())
    assert bool((err <= 2.0 ** -16 * bound).all()), f"error {worst:.3g} x (|A|^T|B|) > 2^-16"


# ---------------------------------------------------------------- K-major GEMM: C = A W^T (+ bias) (ReLU), fp32 or bf16


def _gemm(A, W, bias=None):
    M, K = A.shape
    N = W.shape[0]
    C = torch.full((M, N), NAN, device=DEV)
    _lib.check(_lib.lib().dab_gemm_bf16(ptr(A), ptr(W), ptr(C), ptr(bias), M, N, K, _lib.stream_ptr()), "dab_gemm_bf16")
    return C


def _linear(A, W, bias, relu, out_dtype):
    M, K = A.shape
    N = W.shape[0]
    C = torch.full((M, N), NAN, device=DEV, dtype=out_dtype)
    f32 = out_dtype == F32
    _lib.check(_lib.lib().dab_linear_bf16(ptr(A), ptr(W), ptr(bias), int(relu), M, N, K, ptr(C) if f32 else None,
                                          None if f32 else ptr(C), _lib.stream_ptr()), "dab_linear_bf16")
    return C


# N tiles of 32 (fewer than 148 64-wide tiles: one tile per CTA), of 64 (N % 128 != 0: 600 tiles, four or five per CTA)
# and of 128 (at least 296 128-wide tiles: 2400, sixteen or seventeen per CTA - both TMEM accumulators, many phase wraps)
KMAJOR_SHAPES = [(1024, 128), (128 * 200, 192), (128 * 300, 1024)]


@pytest.mark.parametrize("K", [64, 1344])           # one K chunk; 21 chunks, more than the 6- and 8-slot rings
@pytest.mark.parametrize("M,N", KMAJOR_SHAPES)
def test_kmajor_gemm_every_epilogue_is_exact_on_integers(M, N, K):
    A = _ints((M, K), seed=M + K)
    W = _ints((N, K), seed=N + K + 1)
    bias = _ints((N,), seed=N + 2, lo=-8, hi=8, dtype=F32)
    prod = A.double() @ W.double().t()
    for with_bias in (False, True):
        b = bias if with_bias else None
        ref = prod + bias.double() if with_bias else prod
        assert torch.equal(_gemm(A, W, b).double(), ref), f"dab_gemm_bf16 bias={with_bias}"
        for relu in (False, True):
            want = ref.clamp_min(0) if relu else ref
            got = _linear(A, W, b, relu, F32)
            assert torch.equal(got.double(), want), f"dab_linear_bf16 fp32 bias={with_bias} relu={relu}"
            # the sums are exact, so the kernel rounds to bf16 the same value torch rounds
            got = _linear(A, W, b, relu, BF)
            assert torch.equal(_bits(got), _bits(want.float().bfloat16())), f"dab_linear_bf16 bf16 bias={with_bias} relu={relu}"


@pytest.mark.parametrize("M,N", KMAJOR_SHAPES)
def test_kmajor_gemm_random_normal_within_accumulation_bound(M, N):
    K = 1344
    A, W = _normal((M, K), seed=M), _normal((N, K), seed=N + 7)
    Ad, Wd = A.double(), W.double()
    got = _gemm(A, W)
    _within_product_bound(got, Ad @ Wd.t(), Ad.abs() @ Wd.abs().t())


@pytest.mark.parametrize("M,N,K", [(100, 128, 64), (128, 96, 64), (128, 128, 96)])
def test_kmajor_gemm_rejects_unsupported_shapes(M, N, K):
    # buffers of whole 128 x 128 tiles: even a launch that slipped past the check would stay inside them
    Mp = 128 * ((M + 127) // 128)
    A = torch.zeros(Mp, 128, device=DEV, dtype=BF)
    W = torch.zeros(128, 128, device=DEV, dtype=BF)
    C = torch.zeros(Mp, 128, device=DEV)
    msg = rf"gemm_bf16: M % 128, N % \d+, K % 64 required \(M={M} N={N} K={K}\)"
    lib = _lib.lib()
    with pytest.raises(RuntimeError, match=msg):
        _lib.check(lib.dab_gemm_bf16(ptr(A), ptr(W), ptr(C), None, M, N, K, _lib.stream_ptr()), "dab_gemm_bf16")
    with pytest.raises(RuntimeError, match=msg):
        _lib.check(lib.dab_linear_bf16(ptr(A), ptr(W), None, 0, M, N, K, ptr(C), None, _lib.stream_ptr()), "dab_linear_bf16")
    torch.cuda.synchronize()
    assert not C.any()


def test_linear_needs_exactly_one_output():
    A = torch.zeros(128, 64, device=DEV, dtype=BF)
    W = torch.zeros(64, 64, device=DEV, dtype=BF)
    C = torch.zeros(128, 64, device=DEV)
    C16 = torch.zeros(128, 64, device=DEV, dtype=BF)
    lib = _lib.lib()
    for c32, c16 in ((ptr(C), ptr(C16)), (None, None)):
        with pytest.raises(RuntimeError, match=r"exactly one of C_f32 / C_bf16 must be given"):
            _lib.check(lib.dab_linear_bf16(ptr(A), ptr(W), None, 0, 128, 64, 64, c32, c16, _lib.stream_ptr()),
                       "dab_linear_bf16")


# ---------------------------------------------------------------- MN-major split-K GEMM: C = A[K, M]^T B[K, N]


def _tn(A, lda, Bm, ldb, c_addr, ldc, M, N, K, acc=False):
    lib = _lib.lib()
    name = "dab_gemm_bf16_tn_acc" if acc else "dab_gemm_bf16_tn"
    _lib.check(getattr(lib, name)(ptr(A), lda, ptr(Bm), ldb, ctypes.c_void_p(c_addr), ldc, M, N, K, _lib.stream_ptr()),
               name)


# M: inside one tile, one whole tile, a partial last tile, the IPA dWcat shape.  N: the 64-wide path, N % 128 != 0
# (64-wide), the 128-wide path.  K: one chunk, fewer than four chunks (a single split), 130 chunks (uneven last split
# for some tile counts), 512 chunks (up to 128 splits of four chunks: the pair-MLP shape).
@pytest.mark.parametrize("K", [64, 192, 64 * 130, 32768])
@pytest.mark.parametrize("N", [64, 192, 1024])
@pytest.mark.parametrize("M", [32, 64, 200, 1344])
def test_weight_gradient_gemm_is_exact_on_integers(M, N, K):
    A = _ints((K, M), seed=M + N + K)
    Bm = _ints((K, N), seed=M + N + K + 1)
    ref = A.double().t() @ Bm.double()
    C = torch.full((M, N), NAN, device=DEV)
    _tn(A, M, Bm, N, C.data_ptr(), N, M, N, K)
    assert torch.equal(C.double(), ref)
    pre = _ints((M, N), seed=K, lo=-1000, hi=1000, dtype=F32)
    C.copy_(pre)
    _tn(A, M, Bm, N, C.data_ptr(), N, M, N, K, acc=True)          # adds onto what C holds
    _tn(A, M, Bm, N, C.data_ptr(), N, M, N, K, acc=True)
    assert torch.equal(C.double(), pre.double() + 2 * ref)


@pytest.mark.parametrize("M,N,K", [(200, 192, 64 * 130), (36, 64, 192), (1344, 1024, 640)])
def test_weight_gradient_gemm_with_padded_strides(M, N, K):
    """lda > M, ldb > N, ldc > N (and an M that is no multiple of 8): the padding of A and B is never read, the padding
    columns of C are never written."""
    lda, ldb, ldc = (M + 7) // 8 * 8 + 24, N + 40, N + 20
    Af = _ints((K, lda), seed=M, lo=50, hi=60)          # padding: large values that would show in any sum
    Bf = _ints((K, ldb), seed=N, lo=50, hi=60)
    Af[:, :M] = _ints((K, M), seed=M + 1)
    Bf[:, :N] = _ints((K, N), seed=N + 1)
    ref = Af[:, :M].double().t() @ Bf[:, :N].double()
    Cf = torch.full((M, ldc), -3.5, device=DEV)
    _tn(Af, lda, Bf, ldb, Cf.data_ptr(), ldc, M, N, K)
    assert torch.equal(Cf[:, :N].double(), ref)
    assert bool((Cf[:, N:] == -3.5).all()), "dab_gemm_bf16_tn wrote the padding columns of C"
    _tn(Af, lda, Bf, ldb, Cf.data_ptr(), ldc, M, N, K, acc=True)
    assert torch.equal(Cf[:, :N].double(), 2 * ref)
    assert bool((Cf[:, N:] == -3.5).all()), "dab_gemm_bf16_tn_acc wrote the padding columns of C"


def test_weight_gradient_gemm_writes_only_its_block_of_c():
    """C is the column block base[:M, c0:c0 + N] of a wider matrix: nothing outside it may change.  The buffer has one
    row more than the block, so that a clear of M * ldc floats from C (c0 floats past row M - 1) still lands in memory
    this test owns."""
    M, N, K, c0 = 200, 192, 64 * 130, 12
    ldc = c0 + N + 20
    A, Bm = _ints((K, M), seed=1), _ints((K, N), seed=2)
    ref = A.double().t() @ Bm.double()
    base = torch.full((M + 1, ldc), 777.0, device=DEV)
    outside = torch.ones(M + 1, ldc, device=DEV, dtype=torch.bool)
    outside[:M, c0:c0 + N] = False
    for acc, mult in ((False, 1), (True, 2)):
        _tn(A, M, Bm, N, base.data_ptr() + 4 * c0, ldc, M, N, K, acc=acc)
        assert bool((base[outside] == 777.0).all()), f"{'dab_gemm_bf16_tn_acc' if acc else 'dab_gemm_bf16_tn'} " \
                                                     f"changed {int((base[outside] != 777.0).sum())} elements outside C"
        assert torch.equal(base[:M, c0:c0 + N].double(), mult * ref)


def test_weight_gradient_gemm_random_normal_within_accumulation_bound():
    M, N, K = 200, 192, 64 * 130
    A, Bm = _normal((K, M), seed=3), _normal((K, N), seed=4)
    C = torch.full((M, N), NAN, device=DEV)
    _tn(A, M, Bm, N, C.data_ptr(), N, M, N, K)
    Ad, Bd = A.double(), Bm.double()
    _within_product_bound(C, Ad.t() @ Bd, Ad.abs().t() @ Bd.abs())


@pytest.mark.parametrize("M,N,K,lda,ldb,ldc", [
    (64, 64, 96, 64, 64, 64),         # K % 64
    (64, 96, 64, 64, 96, 96),         # N % 64
    (64, 64, 64, 68, 64, 64),         # lda % 8
    (64, 64, 64, 64, 68, 64),         # ldb % 8
    (64, 64, 64, 64, 64, 66),         # ldc % 4
    (64, 64, 64, 56, 64, 64),         # lda < M
    (64, 64, 64, 64, 56, 64),         # ldb < N
    (64, 128, 64, 64, 128, 64),       # ldc < N
    (0, 64, 64, 64, 64, 64),          # M = 0
])
def test_weight_gradient_gemm_rejects_unsupported_arguments(M, N, K, lda, ldb, ldc):
    A = torch.zeros(128, 128, device=DEV, dtype=BF)      # large enough for every case even if a check slipped
    Bm = torch.zeros(128, 128, device=DEV, dtype=BF)
    C = torch.full((256, 128), 5.0, device=DEV)
    for acc in (False, True):
        name = "dab_gemm_bf16_tn_acc" if acc else "dab_gemm_bf16_tn"
        with pytest.raises(RuntimeError, match=rf"{name}: K % 64, N % 64, lda/ldb % 8, ldc % 4 required \(M={M} N={N} K={K}\)"):
            _tn(A, lda, Bm, ldb, C.data_ptr(), ldc, M, N, K, acc=acc)
    torch.cuda.synchronize()
    assert bool((C == 5.0).all())


# ---------------------------------------------------------------- column sums: dab_colsum_f32, dab_bias_grad

COLS = [4, 12, 64, 128, 1000, 1024]      # float4 lanes 1, 3, 16, 32, 250, 256: dividing 256 or not, one or many row groups
# 2^20 + 7 rows reach the 592-block cap of dab_colsum_f32 at every width (8191 rows from 128 columns up) and 8191 rows
# the 148-block cap of dab_bias_grad: the blocks then walk the rows with the grid stride
ROWS = [0, 1, 33, 8191, (1 << 20) + 7]


@pytest.mark.parametrize("rows", ROWS)
@pytest.mark.parametrize("cols", COLS)
def test_column_sums_are_exact_on_integers(cols, rows):
    lib = _lib.lib()
    st = _lib.stream_ptr()
    R = max(rows, 1)                             # rows = 0: real buffers, none of which may be read or written
    x = _ints((R, cols), seed=cols + rows, dtype=F32)
    y = _relu_outputs((R, cols), seed=cols + rows + 1)
    xs, ys = x[:rows], y[:rows]
    keep = ys > 0
    masked = torch.where(keep, xs, 0.0)
    want = {False: xs.sum(0, dtype=F64), True: masked.sum(0, dtype=F64)}
    want_bf = {False: _bits(xs.bfloat16()), True: _bits(masked.bfloat16())}

    for with_copy in (False, True):
        out = torch.full((cols,), NAN, device=DEV)
        xb = torch.full((R, cols), NAN, device=DEV, dtype=BF)
        _lib.check(lib.dab_colsum_f32(ptr(x), rows, cols, ptr(out), ptr(xb) if with_copy else None, st), "dab_colsum_f32")
        assert torch.equal(out.double(), want[False]), f"dab_colsum_f32 copy={with_copy}"
        if with_copy:
            assert torch.equal(_bits(xb[:rows]), want_bf[False])
        assert bool(xb[rows if with_copy else 0:].isnan().all())

    g_bf = x.bfloat16()                          # integers: exact in bf16
    for g_is_bf16 in ((0, 1) if cols % 8 == 0 else (0,)):
        g = g_bf if g_is_bf16 else x
        for mask in (False, True):
            db = torch.full((cols,), NAN, device=DEV)
            gb = torch.full((R, cols), NAN, device=DEV, dtype=BF)
            _lib.check(lib.dab_bias_grad(ptr(g), g_is_bf16, ptr(y) if mask else None, rows, cols, ptr(db), ptr(gb), st),
                       "dab_bias_grad")
            what = f"dab_bias_grad bf16={g_is_bf16} mask={mask}"
            assert torch.equal(db.double(), want[mask]), what
            assert torch.equal(_bits(gb[:rows]), want_bf[mask]), what
            assert bool(gb[rows:].isnan().all()), what


def test_bias_grad_rejects_bf16_rows_of_odd_quads():
    g = torch.zeros(4, 12, device=DEV, dtype=BF)
    db = torch.full((12,), 5.0, device=DEV)
    with pytest.raises(RuntimeError, match=r"dab_bias_grad: bad argument"):
        _lib.check(_lib.lib().dab_bias_grad(ptr(g), 1, None, 4, 12, ptr(db), None, _lib.stream_ptr()), "dab_bias_grad")
    torch.cuda.synchronize()
    assert bool((db == 5.0).all())


@pytest.mark.parametrize("cols", [12, 1000])
def test_column_sums_random_normal(cols):
    """Random fp32 gradients: the sums within 2^-16 of the sum of magnitudes, and the bf16 copy of the masked gradient
    (round to nearest even) equal to torch's rounding bit for bit."""
    rows = (1 << 20) + 7
    lib = _lib.lib()
    st = _lib.stream_ptr()
    g = _normal((rows, cols), seed=cols, dtype=F32)
    y = _relu_outputs((rows, cols), seed=cols + 1)
    masked = torch.where(y > 0, g, 0.0)
    out = torch.empty(cols, device=DEV)
    gb = torch.empty(rows, cols, device=DEV, dtype=BF)
    _lib.check(lib.dab_colsum_f32(ptr(g), rows, cols, ptr(out), ptr(gb), st), "dab_colsum_f32")
    _within_product_bound(out, g.sum(0, dtype=F64), g.abs().sum(0, dtype=F64))
    assert torch.equal(_bits(gb), _bits(g.bfloat16()))
    _lib.check(lib.dab_bias_grad(ptr(g), 0, ptr(y), rows, cols, ptr(out), ptr(gb), st), "dab_bias_grad")
    _within_product_bound(out, masked.sum(0, dtype=F64), masked.abs().sum(0, dtype=F64))
    assert torch.equal(_bits(gb), _bits(masked.bfloat16()))


# ---------------------------------------------------------------- dab_cast_f32_to_bf16

# fp32 bit patterns and their bf16 under round-to-nearest-even: ties to even (up and down), ties and near-ties at the
# top of the range (to +-inf or to the largest finite value), +-0, subnormals (ties included), +-inf
_CAST_CASES = [
    (0x3F808000, 0x3F80), (0x3F818000, 0x3F82), (0xBF808000, 0xBF80), (0xBF818000, 0xBF82), (0x3F808001, 0x3F81),
    (0x7F7FFFFF, 0x7F80), (0xFF7FFFFF, 0xFF80), (0x7F7F8000, 0x7F80), (0x7F7F7FFF, 0x7F7F), (0x7F7EFFFF, 0x7F7F),
    (0x00000000, 0x0000), (0x80000000, 0x8000), (0x00000001, 0x0000), (0x80000001, 0x8000), (0x00008000, 0x0000),
    (0x00018000, 0x0002), (0x80018000, 0x8002), (0x007FFFFF, 0x0080), (0x807FFFFF, 0x8080), (0x00400000, 0x0040),
    (0x7F800000, 0x7F80), (0xFF800000, 0xFF80),
]
_NAN_BITS = [0x7FC00000, 0xFFC00001, 0x7F800001, 0xFF800100]


def _cast(x, n):
    out = torch.full((n + 16,), NAN, device=DEV, dtype=BF)    # the 16 elements after n must stay untouched
    guard = _bits(out[n:]).clone()
    _lib.check(_lib.lib().dab_cast_f32_to_bf16(ptr(x), ptr(out), n, _lib.stream_ptr()), "dab_cast_f32_to_bf16")
    assert torch.equal(_bits(out[n:]), guard), "dab_cast_f32_to_bf16 wrote past n"
    return out[:n]


def test_cast_rounds_to_nearest_even_at_every_edge():
    x = _f32_from_bits([a for a, _ in _CAST_CASES] + _NAN_BITS)
    got = _cast(x, x.numel())
    want = _bf16_from_bits([b for _, b in _CAST_CASES])
    k = len(_CAST_CASES)
    assert torch.equal(_bits(got[:k]), _bits(want))
    assert torch.equal(_bits(x[:k].bfloat16()), _bits(want))         # the reference below rounds the same way
    assert bool(got[k:].isnan().all())


# the launch is capped at 148 * 16 blocks of 256 threads, eight elements each; the last n has a tail of 3 beyond the cap
@pytest.mark.parametrize("n", [1, 7, 8, 9, 2047, N_SM * 16 * 256 * 8 + 8 * 37 + 3])
def test_cast_matches_torch_bitwise(n):
    # random bit patterns cover every exponent (subnormals, inf and NaN included) and about one tie per 2^16 values
    x = (torch.randint(0, 1 << 32, (n,), device=DEV, generator=_gen(n), dtype=torch.int64) - (1 << 31)).to(torch.int32)
    x = x.view(F32)
    special = _f32_from_bits([a for a, _ in _CAST_CASES])
    k = min(n, special.numel())
    x[:k] = special[:k]
    x[n - k:] = special[special.numel() - k:]
    got = _cast(x, n)
    nan = x.isnan()
    assert bool(got[nan].isnan().all())                  # CUDA's canonical NaN bits differ from torch's
    assert torch.equal(_bits(got[~nan]), _bits(x[~nan].bfloat16()))


# ---------------------------------------------------------------- dab_sum_bf16

# grid capped at 148 * 16 blocks of 256 threads, eight elements each: the last n walks the grid stride
@pytest.mark.parametrize("n", [8, 8 * 1001, 8 * (N_SM * 16 * 256 + 5)])
def test_sum_bf16_is_the_rounded_exact_sum(n):
    """Integers in [-100, 100]: exact in bf16, their sums exact in fp32; sums beyond 256 round (to nearest even)."""
    srcs = [_ints((n,), seed=n + k, lo=-100, hi=100) for k in range(8)]
    lib = _lib.lib()
    for n_src in range(1, 9):
        want = _bits(torch.stack(srcs[:n_src]).double().sum(0).float().bfloat16())
        out = torch.full((n + 16,), NAN, device=DEV, dtype=BF)
        ptrs = (ctypes.c_void_p * n_src)(*(s.data_ptr() for s in srcs[:n_src]))
        _lib.check(lib.dab_sum_bf16(ptrs, n_src, n, ptr(out), _lib.stream_ptr()), "dab_sum_bf16")
        assert torch.equal(_bits(out[:n]), want), f"n_src={n_src}"
        assert bool(out[n:].isnan().all())
        # the output may be one of the sources (the running total of _PairFanOut is the first)
        for k in (sorted({0, n_src - 1}) if n_src > 1 else ()):
            part = [s.clone() for s in srcs[:n_src]]
            ptrs = (ctypes.c_void_p * n_src)(*(s.data_ptr() for s in part))
            _lib.check(lib.dab_sum_bf16(ptrs, n_src, n, ptr(part[k]), _lib.stream_ptr()), "dab_sum_bf16")
            assert torch.equal(_bits(part[k]), want), f"n_src={n_src}, out = source {k}"


# ---------------------------------------------------------------- dab_relu_bwd_colsum

# rows of 64 channels; the grid is capped at 148 * 8 blocks of 256 16-byte chunks = 37,888 rows
@pytest.mark.parametrize("in_place", [False, True])
@pytest.mark.parametrize("n", [1, 33, N_SM * 8 * 256 // 8 + 5, 100003])
def test_relu_bwd_colsum_accumulates_exactly(n, in_place):
    g = _ints((n, 64), seed=n, lo=-8, hi=8)
    y = _relu_outputs((n, 64), seed=n + 1)
    pre = _ints((64,), seed=n + 2, lo=-1000, hi=1000, dtype=F32)
    want_g = torch.where(y > 0, g, torch.zeros((), device=DEV, dtype=BF))
    want_sum = pre.double() + want_g.sum(0, dtype=F64)
    colsum = pre.clone()
    out = g if in_place else torch.full_like(g, NAN)
    _lib.check(_lib.lib().dab_relu_bwd_colsum(ptr(g), ptr(y), n, ptr(out), ptr(colsum), _lib.stream_ptr()),
               "dab_relu_bwd_colsum")
    assert torch.equal(_bits(out), _bits(want_g))
    assert torch.equal(colsum.double(), want_sum)


# ---------------------------------------------------------------- dab_pair_zero_masked


@pytest.mark.parametrize("L", [20, 100, 128, 256])
def test_pair_zero_masked_matches_masked_fill_bitwise(L):
    B = 3
    # random bf16 bit patterns: NaN payloads of every kind sit in rows that must come back untouched
    bits = (torch.randint(0, 1 << 16, (B, L, L, 64), device=DEV, generator=_gen(L), dtype=torch.int32)
            - (1 << 15)).to(torch.int16)
    m = torch.ones(B, L, device=DEV, dtype=torch.uint8)
    m[0, 0] = 0                       # first residue
    m[1, L - 1] = 0                   # last residue
    m[2, L // 2] = 0                  # an interior one
    m[2, 3] = 0
    pm = (m[:, :, None] & m[:, None, :]).bool()
    want = bits.masked_fill(~pm[..., None], 0)
    assert bool(bits.view(BF)[pm].isnan().any())
    x = bits.clone()
    _lib.check(_lib.lib().dab_pair_zero_masked(ptr(x), ptr(m), B, L, _lib.stream_ptr()), "dab_pair_zero_masked")
    assert torch.equal(x, want)


# ---------------------------------------------------------------- the to_out gradients of the bf16 IPA training layer


@pytest.mark.parametrize("B", [3, 65])
def test_ipa_layer_output_projection_gradients_are_exact_products(B):
    """_IpaFastFunction.backward: d b_out is the column sum of dy (dab_colsum_f32 on a side stream) and d W_out is
    bf16(dy)^T cat (dy rounded by dab_cast_f32_to_bf16 on the main stream, then dab_gemm_bf16_tn_acc on the other side
    stream into a buffer filled there, joined back into the main stream) - plain sums of values the layer holds, checked
    against fp64 on the same values.
    B = 65: K = 8320 residues, 130 chunks in 19 splits, the last one shorter."""
    from diffab_pytorch_b200 import diffab_pytorch as dp
    from diffab_pytorch_b200 import synth
    torch.manual_seed(B)
    layer = dp.InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(DEV)
    layer.load_state_dict(synth.synthetic_state(synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8), seed=1))
    x, e, R, t = (v.to(DEV) for v in synth.make_ipa_inputs(B, 128, 128, 64, seed=20 + B))
    gy = torch.randn(B, 128, 128, device=DEV)
    seen = {}
    orig = dp._IpaFastFunction.backward

    def spy(ctx, dy):
        x_, _, _, saved = ctx.saved_tensors[:4]
        Bq, Lq, D = x_.shape
        M = Bq * Lq
        ncat = ctx.layer.to_out.weight.shape[1]
        dims = dp._ipa_structs(ctx.layer, Bq, Lq)
        offs = (ctypes.c_size_t * 8)()
        _lib.check(_lib.lib().dab_ipa_sm100_workspace_layout(ctypes.byref(dims), offs), "dab_ipa_sm100_workspace_layout")
        seen["dy"] = dy.detach().reshape(M, D).clone()
        seen["cat"] = saved[offs[4]: offs[4] + M * ncat * 2].view(BF).view(M, ncat).clone()
        return orig(ctx, dy)

    dp._IpaFastFunction.backward = staticmethod(spy)
    try:
        (layer(x, e.bfloat16(), R, t) * gy).sum().backward()
    finally:
        dp._IpaFastFunction.backward = staticmethod(orig)
    dy, cat = seen["dy"].double(), seen["cat"].double()
    assert dy.shape == (B * 128, 128) and cat.shape == (B * 128, 1024)
    db = layer.to_out.bias.grad.double()
    assert bool(((db - dy.sum(0)).abs() <= 1e-6 * dy.abs().sum(0)).all())
    dyb = seen["dy"].bfloat16().double()        # the backward's own copy: dab_cast_f32_to_bf16 rounds as torch does
    _within_product_bound(layer.to_out.weight.grad, dyb.t() @ cat, dyb.abs().t() @ cat.abs())
