"""Tensor-core GEMMs (tcgen05: tf32x3, tf32x3c2, tf32, tf32c2) and the fused edge-MLP forward on the paths the
workload shapes do not reach: the scalar-load instantiations (misaligned bases, odd leading dimensions, widths that
are not a multiple of 4), ragged tiles at the 16 / 128 / 256 boundaries, K = 0, both sides of every dispatch guard of
``gemm_raw``, and the row-count invariance ``fixed_backend`` promises.

Results are checked entry by entry against fp64 with the error bound of the kernels' arithmetic (``coef``), not with
the per-tensor max|a-b| / max|b|: the inputs span 1e-4 .. 1e4 over output rows and columns, and an error confined to
the small entries would vanish in a per-tensor ratio."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

U24 = 2.0 ** -24            # unit roundoff of fp32 (round to nearest)
KCAP = 1088                 # _ops.TF32X3_KCAP: most k-terms one 3xTF32 accumulator takes
EPI = 2.0 ** -22            # relative error of the epilogue's fp32 adds (beta*C0, bias), a few roundings
TC_BACKENDS = ("tf32x3", "tf32x3c2", "tf32", "tf32c2")
THREE_PASS = {"tf32x3": "tf32x3", "tf32x3c2": "tf32x3c2", "tf32": "tf32x3", "tf32c2": "tf32x3c2"}
LAYOUTS = [(False, True), (False, False), (True, False), (True, True)]


@pytest.fixture(scope="module")
def ops():
    from plnlp_b200 import _lib, _ops
    assert _lib.load().plnlp_check_device() == 0
    return _ops


# ------------------------------------------------------------------ reference and bound
def coef(arith, K, kacc=KCAP):
    """c of the entry-wise bound |got - exact| <= c * (|op(A)| @ |op(B)|)_ij for a K-term product:

    "3x"  3xTF32 (tf32x3, tf32x3c2, and the scalar-load instantiations of every tensor-core backend): 2^-19 for the
          operand split -- the dropped lo*lo term (2^-22) plus both lo parts read with 11 significant bits
          (2 x 2^-21) -- plus one round-toward-zero step of the accumulator (< 2^-23 of a partial sum, itself at
          most (|A||B|)_ij) for each of the 3 MMAs per 8 k-terms, over at most ``kacc`` k-terms per accumulator
          (1088 for a 3xTF32 request), plus 2^-24 per round-to-nearest add of the split-k partials.  At K = 64:
          4.8e-6; at K = 1088: 5.1e-5.
    "1x"  plain TF32: 2^-10 + 2^-20 (both operands rounded to 11 significant bits) + one step per 8 k-terms.
    "f32" FFMA on the CUDA cores: (K + 2) * 2^-24."""
    if arith == "f32":
        return (K + 2) * U24
    if arith == "1x":
        return 2.0 ** -10 + 2.0 ** -20 + math.ceil(K / 8) * 2 * U24
    return 2.0 ** -19 + 3 * math.ceil(min(K, kacc) / 8) * 2 * U24 + math.ceil(K / kacc) * U24


def product(A, B, ta, tb):
    """exact op(A) @ op(B) and |op(A)| @ |op(B)|, fp64 on the device"""
    a = (A.t() if ta else A).cuda().double()
    b = (B.t() if tb else B).cuda().double()
    return a @ b, a.abs() @ b.abs()


def assert_within(got, exact, bnd, what):
    """|got - exact| <= bnd for every entry (NaN fails); returns the worst err / bound"""
    err = (got.double() - exact).abs()
    bad = ~(err <= bnd)
    if bool(bad.any()):
        idx = tuple(bad.nonzero()[0].tolist())
        worst = float((err[bad] / bnd[bad]).nan_to_num(float("inf")).max())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} entries outside the bound, worst err/bound "
                             f"{worst:.3g}; first at {idx}: got {float(got[idx])!r}, exact {float(exact[idx])!r}, "
                             f"bound {float(bnd[idx]):.3g}")
    live = bnd > 0
    return float((err[live] / bnd[live]).max()) if bool(live.any()) else 0.0


def spread(n, g):
    """n factors log-spaced over 1e-4 .. 1e4 (both ends present when n > 1), in random order"""
    if n <= 1:
        return torch.ones(n)
    return (10.0 ** torch.linspace(-4.0, 4.0, n))[torch.randperm(n, generator=g)]


def operands(M, N, K, ta, tb, g):
    """op(A) [M, K] with its rows scaled over 1e-4 .. 1e4 and op(B) [K, N] with its columns scaled the same way, in the
    stored layout (A = op(A)^T when ta, B = op(B)^T when tb), plus the row scales.  The scales sit on the output rows
    and columns: each output entry is a sum of terms of one magnitude, and entries from 1e-8 to 1e8 are each held to
    their own bound."""
    rs = spread(M, g)
    a = torch.randn(M, K, generator=g) * rs[:, None]
    b = torch.randn(K, N, generator=g) * spread(N, g)[None, :]
    return (a.t().contiguous() if ta else a), (b.t().contiguous() if tb else b), rs


def strided(x, off, ld=None):
    """x copied into a NaN-filled CUDA buffer as a view whose base lies ``off`` floats past a 16-byte boundary, with
    leading dimension ``ld`` (default: the smallest odd number > x.size(1)) -- a column slice of a wider table.  A read
    past the end of a row brings NaN into the result."""
    r, c = x.shape
    if ld is None:
        ld = c + 1 if c % 2 == 0 else c + 2
    buf = torch.full((off + max(r, 1) * ld,), float("nan"), device="cuda")
    v = buf[off:off + r * ld].view(r, ld)[:, :c]
    v.copy_(x)
    return v


def vector_loads(ops, M, N, K, ta, tb, A, B):
    """whether the tensor-core launch tables pick the 16-byte (vector) loaders for both operands (with the leading
    dimension gemm_raw passes: a one-row tensor may carry any row stride)"""
    def ok(t, extent):
        return t.data_ptr() % 16 == 0 and ops._ld(t) % 4 == 0 and extent % 4 == 0
    return ok(A, M if ta else K) and ok(B, K if tb else N)


def kernels_of(fn):
    """run fn with profiling spans on -> (result, names of the kernels it launched)"""
    from plnlp_b200 import profiling
    profiling.enable()
    try:
        out = fn()
    finally:
        spans = profiling.disable()
    return out, {name.split()[0] for name in spans}


# ------------------------------------------------------------------ generic tcgen05 GEMMs: loaders and ragged tiles
SWEEP = [(127, 16, 15), (128, 17, 16), (129, 255, 17), (255, 128, 1), (256, 129, 0), (257, 256, 33), (1, 257, 130),
         (300, 1, 64)]


@pytest.mark.parametrize("M,N,K", SWEEP, ids=[f"{m}x{n}x{k}" for m, n, k in SWEEP])
@pytest.mark.parametrize("ta,tb", LAYOUTS, ids=["NT", "NN", "TN", "TT"])
@pytest.mark.parametrize("backend", TC_BACKENDS)
def test_gemm_unaligned_views_and_contiguous(ops, backend, ta, tb, M, N, K):
    """the same product from operands given as misaligned views with odd leading dimensions (scalar loaders) and
    contiguous (vector loaders where the extents allow), on the tensor-core kernel itself (fixed_backend), at tile
    edges around 16 / 128 / 256 and K in {0, 1, 15, 16, 17, ...}"""
    g = torch.Generator().manual_seed(1000 * M + 10 * N + K)
    A, B, _ = operands(M, N, K, ta, tb, g)
    off = 1 + (M + N + K) % 3
    Av, Bv = strided(A, off), strided(B, 4 - off)
    Ac, Bc = A.cuda(), B.cuda()
    kw = dict(transa=ta, transb=tb, split_k=1, fixed_backend=True)
    exact, absab = product(A, B, ta, tb)
    got_v = ops.gemm_raw(Av, Bv, backend=backend, **kw)
    assert_within(got_v, exact, coef("3x", K) * absab, f"{backend} views")
    got_c = ops.gemm_raw(Ac, Bc, backend=backend, **kw)
    plain = backend in ("tf32", "tf32c2") and vector_loads(ops, M, N, K, ta, tb, Ac, Bc)
    assert_within(got_c, exact, coef("1x" if plain else "3x", K) * absab, f"{backend} contiguous")
    # the scalar instantiations are 3xTF32 whatever the request: bit for bit the 3-pass result on the same views
    assert torch.equal(got_v, ops.gemm_raw(Av, Bv, backend=THREE_PASS[backend], **kw))
    if not plain:
        assert torch.equal(got_v, got_c)           # same split, same MMA order: the loaders change no bit


@pytest.mark.parametrize("ta,tb", LAYOUTS, ids=["NT", "NN", "TN", "TT"])
@pytest.mark.parametrize("backend", TC_BACKENDS + ("ffma",))
def test_gemm_k0_is_beta_c_plus_bias(ops, backend, ta, tb):
    """K = 0 (empty operands as torch allocates them): C = beta*C0 + bias exactly, through relu too"""
    M, N = 129, 257
    g = torch.Generator().manual_seed(7)
    A = torch.empty((0, M) if ta else (M, 0), device="cuda")
    B = torch.empty((N, 0) if tb else (0, N), device="cuda")
    C0, bias = torch.randn(M, N, generator=g).cuda(), torch.randn(N, generator=g).cuda()
    kw = dict(transa=ta, transb=tb, split_k=1, backend=backend, fixed_backend=True)
    C = C0.clone()
    ops.gemm_raw(A, B, C=C, beta=0.5, bias=bias, **kw)
    assert torch.equal(C, 0.5 * C0 + bias)
    assert torch.equal(ops.gemm_raw(A, B, bias=bias, act=ops.ACT_RELU, **kw), bias.clamp_min(0).expand(M, N))
    assert torch.equal(ops.gemm_raw(A, B, **kw), torch.zeros(M, N, device="cuda"))


@pytest.mark.parametrize("ta,tb", [(False, True), (True, False)], ids=["NT", "TN"])
@pytest.mark.parametrize("backend", TC_BACKENDS)
def test_gemm_epilogues_on_scalar_path(ops, backend, ta, tb):
    """beta + bias + relu into a misaligned column slice of a wider C (neighbours untouched), relu-grad with aux as a
    view, and dropout with the FFMA kernel's Philox mask -- every operand unaligned"""
    M, N, K = 257, 131, 67
    g = torch.Generator().manual_seed(11)
    A, B, rs = operands(M, N, K, ta, tb, g)
    cs = spread(N, g)
    Av, Bv = strided(A, 1), strided(B, 3)
    kw = dict(transa=ta, transb=tb, split_k=1, backend=backend, fixed_backend=True)
    exact, absab = product(A, B, ta, tb)
    c = coef("3x", K)
    C0 = (torch.randn(M, N, generator=g) * rs[:, None] * cs[None, :]).cuda()
    bias = (torch.randn(N, generator=g) * cs).cuda()
    bias_v = strided(bias.cpu()[None], 2)[0]

    wide = torch.full((M, N + 5), -7.0, device="cuda")
    Cv = wide[:, 2:2 + N]
    Cv.copy_(C0)
    ops.gemm_raw(Av, Bv, C=Cv, beta=0.5, bias=bias_v, act=ops.ACT_RELU, **kw)
    ref = (exact + 0.5 * C0.double() + bias.double()).clamp_min(0)
    assert_within(Cv, ref, c * absab + EPI * (0.5 * C0.double().abs() + bias.double().abs()), "beta+bias+relu")
    assert bool((wide[:, :2] == -7.0).all()) and bool((wide[:, 2 + N:] == -7.0).all())

    aux = strided(torch.randn(M, N, generator=g), 2)
    keep = (aux > 0).double()
    G = ops.gemm_raw(Av, Bv, act=ops.ACT_RELU_GRAD, aux=aux, **kw)
    assert_within(G, exact * keep, c * absab * keep, "relu-grad")

    # dropout: non-negative operands and a positive bias keep every pre-activation > 0, so a zero is a dropped entry
    Ap, Bp, bp = strided(A.abs(), 1), strided(B.abs(), 3), bias.abs() + 1.0
    d_tc = ops.gemm_raw(Ap, Bp, bias=bp, act=ops.ACT_RELU, drop_p=0.5, seed=1234, **kw)
    d_ff = ops.gemm_raw(Ap, Bp, transa=ta, transb=tb, bias=bp, act=ops.ACT_RELU, drop_p=0.5, seed=1234, backend="ffma")
    kept = d_tc != 0
    assert torch.equal(kept, d_ff != 0)
    assert 0.45 < float(kept.float().mean()) < 0.55
    exact_p, abs_p = product(A.abs(), B.abs(), ta, tb)
    k = kept.double()
    assert_within(d_tc, 2 * (exact_p + bp.double()) * k, 2 * (c * abs_p + EPI * bp.double()) * k, "dropout")


@pytest.mark.parametrize("backend", ["tf32", "tf32c2"])
def test_plain_tf32_request_and_the_bound(ops, backend):
    """A plain-TF32 request runs one pass on the vector-load instantiations only.  On the scalar path it runs 3xTF32,
    bit for bit the tf32x3 result (gemm_raw's docstring).  The 3xTF32 bound tells the two apart: the single-pass product
    fails it, in the rows scaled down to 1e-2 and below as well."""
    M, N, K = 256, 256, 64
    g = torch.Generator().manual_seed(5)
    A, B, rs = operands(M, N, K, False, True, g)
    exact, absab = product(A, B, False, True)
    kw = dict(transb=True, split_k=1, fixed_backend=True)
    fast = ops.gemm_raw(A.cuda(), B.cuda(), backend=backend, **kw)
    assert_within(fast, exact, coef("1x", K) * absab, "plain TF32")
    outside = (fast.double() - exact).abs() > coef("3x", K) * absab
    assert bool(outside.any()), "the 3xTF32 bound accepts a single-pass product"
    assert bool(outside[(rs <= 1e-2).cuda()].any()), "the small rows are not checked"
    Av, Bv = strided(A, 1), strided(B, 2)
    slow = ops.gemm_raw(Av, Bv, backend=backend, **kw)
    assert torch.equal(slow, ops.gemm_raw(Av, Bv, backend=THREE_PASS[backend], **kw))
    assert_within(slow, exact, coef("3x", K) * absab, "plain request, scalar path")


@pytest.mark.parametrize("backend", ["tf32", "tf32c2"])
def test_plain_tf32_request_long_k_on_scalar_path(ops, backend):
    """K > 1088 on the scalar path, as gemm_raw dispatches it (no fixed_backend): the 3 passes run in the split the
    plain request asked for -- bit for bit the tf32x3 result under the same split, and in one accumulator over all of
    K when the split is 1 (the 3xTF32 bound with 2000 k-terms per accumulator)"""
    M, N, K = 256, 200, 2000
    g = torch.Generator().manual_seed(17)
    A, B, _ = operands(M, N, K, False, True, g)
    exact, absab = product(A, B, False, True)
    Av, Bv = strided(A, 1), strided(B, 2)
    two = ops.gemm_raw(Av, Bv, transb=True, split_k=2, backend=backend)
    assert torch.equal(two, ops.gemm_raw(Av, Bv, transb=True, split_k=2, backend=THREE_PASS[backend]))
    assert_within(two, exact, coef("3x", K) * absab, "split 2")
    one = ops.gemm_raw(Av, Bv, transb=True, split_k=1, backend=backend)
    assert_within(one, exact, coef("3x", K, kacc=K) * absab, "split 1")


def test_plain_tf32_request_on_tma_kernel(ops, monkeypatch):
    """the TMA-fed tall-skinny kernel needs only A aligned: with B misaligned, at an odd leading dimension, a plain
    request still runs one pass there (outside the 3xTF32 bound, inside the plain-TF32 one)"""
    monkeypatch.setattr(ops, "GEMM_TMA", "auto")
    M, N, K = 16384, 64, 64
    g = torch.Generator().manual_seed(19)
    A, B, _ = operands(M, N, K, False, True, g)
    exact, absab = product(A, B, False, True)
    got, ran = kernels_of(lambda: ops.gemm_raw(A.cuda(), strided(B, 1), transb=True, backend="tf32c2"))
    assert ran == {"gemm_tf32x1_tma"}, ran
    assert_within(got, exact, coef("1x", K) * absab, "plain TF32 on the TMA kernel")
    assert bool(((got.double() - exact).abs() > coef("3x", K) * absab).any())


# ------------------------------------------------------------------ fixed_backend: rows do not depend on the row count
@pytest.mark.parametrize("H", [50, 200, 256])
@pytest.mark.parametrize("backend", TC_BACKENDS)
def test_fixed_backend_rows_independent_of_row_count(ops, backend, H):
    """gemm_raw(A[:m], B, transb=True, split_k=1, fixed_backend=True) is rows [:m] of the full product, bit for bit
    (recommend scores query chunks of any size with it)"""
    M, N = 700, 3001
    g = torch.Generator().manual_seed(H)
    A, B, _ = operands(M, N, H, False, True, g)
    Ag, Bg = A.cuda(), B.cuda()
    kw = dict(transb=True, split_k=1, backend=backend, fixed_backend=True)
    full = ops.gemm_raw(Ag, Bg, **kw)
    exact, absab = product(A, B, False, True)
    plain = backend in ("tf32", "tf32c2") and H % 4 == 0
    assert_within(full, exact, coef("1x" if plain else "3x", H) * absab, backend)
    for m in (1, 127, 128, 129, 255, 256, 257):
        assert torch.equal(ops.gemm_raw(Ag[:m], Bg, **kw), full[:m]), m


# ------------------------------------------------------------------ dispatch guards of gemm_raw
TC, F32 = "gemm_tf32x3_2cta", "gemm_f32"
TMA, TN = "gemm_tf32x3_tma", "gemm_tf32x3_tma_tn"
# (id, M, N, K, transa, transb, options, kernel that must run).  Options: a_ld / a_off / b_ld / b_off = operand as a
# view, epi = "bias" / "beta" / "relu", split_k, fixed = fixed_backend, tma / tma_tn = _ops.GEMM_TMA / GEMM_TMA_TN.
GUARDS = [
    # the CUDA-core fallback: K < 32, N < 16, M*N*K < 2^20
    ("mnk_2p20", 64, 128, 128, False, True, {}, TC),
    ("mnk_below", 63, 128, 128, False, True, {}, F32),
    ("k32", 256, 256, 32, False, True, {}, TC),
    ("k31", 256, 256, 31, False, True, {}, F32),
    ("n16", 4096, 16, 64, False, True, {}, TC),
    ("n15", 4096, 15, 64, False, True, {}, F32),
    # TMA-fed tall-skinny kernel, "auto": M >= 16384, N <= 256, K <= 512
    ("tma_m16384", 16384, 64, 64, False, True, {}, TMA),
    ("tma_m16383", 16383, 64, 64, False, True, {}, TC),
    ("tma_n256", 16384, 256, 64, False, False, {}, TMA),
    ("tma_n257", 16384, 257, 64, False, False, {}, TC),
    ("tma_k512", 16384, 64, 512, False, True, {}, TMA),
    ("tma_k513", 16384, 64, 513, False, True, {}, TC),
    # ... whenever legal ("1"): K >= 32, N <= 512
    ("tma_any_n512", 1000, 512, 64, False, True, {"tma": "1"}, TMA),
    ("tma_any_n513", 1000, 513, 64, False, True, {"tma": "1"}, TC),
    ("tma_any_k32", 1000, 64, 32, False, True, {"tma": "1"}, TMA),
    ("tma_any_k31", 1000, 64, 31, False, True, {"tma": "1"}, F32),
    # ... and on A: ld % 4 == 0, 16-byte base, split_k == 1, not transposed, no fixed_backend
    ("tma_lda68", 16384, 64, 64, False, True, {"a_ld": 68}, TMA),
    ("tma_lda66", 16384, 64, 64, False, True, {"a_ld": 66}, TC),
    ("tma_a_off4", 16384, 64, 64, False, True, {"a_ld": 68, "a_off": 4}, TMA),
    ("tma_a_off2", 16384, 64, 64, False, True, {"a_ld": 68, "a_off": 2}, TC),
    ("tma_split2", 16384, 64, 64, False, True, {"split_k": 2}, TC),
    ("tma_transa", 16384, 64, 64, True, True, {}, TC),
    ("tma_fixed", 16384, 64, 64, False, True, {"fixed": True}, TC),
    # TMA-fed weight-gradient kernel (C = A^T B), "auto": K >= 4 * 148 * 1088
    ("tn_k644096", 16, 16, 644096, True, False, {}, TN),
    ("tn_k644095", 16, 16, 644095, True, False, {}, TC),
    # ... whenever legal ("1"): M <= 256, 8 <= N <= 256 (N < 16 goes to the CUDA cores first), no epilogue,
    # both operands with ld % 4 == 0 and a 16-byte base, B not transposed, no fixed_backend
    ("tn_m256", 256, 64, 4096, True, False, {"tma_tn": "1"}, TN),
    ("tn_m257", 257, 64, 4096, True, False, {"tma_tn": "1"}, TC),
    ("tn_n256", 64, 256, 4096, True, False, {"tma_tn": "1"}, TN),
    ("tn_n257", 64, 257, 4096, True, False, {"tma_tn": "1"}, TC),
    ("tn_n16", 64, 16, 4096, True, False, {"tma_tn": "1"}, TN),
    ("tn_n15", 64, 15, 4096, True, False, {"tma_tn": "1"}, F32),
    ("tn_bias", 64, 64, 4096, True, False, {"tma_tn": "1", "epi": "bias"}, TC),
    ("tn_beta", 64, 64, 4096, True, False, {"tma_tn": "1", "epi": "beta"}, TC),
    ("tn_relu", 64, 64, 4096, True, False, {"tma_tn": "1", "epi": "relu"}, TC),
    ("tn_ldb68", 64, 64, 4096, True, False, {"tma_tn": "1", "b_ld": 68}, TN),
    ("tn_ldb66", 64, 64, 4096, True, False, {"tma_tn": "1", "b_ld": 66}, TC),
    ("tn_lda68", 64, 64, 4096, True, False, {"tma_tn": "1", "a_ld": 68}, TN),
    ("tn_lda66", 64, 64, 4096, True, False, {"tma_tn": "1", "a_ld": 66}, TC),
    ("tn_a_off4", 64, 64, 4096, True, False, {"tma_tn": "1", "a_ld": 68, "a_off": 4}, TN),
    ("tn_a_off2", 64, 64, 4096, True, False, {"tma_tn": "1", "a_ld": 68, "a_off": 2}, TC),
    ("tn_b_off4", 64, 64, 4096, True, False, {"tma_tn": "1", "b_ld": 68, "b_off": 4}, TN),
    ("tn_b_off2", 64, 64, 4096, True, False, {"tma_tn": "1", "b_ld": 68, "b_off": 2}, TC),
    ("tn_transb", 64, 64, 4096, True, True, {"tma_tn": "1"}, TC),
    ("tn_fixed", 64, 64, 4096, True, False, {"tma_tn": "1", "fixed": True}, TC),
]


@pytest.mark.parametrize("M,N,K,ta,tb,opt,kernel", [c[1:] for c in GUARDS], ids=[c[0] for c in GUARDS])
def test_gemm_dispatch_guards(ops, M, N, K, ta, tb, opt, kernel, monkeypatch):
    """each guard of gemm_raw, one shape just inside and one just outside: the kernel that ran (profiling span), the
    entry-wise bound of its arithmetic, and where the TMA kernel runs, bit for bit the CTA-pair result"""
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
    monkeypatch.setattr(ops, "GEMM_TMA", opt.get("tma", "auto"))
    monkeypatch.setattr(ops, "GEMM_TMA_TN", opt.get("tma_tn", "auto"))
    g = torch.Generator().manual_seed(M + 3 * N + 7 * K)
    A, B, rs = operands(M, N, K, ta, tb, g)
    Ag = strided(A, opt.get("a_off", 0), opt["a_ld"]) if "a_ld" in opt else A.cuda()
    Bg = strided(B, opt.get("b_off", 0), opt["b_ld"]) if "b_ld" in opt else B.cuda()
    exact, absab = product(A, B, ta, tb)
    bnd = coef("f32" if kernel == F32 else "3x", K) * absab
    kw = dict(transa=ta, transb=tb, split_k=opt.get("split_k"), fixed_backend=opt.get("fixed", False))
    epi = opt.get("epi")
    C = None
    if epi == "bias":
        bias = torch.randn(N, generator=g).cuda()
        kw["bias"] = bias
        exact, bnd = exact + bias.double(), bnd + EPI * bias.double().abs()
    elif epi == "beta":
        C0 = (torch.randn(M, N, generator=g) * rs[:, None]).cuda()
        C, kw["beta"] = C0.clone(), 0.5
        exact, bnd = exact + 0.5 * C0.double(), bnd + EPI * 0.5 * C0.double().abs()
    elif epi == "relu":
        kw["act"] = ops.ACT_RELU
        exact = exact.clamp_min(0)
    got, ran = kernels_of(lambda: ops.gemm_raw(Ag, Bg, C=C, **kw))
    assert ran == {kernel}, ran
    assert_within(got, exact, bnd, kernel)
    if kernel == TMA:
        monkeypatch.setattr(ops, "GEMM_TMA", "0")
        pair, ran = kernels_of(lambda: ops.gemm_raw(Ag, Bg, **kw))
        assert ran == {TC} and torch.equal(got, pair), float((got - pair).abs().max())


# ------------------------------------------------------------------ fused edge-MLP forward
def edge_problem(N, H, N1, P, g, nonneg=False):
    """embedding table, pair list (negative ids, (u, u) pairs) and head parameters; node rows and hidden columns scaled
    over 1e-4 .. 1e4"""
    h = torch.randn(N, H, generator=g) * spread(N, g)[:, None]
    cs = spread(N1, g)
    W1 = torch.randn(N1, H, generator=g) * cs[:, None] / H ** 0.5
    b1 = torch.randn(N1, generator=g) * cs
    w2, b2 = torch.randn(1, N1, generator=g) / N1 ** 0.5, torch.randn(1, generator=g)
    edges = torch.randint(0, N, (P, 2), generator=g)
    special = torch.tensor([[-1, 3], [5, 5], [-N, -N], [N - 1, -2], [0, 0]])[:P]
    edges[:special.size(0)] = special
    if nonneg:
        h, W1, b1 = h.abs(), W1.abs(), b1.abs() + 1.0
    return h, edges, W1, b1, w2, b2


def edge_reference(h, edges, W1, b1, w2, b2, drop_scale=None, keep=None, arith="3x"):
    """exact a1 = relu(a0 W1^T + b1) (* mask * scale) and score = a1 w2 + b2 in fp64, with their entry-wise bounds:
    the bound of ``arith`` for layer 1 (the fp32 Hadamard product is within 2^-24 of a0, inside the 2^-19 of 3xTF32),
    and for the out layer the propagated layer-1 bound plus one fp32 rounding per term and per partial"""
    hd = h.cuda().double()
    e = edges.cuda()
    a0 = hd[e[:, 0]] * hd[e[:, 1]]
    W1d, b1d, w2d = W1.cuda().double(), b1.cuda().double(), w2.cuda().double().reshape(-1)
    a1 = (a0 @ W1d.t() + b1d).clamp_min(0)
    bnd1 = coef(arith, h.size(1)) * (a0.abs() @ W1d.abs().t()) + EPI * b1d.abs()
    if keep is not None:
        a1, bnd1 = a1 * keep * drop_scale, bnd1 * keep * drop_scale
    N1 = W1.size(0)
    nq = 2 * ((N1 + 255) // 256)
    score = a1 @ w2d + float(b2)
    bnd_s = bnd1 @ w2d.abs() + (N1 + nq + 2) * U24 * ((a1.abs() + bnd1) @ w2d.abs() + abs(float(b2)))
    return a1, bnd1, score, bnd_s


def fused_inputs(N, H, N1, P, layout, seed):
    """(CPU problem, device arguments of edge_mlp_fwd_raw); "views": h and W1 as misaligned column slices"""
    g = torch.Generator().manual_seed(seed)
    h, edges, W1, b1, w2, b2 = edge_problem(N, H, N1, P, g)
    if layout == "views":
        hg, W1g = strided(h, 1), strided(W1, 2)
    else:
        hg, W1g = h.cuda(), W1.cuda()
    return (h, edges, W1, b1, w2, b2), (hg, edges.cuda(), W1g, b1.cuda(), w2.cuda(), b2.cuda())


def check_fused(ops, N, H, N1, P, layout, seed):
    cpu, (hg, eg, W1g, b1g, w2g, b2g) = fused_inputs(N, H, N1, P, layout, seed)
    score, a1 = ops.edge_mlp_fwd_raw(hg, eg, W1g, b1g, w2g, b2g)
    assert score.shape == (P,) and a1.shape == (P, N1)
    ra1, bnd1, rs, bnds = edge_reference(*cpu)
    assert_within(a1, ra1, bnd1, "a1")
    assert_within(score, rs, bnds, "score")
    s2, none = ops.edge_mlp_fwd_raw(hg, eg, W1g, b1g, w2g, b2g, need_a1=False)
    assert none is None and torch.equal(s2, score)


@pytest.mark.parametrize("layout", ["contiguous", "views"])
@pytest.mark.parametrize("H", [32, 33, 50, 130, 1023, 1024])
def test_fused_edge_mlp_widths(ops, H, layout, monkeypatch):
    """embedding widths at both ends of the fused range and between, with h and W1 contiguous or as misaligned column
    slices of wider tables (scalar GatherLoader whenever H % 4 != 0 or a base / leading dimension is unaligned)"""
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
    check_fused(ops, 300, H, 129, 257, layout, seed=H)


@pytest.mark.parametrize("N1", [1, 8, 16, 37, 127, 128, 129, 256, 257, 513, 1024])
@pytest.mark.parametrize("H", [50, 64])
def test_fused_edge_mlp_hidden_widths(ops, H, N1, monkeypatch):
    """hidden widths below the smallest UMMA N (16) and below one tile, ragged, at and across the 128 / 256-column
    halves (the 2 * ceil(N1 / 256) score partials), scalar (H = 50, misaligned views) and vector (H = 64, contiguous)
    gather"""
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
    check_fused(ops, 400, H, N1, 300, "views" if H % 4 else "contiguous", seed=N1 + H)


@pytest.mark.parametrize("P", [0, 1, 127, 128, 129, 255, 256, 257])
def test_fused_edge_mlp_pair_counts(ops, P, monkeypatch):
    """pair counts around the 128-row CTA and the 256-row CTA pair, and none"""
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
    check_fused(ops, 200, 33, 257, P, "views", seed=P)


@pytest.mark.parametrize("layout", ["contiguous", "views"])
def test_fused_edge_mlp_plain_tf32(ops, layout, monkeypatch):
    """GEMM_BACKEND = "tf32c2": one TF32 pass on the vector gather (contiguous, H = 64: inside the plain-TF32 bound,
    outside the 3xTF32 one); on the scalar gather (misaligned views) the "tf32x3c2" result, bit for bit"""
    cpu, args = fused_inputs(400, 64, 257, 300, layout, seed=64)
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32c2")
    score, a1 = ops.edge_mlp_fwd_raw(*args)
    if layout == "contiguous":
        ra1, bnd1, rs, bnds = edge_reference(*cpu, arith="1x")
        assert_within(a1, ra1, bnd1, "a1, one pass")
        assert_within(score, rs, bnds, "score, one pass")
        bnd3 = edge_reference(*cpu)[1]
        assert bool(((a1.double() - ra1).abs() > bnd3).any()), "the 3xTF32 bound accepts a single-pass layer"
    else:
        monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
        s3, a3 = ops.edge_mlp_fwd_raw(*args)
        assert torch.equal(a1, a3) and torch.equal(score, s3)
        ra1, bnd1, rs, bnds = edge_reference(*cpu)
        assert_within(a1, ra1, bnd1, "a1, scalar gather")


@pytest.mark.parametrize("H", [50, 64])
def test_fused_edge_mlp_dropout_mask(ops, H, monkeypatch):
    """dropout in the fused epilogue draws the mask of the unfused gather_hadamard_raw + gemm_raw epilogue (same seed);
    non-negative operands and a positive bias keep every pre-activation > 0, so a zero is a dropped entry"""
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
    g = torch.Generator().manual_seed(77 + H)
    h, edges, W1, b1, w2, b2 = edge_problem(500, H, 257, 2000, g, nonneg=True)
    hg, W1g = (strided(h, 3), strided(W1, 1)) if H % 4 else (h.cuda(), W1.cuda())
    eg, b1g, w2g, b2g = edges.cuda(), b1.cuda(), w2.cuda(), b2.cuda()
    sd, ad = ops.edge_mlp_fwd_raw(hg, eg, W1g, b1g, w2g, b2g, 0.5, 4242)
    au = ops.gemm_raw(ops.gather_hadamard_raw(hg, eg), W1g, transb=True, bias=b1g, act=ops.ACT_RELU, drop_p=0.5,
                      seed=4242)
    kept = ad != 0
    assert torch.equal(kept, au != 0)
    assert 0.45 < float(kept.float().mean()) < 0.55
    ra1, bnd1, rs, bnds = edge_reference(h, edges, W1, b1, w2, b2, drop_scale=2.0, keep=kept.double())
    assert_within(ad, ra1, bnd1, "a1 with dropout")
    assert_within(sd, rs, bnds, "score with dropout")


@pytest.mark.parametrize("H", [16, 31, 32, 33, 1024, 1025])
def test_fused_edge_mlp_predicate_matches_kernel(ops, H, monkeypatch):
    """fused_edge_mlp_ok accepts a head exactly when the fused kernel does (status 0), except H < 32, which the
    predicate leaves to the unfused path on purpose (see its docstring)"""
    monkeypatch.setattr(ops, "GEMM_BACKEND", "tf32x3c2")
    monkeypatch.setattr(ops, "FUSED_EDGE_MLP", True)
    g = torch.Generator().manual_seed(H)
    for N1 in (1, 16, 300):
        for layout in ("contiguous", "views"):
            h, edges, W1, b1, w2, b2 = edge_problem(40, H, N1, 9, g)
            hg, W1g = (strided(h, 1), strided(W1, 3)) if layout == "views" else (h.cuda(), W1.cuda())
            params = [W1g, b1.cuda(), w2.cuda(), b2.cuda()]
            ok = ops.fused_edge_mlp_ok(hg, params)
            try:
                ops.edge_mlp_fwd_raw(hg, edges.cuda(), *params)
                runs = True
            except RuntimeError as e:
                assert "invalid argument" in str(e), e
                runs = False
            assert runs == (H <= 1024), (N1, layout)
            assert ok == (runs and H >= 32), (N1, layout, ok, runs)
