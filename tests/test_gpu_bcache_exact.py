"""The kernels of the cached-projection search route (am.AM_resident with bcache, bench.py's forward_search) against exact
or high-precision references, at the shapes and values where they can go wrong:

  * eg_dev_project_i8 (B = Mt U, the scan's int8 contraction in projection mode) and eg_dev_gemv_i8 (DP4A digit GEMV):
    EQUAL to the exact restatements of tests/digits.py (one rounding of an exact integer sum), and within
    1/2 ulp + n 2^(e_k - 56) + the FP64 reference's own gamma_n bound of an FP64 product;
  * eg_dev_bscan: within a bound derived from its summation order of a long-double reference, and its NaN rule;
  * eg_dev_scan_prepare_eig: the folded W = U diag(w) U^T - E E^T against an FP64 fold, componentwise;
  * eg_emma_eigen_R_wo_Z_eigbasis: the device secular solve against the host back end (tests/csrc/secular_host.cpp)
    and a dense eigh.

Mt stores are built directly as int8 tensors (L, store_pitch(n)) with values in {-1, 0, 1} and NONZERO junk in the pad
columns, which the kernels must ignore (their digits there are zero); a few cases go through decode / transpose_kb."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

import digits as dg
from eagleeverything_b200 import _lib, synth

pytestmark = pytest.mark.gpu

U64 = 2.0 ** -53                         # unit roundoff of binary64
SENTINEL = 0x7FF4DEADBEEF0001           # a signalling-NaN bit pattern no kernel produces


def p(t):
    return C.c_void_p(t.data_ptr())


@pytest.fixture(scope="module")
def lib():
    from eagleeverything_b200 import device
    return device.init(0)


def store(L, n, seed, junk=0x7F):
    """int8 Mt store (L, pitch(n)) with genotypes in {-1, 0, 1} and junk bytes in the pad columns"""
    from eagleeverything_b200 import device
    g = torch.Generator(device="cuda").manual_seed(seed)
    Mt = torch.randint(-1, 2, (L, device.store_pitch(n)), dtype=torch.int8, device="cuda", generator=g)
    Mt[:, n:] = junk
    return Mt


def gamma(k):
    return k * U64 / (1 - k * U64)


# ------------------------------------------------------------------------------------------------ eg_dev_project_i8
def make_U(kind, n, seed):
    """n x n FP64 matrix (rows i contracted with the store, columns k) of one kind"""
    rng = np.random.default_rng(seed)
    if kind == "eig":                                   # eigenvectors of a genotype K
        G = synth.genotypes(n, 3 * n + 7, seed=seed).astype(np.float64) - 1.0
        K = G @ G.T
        return np.linalg.eigh(K / max(K.max(), 1.0) + 0.95 * np.eye(n))[1]
    if kind == "dense":                                 # general, not orthogonal
        return rng.standard_normal((n, n)) + 0.3
    if kind == "scaled":                                # columns scaled by 2^k, k in [-500, 500]
        return rng.standard_normal((n, n)) * 2.0 ** rng.integers(-500, 501, n)[None, :]
    assert kind == "edges"
    U = rng.uniform(-1, 1, (n, n))
    top = 127 / 128
    for k in range(n):
        c = U[:, k] * 2.0 ** int(rng.integers(-60, 60))
        mx = np.abs(c).max() if n > 1 else 1.0
        r = k % 8
        if r == 0:
            c[:] = 0.0                                  # zero column
        elif r in (1, 2, 3):                            # maximum at 127/128 2^e and one ulp either side
            t = (top, np.nextafter(top, 0), np.nextafter(top, 1))[r - 1]
            c = c / mx * t * 0.999
            c[k % n] = t * 2.0 ** (k % 7 - 3) * (-1 if k % 2 else 1)
            c[:] = np.where(np.arange(n) == k % n, c, c * 2.0 ** (k % 7 - 3))
        elif r == 4:                                    # one large entry, the rest below its last digit: round to 0
            c = rng.uniform(-1, 1, n) * 2.0 ** -60
            c[(3 * k) % n] = 1.5
        elif r == 5:                                    # negative maximum
            c = np.abs(c)
            c[k % n] = -2 * mx
        U[:, k] = c
    return U


# (n, L, ldb extra, U kind): every n in {1, 2, 15, 16, 17, 31, 32, 33, 127, 128, 129, 255, 257, 1000, 2049} once, every L in
# {1, 127, 128, 129, 37 * 128 + 1 (one marker past a super-tile), 20,000 (many waves)} several times, every ldb (minimum even
# value >= n, n + 2, n + 64) with odd and even n, every U kind at small and large n
PROJ_CASES = [
    (1, 1, 0, "edges"), (2, 127, 2, "dense"), (15, 128, 64, "edges"), (16, 129, 0, "scaled"), (17, 4737, 2, "edges"),
    (31, 129, 64, "eig"), (32, 1, 2, "edges"), (33, 127, 0, "scaled"), (127, 128, 2, "edges"), (128, 129, 64, "dense"),
    (129, 4737, 0, "eig"), (255, 1, 64, "scaled"), (257, 20000, 2, "edges"), (1000, 4737, 0, "eig"), (2049, 20000, 64, "scaled"),
]


def project(lib, Mt, L, n, U, ldb, extra_rows=128):
    """B = Mt U through eg_dev_project_i8 into a buffer of L + extra_rows rows of ldb doubles filled with SENTINEL;
    asserts that nothing past row L and nothing in columns >= n was written"""
    Ucm = U.T.contiguous()                              # column-major n x n
    buf = torch.full((L + extra_rows, ldb), SENTINEL, dtype=torch.int64, device="cuda")
    B = buf.view(torch.float64)
    _lib.check(lib.eg_dev_project_i8(p(Mt), L, n, Mt.stride(0), p(Ucm), p(B), ldb, None))
    torch.cuda.synchronize()
    assert bool((buf[L:] == SENTINEL).all()), "write past row L"
    assert bool((buf[:, n:] == SENTINEL).all()), "write into the ldb padding"
    return B[:L, :n].clone()


@pytest.mark.parametrize("n,L,extra,kind", PROJ_CASES, ids=[f"n{c[0]}_L{c[1]}_ldb+{c[2]}_{c[3]}" for c in PROJ_CASES])
def test_projection_equals_the_exact_restatement(lib, n, L, extra, kind):
    """B = Mt U bit for bit (up to the sign of zero) against digits_exact_product, the sentinel rows / columns untouched,
    and B against an FP64 product within 1/2 ulp(B) + n 2^(e_k - 56) + gamma_n (|M| |U|)."""
    ldb = (n + 1) // 2 * 2 + extra
    Mt = store(L, n, seed=n * 7 + L)
    U = torch.from_numpy(make_U(kind, n, seed=n + L)).cuda()
    B = project(lib, Mt, L, n, U, ldb)
    ref = dg.digits_exact_product(Mt, U)
    assert dg.same(B, ref), f"{int((B != ref).sum())} entries differ"
    e, scale = dg.colscale(U)
    Mf = Mt[:, :n].double()
    fp = Mf @ U
    bound = (U64 * B.abs() + n * torch.from_numpy(np.ldexp(1.0, e - 56)).cuda()
             + gamma(n) * (Mf.abs() @ U.abs()))
    fin = torch.from_numpy(np.isfinite(scale) & (e >= -1019)).cuda()
    assert bool(((B - fp).abs() <= bound)[:, fin].all())


def test_projection_nan_column_and_determinism(lib):
    """One NaN in U poisons exactly its column of B; identical marker rows in different 128-row blocks and super-tiles
    give identical bits; two runs give identical bits, also with a scan on another matrix in between (the scan and the
    projection share the slicing workspace and the unit table)."""
    from eagleeverything_b200 import device
    n, L = 300, 37 * 128 * 2 + 55
    Mt = store(L, n, seed=3)
    for j in (130, 37 * 128 + 5, L - 1):
        Mt[j] = Mt[5]                                    # another block, another super-tile, the last partial block
    U = torch.from_numpy(make_U("dense", n, seed=4)).cuda()
    ldb = n + 2
    B0 = project(lib, Mt, L, n, U, ldb)
    for j in (130, 37 * 128 + 5, L - 1):
        assert torch.equal(B0[j].view(torch.int64), B0[5].view(torch.int64))
    Un = U.clone()
    Un[17, 41] = float("nan")
    Bn = project(lib, Mt, L, n, Un, ldb)
    assert bool(torch.isnan(Bn[:, 41]).all())
    keep = torch.arange(n, device="cuda") != 41
    assert torch.equal(Bn[:, keep].view(torch.int64), B0[:, keep].view(torch.int64))
    # a scan of a decoded store with another right-hand side in between
    G = synth.genotypes(n, 2000, seed=11)
    img = torch.from_numpy(np.concatenate([synth.ascii_image(G).reshape(-1), np.zeros(64, np.uint8)])).cuda()
    kb, _ = device.decode_kb(img, 2000 + 1, n, 2000)
    tT = device.transpose_kb(kb, n, 2000)
    S, V, a = synth.scan_inputs(n, 5)
    Wp = device.scan_prepare(*(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (S, V, a)), n)
    device.scan(tT, 2000, n, Wp)
    B1 = project(lib, Mt, L, n, U, ldb)
    assert torch.equal(B1.view(torch.int64), B0.view(torch.int64))
    # and the decoded store itself through the projection (zero pad), against the restatement
    Bd = project(lib, tT, 2000, n, U, ldb)
    assert dg.same(Bd, dg.digits_exact_product(tT, U))


def test_projection_underflow_edge_is_flushed(lib):
    """A column of U whose largest magnitude is below 2^-1020 has scale 2^(e-55) = 0 (documented in si_colscale_kernel):
    its products are exactly 0.  Eigenvector columns (unit norm) never come near it."""
    n, L = 40, 300
    Mt = store(L, n, seed=9)
    U = torch.from_numpy(make_U("dense", n, seed=9)).cuda()
    U[:, 3] *= 2.0 ** -1030
    U[:, 4] *= 2.0 ** -1000                             # e = -999 or so: representable, kept
    B = project(lib, Mt, L, n, U, 40)
    assert bool((B[:, 3] == 0).all()) and bool((B[:, 4] != 0).any())
    assert dg.same(B, dg.digits_exact_product(Mt, U))
    # the same edge in eg_dev_gemv_i8 (gv_slice_kernel)
    assert bool((gemv(lib, Mt, L, n, U[:, 3].contiguous(), 1.0) == 0).all())
    y = gemv(lib, Mt, L, n, U[:, 4].contiguous(), 1.0)
    assert bool((y != 0).any()) and dg.same(y, dg.gemv_exact(Mt, U[:, 4].contiguous(), 1.0))


def test_projection_wide_recombination(lib):
    """n = 65,537 > 65,000: the recombination that avoids int32 overflow of P0 256 + P1 (the only test of p.n > 65000)."""
    n, L = 65537, 300
    free, _ = torch.cuda.mem_get_info()
    if free < 100e9:
        pytest.skip(f"needs ~75 GB of device memory for U, its digit slices and the reference; {free / 1e9:.0f} GB free")
    Mt = store(L, n, seed=65537)
    g = torch.Generator(device="cuda").manual_seed(1)
    T = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=g)     # column-major U = T^T
    ldb = n + 1
    buf = torch.full((L + 128, ldb), SENTINEL, dtype=torch.int64, device="cuda")
    B = buf.view(torch.float64)
    _lib.check(lib.eg_dev_project_i8(p(Mt), L, n, Mt.stride(0), p(T), p(B), ldb, None))
    torch.cuda.synchronize()
    assert bool((buf[L:] == SENTINEL).all()) and bool((buf[:, n:] == SENTINEL).all())
    try:
        ref = dg.digits_exact_product(Mt, T.T)
        assert dg.same(B[:L, :n], ref), f"{int((B[:L, :n] != ref).sum())} entries differ"
    finally:
        del T, B, buf
        torch.cuda.empty_cache()
        lib.eg_shutdown()                               # hand the ~30 GB of digit slices back
        _lib.check(lib.eg_init(0))


# ------------------------------------------------------------------------------------------------ eg_dev_gemv_i8
# (n, L): one x chunk (n <= 16,384 individuals = GD_KW words), exactly one, one past it and several chunks with restaging;
# L from one row to 20,000 > 2 x 148 SMs x 64 rows, so the grid-stride loop over row groups runs
GEMV_CASES = [(1, 1), (15, 63), (16, 64), (17, 65), (517, 20000), (16383, 65), (16384, 20000), (16385, 64), (40000, 20000)]


def gemv(lib, Mt, L, n, x, alpha):
    y = torch.full((L + 64,), float("inf"), dtype=torch.float64, device="cuda")
    _lib.check(lib.eg_dev_gemv_i8(p(Mt), L, n, Mt.stride(0), p(x), float(alpha), p(y), None))
    torch.cuda.synchronize()
    assert bool(torch.isinf(y[L:]).all()), "write past row L"
    return y[:L].clone()


@pytest.mark.parametrize("n,L", GEMV_CASES, ids=[f"n{n}_L{L}" for n, L in GEMV_CASES])
def test_gemv_equals_the_exact_restatement(lib, n, L, monkeypatch):
    """y = alpha Mt x on the DP4A path bit for bit against gemv_exact, for x of a wide dynamic range, x = 0 (exact zeros)
    and x holding one NaN or Inf (every y NaN); alpha negative, not a power of two, and zero; identical rows, identical bits.
    EAGLE_GEMV_MODE=f (FP64 FMAs): within gamma_(n+2) |alpha| |M| |x| + |alpha| n 2^(e - 56) + 2u |y| of the same
    restatement (the restatement's own distance from the exact product is the digit residual n 2^(e-56) plus one rounding)."""
    monkeypatch.delenv("EAGLE_GEMV_MODE", raising=False)
    Mt = store(L, n, seed=n + 3 * L, junk=0x01)
    if L > 1:
        Mt[L - 1] = Mt[0]
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    x = x * torch.exp2(torch.randint(-40, 41, (n,), device="cuda", generator=g).double())
    for alpha in (-0.7, 3.3, 0.0, 1.0):
        y = gemv(lib, Mt, L, n, x, alpha)
        assert dg.same(y, dg.gemv_exact(Mt, x, alpha)), alpha
        if L > 1:
            assert y[L - 1].item() == y[0].item() or (math.isnan(y[0].item()) and math.isnan(y[L - 1].item()))
    z = torch.zeros(n, dtype=torch.float64, device="cuda")
    assert bool((gemv(lib, Mt, L, n, z, -1.5) == 0).all())
    for bad in (float("nan"), float("inf")):
        xb = x.clone()
        xb[n // 2] = bad
        assert bool(torch.isnan(gemv(lib, Mt, L, n, xb, 2.0)).all())
    monkeypatch.setenv("EAGLE_GEMV_MODE", "f")
    e, _ = dg.colscale(x.reshape(n, 1))
    Mf = Mt[:, :n].double()
    for alpha in (-0.7, 0.0):
        y = gemv(lib, Mt, L, n, x, alpha)
        ref = dg.gemv_exact(Mt, x, alpha)
        bound = abs(alpha) * (gamma(n + 2) * (Mf.abs() @ x.abs()) + n * math.ldexp(1.0, int(e[0]) - 56)) + 2 * U64 * ref.abs()
        assert bool(((y - ref).abs() <= bound).all())


# ------------------------------------------------------------------------------------------------ eg_dev_bscan
def bscan_bound_depth(n):
    """Roundings on the path of every term of s_j = sum_k w_k B_jk^2 in bscan_kernel: 1 (w b) + the longest accumulator
    chain + 2 (the four accumulators) + 5 (the warp's shuffle tree).  Lane l's acc[0] takes 2 FMAs per step of the
    vectorised loop (at most ceil(n / 256) steps) and 2 per step of the 64-wide tail (at most 4 steps: the loop ends
    at k >= n - 193), so the chain is at most 2 ceil(n / 256) + 8.  All terms are >= 0 for w > 0, hence
    |s - s_ref| <= gamma_depth sum_k w_k B_jk^2."""
    return 1 + (2 * ((n + 255) // 256) + 8) + 2 + 5


# n at the hand-over between the vectorised loop (k + 193 < n) and the tail, below one warp's 64 columns, and large;
# L > 148 * 16 * 8 = 18,944 rows for some, so warps take a second row in the grid-stride loop
BSCAN_CASES = [(1, 19000, 0), (2, 777, 2), (63, 777, 64), (64, 19000, 2), (65, 777, 0), (193, 777, 64), (194, 19000, 0),
               (255, 777, 2), (256, 777, 64), (257, 19000, 2), (449, 777, 0), (450, 19000, 64), (10001, 300, 2)]


@pytest.mark.parametrize("n,L,extra", BSCAN_CASES, ids=[f"n{n}_L{L}_ldb+{x}" for n, L, x in BSCAN_CASES])
def test_bscan_against_long_double(lib, n, L, extra):
    """s_j within gamma_depth sum w B^2 (bscan_bound_depth) of a long-double sum (whose own error, <= (n + 2) 2^-64 of the
    same sum, is added); the ldb padding and the rows past L hold NaN, which must never be read; identical rows at
    positions of different warps, blocks and grid-stride passes give identical bits; q = 0 returns s itself."""
    ldb = (n + 1) // 2 * 2 + extra
    g = torch.Generator(device="cuda").manual_seed(n + L)
    Bbuf = torch.full((L + 16, ldb), float("nan"), dtype=torch.float64, device="cuda")
    Bbuf[:L, :n] = torch.randn((L, n), dtype=torch.float64, device="cuda", generator=g) * \
        torch.exp2(torch.randint(-20, 21, (L, 1), device="cuda", generator=g).double())
    for j in (3 + 8, 5 + 8 * 148, L - 1):
        if j < L:
            Bbuf[j] = Bbuf[3]
    w = torch.rand(n, dtype=torch.float64, device="cuda", generator=g) * 10 + 1e-3
    tmp = torch.empty(L, dtype=torch.float64, device="cuda")
    vara = torch.empty(L, dtype=torch.float64, device="cuda")
    _lib.check(lib.eg_dev_bscan(p(Bbuf), L, n, ldb, p(w), None, 0, p(tmp), p(vara), None))
    torch.cuda.synchronize()
    assert torch.equal(vara.view(torch.int64), tmp.view(torch.int64))
    Bh = Bbuf[:L, :n].cpu().numpy().astype(np.longdouble)
    terms = w.cpu().numpy().astype(np.longdouble)[None, :] * Bh * Bh
    ref = terms.sum(axis=1)
    s = tmp.cpu().numpy().astype(np.longdouble)
    tol = np.longdouble(gamma(bscan_bound_depth(n))) * ref + np.longdouble((n + 2) * 2.0 ** -64) * ref
    assert (np.abs(s - ref) <= tol).all(), float(np.max(np.abs(s - ref) / ref))
    sb = tmp.view(torch.int64)
    for j in (3 + 8, 5 + 8 * 148, L - 1):
        if j < L:
            assert sb[j].item() == sb[3].item()


def test_bscan_combine_nan_rule(lib):
    """vara = s - sum_c e_c^2, reported NaN (not testable) when q > 0, s > 0 and vara <= 1e-10 s: rows just below and just
    above the threshold fall on either side; q = 0 never gives NaN; a zero row of B (s = 0) is never NaN."""
    n, L = 70, 600
    g = torch.Generator(device="cuda").manual_seed(5)
    B = torch.randn((L, n), dtype=torch.float64, device="cuda", generator=g)
    B[7] = 0.0
    B[8] = 0.0
    w = torch.rand(n, dtype=torch.float64, device="cuda", generator=g) + 0.5
    tmp, vara = torch.empty(L, dtype=torch.float64, device="cuda"), torch.empty(L, dtype=torch.float64, device="cuda")
    _lib.check(lib.eg_dev_bscan(p(B), L, n, n, p(w), None, 0, p(tmp), p(vara), None))
    torch.cuda.synchronize()
    s = tmp.cpu().numpy()
    assert not np.isnan(vara.cpu().numpy()).any()
    # e_0 with e_0^2 = s (1 - f 1e-10): f cycles through just below / just above the threshold, far above, and exactly 1
    f = np.array([0.9, 1.1, 0.5, 2.0, 1e3, 1.0])[np.arange(L) % 6]
    e = np.zeros((2, L))
    e[0] = np.sqrt(s * (1 - f * 1e-10))
    e[0, 8] = 1e-3                                   # s = 0 with a nonzero e: v < 0 but s > 0 fails: not NaN
    c = e[0] * e[0]                                  # fma(e, e, 0) = RN(e^2); the second (zero) vector adds exactly 0
    v = s - c
    expect_nan = (s > 0) & (v <= 1e-10 * s)
    assert expect_nan[f == 0.9].all() and not expect_nan[(f == 1.1) | (f == 2.0) | (f == 1e3)].any()
    de = torch.from_numpy(e).cuda()
    _lib.check(lib.eg_dev_bscan(p(B), L, n, n, p(w), p(de), 2, p(tmp), p(vara), None))
    torch.cuda.synchronize()
    got = vara.cpu().numpy()
    assert np.array_equal(np.isnan(got), expect_nan)
    assert np.array_equal(got[~expect_nan], v[~expect_nan])
    assert not np.isnan(got[[7, 8]]).any()


# ------------------------------------------------------------------------------------------------ eg_dev_scan_prepare_eig
# n across one 32-tile, its edges and the FP64 / int8 switch of eg_prep_uses_i8 (511 / 512); q from 0 (Et NULL, the fold's
# one-column dummy buffer) to the cap of 64
PREP_CASES = [(1, 0), (31, 1), (32, 64), (33, 7), (511, 64), (512, 0), (1025, 7), (2000, 1)]


@pytest.mark.parametrize("mode", ["i8", "f64"])
@pytest.mark.parametrize("n,q", PREP_CASES, ids=[f"n{n}_q{q}" for n, q in PREP_CASES])
def test_prepare_eig_against_the_dense_fold(lib, n, q, mode, monkeypatch):
    """The packed right-hand side: diag(W), 2 strict_upper(W), a zero strict lower triangle, zero rows n..Kpad-1, and
    column n = U vt, for W = U diag(w) U^T - E E^T, E = U Et, against FP64 on the device.  Componentwise bounds, both
    operands' rounding counted (reference and kernel): the int8 path's digit residual 2^-56 per entry relative to the
    row maxima of A = U diag(sqrt w), 8 n of them per product as in test_preproducts_int8_slices_match_float64, plus
    (2n + 4) u |U| diag(w) |U|^T (sqrt w, the reference's GEMM and the recombination); the FP64 path (2n + 4) u
    |U| diag(w) |U|^T; E E^T: (4n + 2q + 4) u |E|~ |E|~^T with |E|~ = |U| |Et| (two GEMMs of n terms, q-term sums);
    the subtraction 2u |W|; column n: 2 (n + 1) u |U| |vt|."""
    monkeypatch.setenv("EAGLE_PREP_MODE", mode)
    f64 = dict(dtype=torch.float64, device="cuda")
    rng = np.random.default_rng(n * 100 + q)
    U = np.linalg.qr(rng.standard_normal((n, n)))[0]
    w = rng.uniform(0.05, 20.0, n)
    Et = rng.standard_normal((n, q)) * 0.3
    vt = rng.standard_normal(n)
    dU, dUt = torch.from_numpy(U.T.copy()).cuda(), torch.from_numpy(U.copy()).cuda()
    d_w, d_vt = torch.from_numpy(w).cuda(), torch.from_numpy(vt).cuda()
    d_Et = torch.from_numpy(Et.T.copy()).cuda() if q else None
    Wp = torch.full((lib.eg_scan_wp_elems(n),), 7.0, **f64)
    work = torch.empty(n * max(q, 1), **f64)
    work2 = torch.empty(n * n, **f64)
    _lib.check(lib.eg_dev_scan_prepare_eig(p(dU), p(dUt), n, p(d_w), p(d_Et) if q else None, q, p(d_vt), p(work), p(work2),
                                           p(Wp), None))
    torch.cuda.synchronize()
    Kpad = (n + 31) // 32 * 32
    cols = Wp[: Kpad * (n + 1)].view(n + 1, Kpad)          # row c = column c of the packed matrix
    Wk = cols[:n, :n].T                                    # Wk[i, j] = packed (i, j)
    assert bool((cols[:, n:] == 0).all()), "rows n..Kpad-1 must be zero"
    assert bool((torch.tril(Wk, -1) == 0).all()), "strict lower triangle must be zero"
    Ut = torch.from_numpy(U).cuda()
    Etd = torch.from_numpy(Et).cuda()
    E = Ut @ Etd
    W = (Ut * d_w) @ Ut.T - E @ E.T
    fold = torch.triu(W, 1) * 2 + torch.diag(torch.diag(W))
    absUwU = (Ut.abs() * d_w) @ Ut.abs().T
    Ea = Ut.abs() @ Etd.abs()
    tol = (2 * n + 4) * U64 * absUwU + (4 * n + 2 * q + 4) * U64 * (Ea @ Ea.T) + 2 * U64 * W.abs()
    if mode == "i8":
        rA = (Ut.abs() * d_w.sqrt()).amax(dim=1)
        tol = tol + 8 * n * 2.0 ** -56 * torch.outer(rA, rA)
    tol = torch.triu(tol, 1) * 2 + torch.diag(torch.diag(tol))
    err = (torch.triu(Wk) - fold).abs()
    assert bool((err <= tol).all()), float((err / tol).max())
    v = cols[n, :n]
    vref = Ut @ d_vt
    assert bool(((v - vref).abs() <= 2 * (n + 1) * U64 * (Ut.abs() @ d_vt.abs())).all())


def test_prepare_eig_refusals(lib, monkeypatch):
    f64 = dict(dtype=torch.float64, device="cuda")
    n = 40
    U = torch.eye(n, **f64)
    w, vt = torch.ones(n, **f64), torch.ones(n, **f64)
    Et = torch.zeros(65 * n, **f64)
    work, work2, Wp = torch.empty(65 * n, **f64), torch.empty(n * n, **f64), torch.empty(lib.eg_scan_wp_elems(n), **f64)
    assert lib.eg_dev_scan_prepare_eig(p(U), p(U), n, p(w), p(Et), 65, p(vt), p(work), p(work2), p(Wp), None) == _lib.EG_ERR_ARG
    assert lib.eg_dev_scan_prepare_eig(p(U), p(U), n, p(w), None, 1, p(vt), p(work), p(work2), p(Wp), None) == _lib.EG_ERR_ARG
    monkeypatch.setenv("EAGLE_PREP_MODE", "f64")
    assert lib.eg_dev_scan_prepare_eig(p(U), p(U), n, p(w), p(Et), 1, p(vt), p(work), None, p(Wp), None) == _lib.EG_ERR_ARG
    assert b"needs d_work2" in lib.eg_last_error()
    _lib.check(lib.eg_dev_scan_prepare_eig(p(U), p(U), n, p(w), p(Et), 64, p(vt), p(work), p(work2), p(Wp), None))


# ------------------------------------------------------------------------------------------------ device secular solve
@pytest.fixture(scope="module")
def sec_host(tmp_path_factory):
    """the header's host back end (plain loops), built like test_secular_cpu.py's fixture, into a temporary directory"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path_factory.mktemp("sec") / "libsecular_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", out,
                           os.path.join(root, "tests", "csrc", "secular_host.cpp")])
    return C.CDLL(out)


def _solve(lib, xi, Xt, yt):
    """(rc, values, etas, [steps, deflated, max_iters, roots]) from the device entry point (lib = libeaglegpu) or the host
    back end (lib = the test build of secular_host.cpp)"""
    n, q = Xt.shape
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    Xf, xi, yt = np.asfortranarray(Xt, dtype=np.float64), np.ascontiguousarray(xi, dtype=np.float64), np.ascontiguousarray(yt)
    vals, etas, st = np.empty(n - q), np.empty(n - q), (C.c_int64 * 4)()
    if hasattr(lib, "th_secular_compress"):
        rc = lib.th_secular_compress(C.c_int64(n), q, dp(xi), dp(Xf), dp(yt), dp(vals), dp(etas), st)
    else:
        rc = lib.eg_emma_eigen_R_wo_Z_eigbasis(dp(xi), dp(Xf), dp(yt), n, q, dp(vals), dp(etas), st)
    return rc, vals, etas, list(st)


def _spectral_sums(vals, etasq):
    return np.array([[(etasq / (vals + d)).sum(), (etasq / (vals + d) ** 2).sum()] for d in (1e-5, 1e-2, 1.0, 1e2)])


def _sec_problem(kind, n, q, seed):
    rng = np.random.default_rng(seed)
    if kind == "random":                                   # distinct poles, no component negligible: no deflation
        return np.sort(0.95 + rng.uniform(0, 3, n)), rng.standard_normal((n, q)), rng.standard_normal(n)
    if kind == "graded":                                   # test_secular_graded_and_clustered_poles' spectrum
        xi = np.sort(np.concatenate([0.95 + 10 ** rng.uniform(-14, -1, n // 2), 0.95 + rng.uniform(0, 50, n - n // 2)]))
        xi[40:48] = xi[40]                                 # a cluster of equal poles
        Xt = rng.standard_normal((n, q)) * 10 ** rng.uniform(-16, 0, (n, 1))
        return xi, Xt, rng.standard_normal(n)
    G = rng.integers(0, 3, (n, max(n // 3, 2) if kind == "deflated" else 3 * n))  # genotype K; L < n: repeated 0.95
    M = G.astype(np.float64) - 1.0
    K = M @ M.T
    K = K / max(K.max(), 1.0) + 0.95 * np.eye(n)
    xi, U = np.linalg.eigh(K)
    X = np.column_stack([np.ones(n)] + [rng.standard_normal(n) for _ in range(q - 1)])
    return xi, U.T @ X, U.T @ (rng.standard_normal(n) + M[:, 0])


# the smallest active problems (n = 3 and n = 2 with q = 1: ma = 3, then ma = 2, one CTA), q = 8, 9, 17 carried columns
# around the SEC_RC = 8 chunks of sec_transform_kernel, graded / clustered poles, and a deflating genotype K (L < n)
SEC_CASES = [("graded", 300, 1), ("graded", 300, 4), ("graded", 3000, 2), ("deflated", 600, 3), ("random", 3, 1),
             ("random", 2, 1), ("genotype", 200, 8), ("genotype", 200, 9), ("genotype", 250, 17)]


@pytest.mark.parametrize("kind,n,q", SEC_CASES, ids=[f"{k}_n{n}_q{q}" for k, n, q in SEC_CASES])
def test_device_secular_solve_against_host_and_eigh(lib, sec_host, kind, n, q):
    """eg_emma_eigen_R_wo_Z_eigbasis (sec_roots / sec_lowner / sec_transform kernels) against the same header run by the
    host loop back end and a dense eigh of P diag(xi) P.  Deflation is host code: steps and deflated are equal.  Both
    back ends stop a root at |f| <= 4 eps asum or a bracket of relative width 2 eps; f' >= asum / spread(xi) (every
    term's slope is its value over its pole distance), so a root moves by at most (4 eps + the evaluation error of f)
    spread over the two stopping points; with the typical evaluation error sqrt(m) eps asum of the two summation
    orders that is 2 (4 + sqrt(n)) eps spread, plus 4 eps max|xi| for lambda = d_origin + mu."""
    xi, Xt, yt = _sec_problem(kind, n, q, seed=n * 10 + q)
    dev = _solve(lib, xi, Xt, yt)
    host = _solve(sec_host, xi, Xt, yt)
    assert dev[0] == 0 and host[0] == 0
    assert dev[3][0] == host[3][0] == q and dev[3][1] == host[3][1] and dev[3][2] < 60
    if kind == "deflated":
        assert dev[3][1] > 0
    if kind == "random":
        assert dev[3][1] == 0 and dev[3][3] == n - 1      # every pole active: ma = n
    eps = np.finfo(float).eps
    spread = xi.max() - xi.min()
    np.testing.assert_allclose(dev[1], host[1], rtol=0, atol=2 * (4 + math.sqrt(n)) * eps * spread + 4 * eps * np.abs(xi).max())
    Q, _ = np.linalg.qr(Xt)
    P = np.eye(n) - Q @ Q.T
    T = P @ np.diag(xi) @ P
    wv, Vv = np.linalg.eigh((T + T.T) / 2)
    keep = np.sort(np.argsort(np.linalg.norm(Q.T @ Vv, axis=0))[: n - q])
    for _, vals, etas, _ in (dev, host):
        np.testing.assert_allclose(np.sort(vals), np.sort(wv[keep]), rtol=0, atol=1e-12 * np.abs(xi).max())
        np.testing.assert_allclose(_spectral_sums(vals, etas ** 2), _spectral_sums(wv[keep], (Vv[:, keep].T @ yt) ** 2),
                                   rtol=1e-11 if kind != "graded" else 1e-10)
    np.testing.assert_allclose(_spectral_sums(dev[1], dev[2] ** 2), _spectral_sums(host[1], host[2] ** 2), rtol=1e-11)


def test_device_secular_workspace_grows_past_64_columns(lib, sec_host):
    """q = 70 carried columns after a solve with q = 3 on the same thread: the device workspace (sized for 64 columns)
    grows, and the results still match the host back end."""
    for q in (3, 70):
        xi, Xt, yt = _sec_problem("genotype", 400, q, seed=q)
        dev = _solve(lib, xi, Xt, yt)
        host = _solve(sec_host, xi, Xt, yt)
        assert dev[0] == host[0] == 0 and dev[3][:2] == host[3][:2] and dev[3][2] < 60
        eps = np.finfo(float).eps
        atol = 2 * (4 + math.sqrt(400)) * eps * (xi.max() - xi.min()) + 4 * eps * np.abs(xi).max()
        np.testing.assert_allclose(dev[1], host[1], rtol=0, atol=atol)
        np.testing.assert_allclose(_spectral_sums(dev[1], dev[2] ** 2), _spectral_sums(host[1], host[2] ** 2), rtol=1e-11)
