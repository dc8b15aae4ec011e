"""GPU parity tests: the CUDA path (through the C ABI of libeaglegpu.so) against the CPU oracle and
the committed golden fixtures.  Bit-exact for decode / M.Mt / extract.  a and var(a):

    |x - x_ref| <= 1e-9 * |x_ref|  +  4 (n + 10) eps * cond_j

The first term is the north-star tolerance (1e-9 relative).  The second is the floating-point
floor for sums that cancel: markers in span(X) (monomorphic or already selected) have a TRUE value
of 0, and both the reference's Eigen arithmetic and any other summation order return rounding
noise of size gamma_n * sum|terms| there (demo: |a_j| ~ 1e-14 against max|a| ~ 40).  cond_j is that
sum of absolute terms: |m_j| . (|S||a_hat|) for a, |m_j|^T (|S||V||S|) |m_j| for var(a).  For every
marker whose value is not dominated by cancellation the floor is ~1e-12 relative, far inside 1e-9."""
import hashlib
import os

import numpy as np
import pytest

from eagleeverything_b200 import _lib, api, synth
from oracle import am_driver as am
from oracle import eagle_oracle as eo
from oracle import np_oracle as npo

pytestmark = pytest.mark.gpu
NA = api.NA_REAL
RTOL = 1e-9


EPS = np.finfo(np.float64).eps


def scan_conds(G012, S, V, a, zero_rows=()):
    """Rounding-error scales of a_j and vara_j (sums of absolute terms); G012 is n x L."""
    Mabs = np.abs(np.asarray(G012).T.astype(np.float64) - 1.0)  # L x n
    for r in zero_rows:
        Mabs[int(r)] = 0.0
    Sa, Va = np.abs(np.asarray(S)), np.abs(np.asarray(V))
    ca = Mabs @ (Sa @ np.abs(np.asarray(a).reshape(-1)))
    cv = np.einsum("ij,ij->i", Mabs @ (Sa @ (Va @ Sa)), Mabs)
    return ca, cv


def assert_close(x, ref, cond, n, what=""):
    x, ref = np.asarray(x, dtype=np.float64).reshape(-1), np.asarray(ref, dtype=np.float64).reshape(-1)
    tol = RTOL * np.abs(ref) + 4.0 * (n + 10) * EPS * np.asarray(cond).reshape(-1)
    err = np.abs(x - ref)
    bad = ~(err <= tol)
    assert not bad.any(), f"{what}: {bad.sum()} of {bad.size} outside tolerance; worst err/tol " \
                          f"{(err / np.maximum(tol, 1e-300)).max():.3e}"
    # report-style sanity: where the value is not cancellation noise, plain 1e-9 relative holds
    solid = np.abs(ref) > 1e-6 * np.abs(ref).max()
    assert (err[solid] <= RTOL * np.abs(ref[solid])).all(), f"{what}: 1e-9 relative violated on a well-conditioned entry"


@pytest.fixture(params=[0, 1, 2, 3], ids=["dmma_f64", "tcgen05_i8", "tcgen05_i8_cta_pair", "tcgen05_i8_6digits"])
def scan_mode(request):
    """Every scan parity test runs on all contractions of var(a): FP64 DMMA, int8 digit slices with 7 (default) and 6
    digits per column, and the CTA-pair (cta_group::2) variant."""
    prev = api.get_scan_mode()
    prev_pair = os.environ.get("EAGLE_SI_PAIR")
    prev_digits = api.get_scan_digits()
    api.set_scan_mode(min(request.param, 1))
    api.set_scan_digits(6 if request.param == 3 else 7)
    os.environ["EAGLE_SI_PAIR"] = "1" if request.param == 2 else "0"
    yield request.param
    api.set_scan_mode(prev)
    api.set_scan_digits(prev_digits)
    if prev_pair is None:
        os.environ.pop("EAGLE_SI_PAIR", None)
    else:
        os.environ["EAGLE_SI_PAIR"] = prev_pair


def write_pair(tmp_path, G, tag):
    m, mt = str(tmp_path / f"{tag}.M.ascii"), str(tmp_path / f"{tag}.Mt.ascii")
    npo.write_ascii(m, G)
    npo.write_ascii(mt, G.T)
    return m, mt


# ------------------------------------------------------------------------------- decode
def test_readblock_bit_exact(synth_small, monkeypatch):
    s = synth_small
    for piece_bytes in (None, "64"):   # one piece; pieces of 128 lines, whole or a column window of each
        if piece_bytes:
            monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", piece_bytes)
        for (f, start, ncols, nrows) in [(s["M"], 0, s["L"], s["n"]), (s["M"], 7, s["L"], 50), (s["M"], 200, 1, 3),
                                         (s["Mt"], 100, 60, 9), (s["Mt"], 0, s["n"], s["L"]), (s["Mt"], 2999, s["n"], 2),
                                         (s["Mt"], 5, 150, 2990)]:
            got = api.ReadBlock(f, start, ncols, nrows)
            ref = eo.ReadBlock(f, start, ncols, nrows)
            assert got.flags.f_contiguous and got.shape == ref.shape
            assert np.array_equal(got, ref), (piece_bytes, start, ncols, nrows)


def test_open_and_format_errors(tmp_path, synth_small):
    with pytest.raises(_lib.EagleGpuError, match="Could not open") as e:
        api.ReadBlock(str(tmp_path / "nope.ascii"), 0, 3, 3)
    assert e.value.code == _lib.EG_ERR_OPEN
    with pytest.raises(_lib.EagleGpuError, match="Could not open"):
        api.calculateMMt_rcpp(str(tmp_path / "nope.ascii"), 8, 1, [NA], (3, 3))
    bad = tmp_path / "bad.ascii"
    bad.write_bytes(b"0120\n01X0\n2210\n")
    with pytest.raises(_lib.EagleGpuError, match="no-space ASCII") as e:
        api.calculateMMt_rcpp(str(bad), 8, 1, [NA], (3, 4))
    assert e.value.code == _lib.EG_ERR_FORMAT
    s = synth_small
    with pytest.raises(_lib.EagleGpuError) as e:  # dims swapped: the file size does not fit
        api.calculateMMt_rcpp(s["M"], 8, 1, [NA], (s["n"] + 1, s["L"]))
    assert e.value.code == _lib.EG_ERR_FORMAT
    with pytest.raises(_lib.EagleGpuError) as e:
        api.calculateMMt_rcpp(s["M"], 8, 1, [float(s["L"])], (s["n"], s["L"]))  # locus out of range
    assert e.value.code == _lib.EG_ERR_ARG


# ------------------------------------------------------------------------------- M.Mt
def test_mmt_demo_bit_exact(demo):
    z = demo["z"]
    msgs = []
    MMt = api.calculateMMt_rcpp(demo["M"], 8, 4, [NA], (demo["n"], demo["L"]), quiet=False, message=msgs.append)
    assert hashlib.sha256(MMt.astype("<i4").tobytes()).hexdigest() == str(z["mmt_sha256"])
    assert np.array_equal(MMt, eo.calculateMMt_rcpp(demo["M"], 8, 4, [NA], (demo["n"], demo["L"])))
    assert np.array_equal(MMt, MMt.T) and MMt.dtype == np.float64
    assert msgs and "GPU" in msgs[0]


def test_mmt_selected_loci(synth_small):
    s = synth_small
    dims = (s["n"], s["L"])
    for sel in ([5.0], [5.0, 17.0, 2999.0], [0.0, 0.0, 3000.0]):
        assert np.array_equal(api.calculateMMt_rcpp(s["M"], 8, 1, sel, dims), eo.calculateMMt_rcpp(s["M"], 8, 1, sel, dims))
    # NA anywhere but position 0 is not "none": only element 0 is the sentinel (calculateMMt_rcpp.cpp:88)
    assert np.array_equal(api.calculateMMt_rcpp(s["M"], 8, 1, [NA, 5.0], dims), eo.calculateMMt_rcpp(s["M"], 8, 1, [NA], dims))


def test_mmt_product_is_kept_with_the_resident_store(synth_small):
    """SummaryAM calls calculateMMt_rcpp again with the selected loci (R/summary_am.R:142): the repeat reuses the int32
    product kept with the store (no second contraction) and still equals the oracle for every selection."""
    s = synth_small
    dims = (s["n"], s["L"])
    api.cache_clear()
    first = api.calculateMMt_rcpp(s["M"], 8, 1, [7.0, 1500.0], dims)   # the first call already carries a selection
    assert api.last_timing()["syrk_ms"] > 0
    for sel in ([NA], [7.0, 1500.0], [2.0], [NA]):
        got = api.calculateMMt_rcpp(s["M"], 8, 1, sel, dims)
        assert api.last_timing()["syrk_ms"] == 0.0
        assert np.array_equal(got, eo.calculateMMt_rcpp(s["M"], 8, 1, sel, dims)), sel
    assert np.array_equal(first, eo.calculateMMt_rcpp(s["M"], 8, 1, [7.0, 1500.0], dims))


@pytest.mark.parametrize("n,L", [(1, 1), (1, 200), (2, 127), (3, 128), (129, 129), (128, 4096), (257, 1000),
                                 (300, 5000), (513, 777), (640, 20000)])
def test_mmt_ragged_sizes(tmp_path, n, L):
    G = synth.genotypes(n, L, seed=n * 7919 + L)
    m, _ = write_pair(tmp_path, G, f"r{n}x{L}")
    Gi = G.astype(np.int64) - 1
    got = api.calculateMMt_rcpp(m, 8, 1, [NA], (n, L))
    assert np.array_equal(got, (Gi @ Gi.T).astype(np.float64))


def test_mmt_split_k_and_many_tiles(tmp_path):
    """n small / L large exercises the K split (atomic int32 accumulation); n large the tile table."""
    for n, L in [(150, 300000), (1500, 3000)]:
        G = synth.genotypes(n, L, seed=42)
        m, _ = write_pair(tmp_path, G, f"s{n}")
        Gf = G.astype(np.float32) - 1  # exact in fp32: |entries| <= L < 2^24
        ref = (Gf @ Gf.T).astype(np.float64)
        got = api.calculateMMt_rcpp(m, 8, 1, [NA], (n, L))
        assert np.array_equal(got, ref)
        api.cache_clear()


# ------------------------------------------------------------------------------- scan
def test_scan_demo_against_golden(demo, scan_mode):
    z = demo["z"]
    r = api.calculate_a_and_vara_rcpp(demo["Mt"], [NA], z["it1_S"], z["it1_V"], 8, (demo["L"], demo["n"]), z["it1_hat_a"])
    assert r["a"].shape == (demo["L"], 1) and r["vara"].shape == (demo["L"], 1)
    ca, cv = scan_conds(demo["G"], z["it1_S"], z["it1_V"], z["it1_hat_a"])
    assert_close(r["a"], z["it1_a"], ca, demo["n"], "a")
    assert_close(r["vara"], z["it1_vara"], cv, demo["n"], "vara")
    idx, _ = am.pick_locus(r["a"], r["vara"])
    assert idx == 2207  # columns 2207 and 2209 are identical: the tie must go to the first


def test_scan_synth_with_selected_rows(synth_small, scan_mode):
    s = synth_small
    S, V, a = synth.scan_inputs(s["n"], 3)
    dims = (s["L"], s["n"])
    ca, cv = scan_conds(s["G"], S, V, a)
    for sel in ([NA], [3.0, 2500.0]):
        got = api.calculate_a_and_vara_rcpp(s["Mt"], sel, S, V, 8, dims, a)
        ref = eo.calculate_a_and_vara_rcpp(s["Mt"], sel, S, V, 8, dims, a)
        assert_close(got["a"], ref["a"], ca, s["n"], "a")
        assert_close(got["vara"], ref["vara"], cv, s["n"], "vara")
    assert got["a"][3, 0] == 0 and got["vara"][2500, 0] == 0


def test_scan_asymmetric_inputs_take_the_general_path(synth_small, scan_mode):
    """S and V need not be symmetric for the export: the fast path (upper triangle of W only) is guarded by a
    symmetry check, and the symmetric-half contraction only ever uses W + W^T."""
    s = synth_small
    rng = np.random.default_rng(12)
    n = s["n"]
    S = rng.standard_normal((n, n)) / np.sqrt(n) + 2 * np.eye(n)
    V = rng.standard_normal((n, n)) / np.sqrt(n) + 1.5 * np.eye(n)
    a = rng.standard_normal(n)
    got = api.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 8, (s["L"], n), a)
    ref = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 8, (s["L"], n), a)
    ca, cv = scan_conds(s["G"], S, V, a)
    assert_close(got["a"], ref["a"], ca, n, "a")
    assert_close(got["vara"], ref["vara"], cv, n, "vara")


@pytest.mark.parametrize("n,L", [(1, 5), (31, 1), (127, 300), (128, 257), (129, 1000), (255, 129), (640, 1500)])
def test_scan_ragged_sizes(tmp_path, n, L, scan_mode):
    G = synth.genotypes(n, L, seed=n + L)
    _, mt = write_pair(tmp_path, G, f"q{n}x{L}")
    S, V, a = synth.scan_inputs(n, n)
    got = api.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    ref = npo.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    ca, cv = scan_conds(G, S, V, a)
    assert_close(got["a"], ref["a"], ca, n, "a")
    assert_close(got["vara"], ref["vara"], cv, n, "vara")


@pytest.mark.parametrize("n,L", [(1, 7), (2, 64), (33, 100), (129, 300), (257, 129)])
def test_tiny_shapes_on_the_forced_digit_slice_paths(tmp_path, n, L, monkeypatch):
    """Far below the sizes where they are chosen automatically: pre-products, scan and GEMV all on int8 digit slices."""
    monkeypatch.setenv("EAGLE_PREP_MODE", "i8")
    monkeypatch.setenv("EAGLE_GEMV_MODE", "i8")
    G = synth.genotypes(n, L, seed=3 * n + L)
    _, mt = write_pair(tmp_path, G, f"t{n}x{L}")
    S, V, a = synth.scan_inputs(n, n + 1)
    prev = api.get_scan_mode()
    api.set_scan_mode(1)
    try:
        got = api.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    finally:
        api.set_scan_mode(prev)
    ref = npo.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    ca, cv = scan_conds(G, S, V, a)
    assert_close(got["a"], ref["a"], ca, n, "a")
    assert_close(got["vara"], ref["vara"], cv, n, "vara")


@pytest.mark.parametrize("prep", ["i8", "f64"])
def test_non_finite_inputs_poison_instead_of_passing_silently(synth_small, prep, scan_mode, monkeypatch):
    """A NaN / Inf in S, V or a_hat reaches every marker in the reference's FP64 products (0 * NaN = NaN).  No path,
    integer or floating, may turn it into a finite number: every marker comes back non-finite, as from the oracle.
    (An fmax-based column maximum once dropped the NaNs and returned zeros.)"""
    monkeypatch.setenv("EAGLE_PREP_MODE", prep)
    s = synth_small
    S, V, a = synth.scan_inputs(s["n"], 2)
    dims = (s["L"], s["n"])
    for which, val in (("V", np.nan), ("S", np.inf), ("a", np.nan)):
        S2, V2, a2 = S.copy(), V.copy(), a.copy()
        if which == "V":
            V2[5, 7] = V2[7, 5] = val
        elif which == "S":
            S2[11, 3] = S2[3, 11] = val
        else:
            a2[9] = val
        got = api.calculate_a_and_vara_rcpp(s["Mt"], [NA], S2, V2, 8, dims, a2)
        ref = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S2, V2, 8, dims, a2)
        key = "a" if which == "a" else "vara"
        rbad = ~np.isfinite(ref[key].reshape(-1))
        gbad = ~np.isfinite(got[key].reshape(-1))
        assert rbad.all() and gbad.all(), (which, int(rbad.sum()), int(gbad.sum()))


@pytest.mark.parametrize("digits", [7, 6])
def test_scan_digit_slices_against_extended_precision(tmp_path, digits):
    """With 7 digits the int8 contraction claims one rounding per entry of T = Mt U plus the FP64 row-dot: against an
    80-bit evaluation of the same quantity it must be at least as close as the FP64 restatement is, on inputs with
    columns of very different scale and heavy cancellation.  With 6 digits (opt-in) the columns of U are truncated
    at 2^-48 of their largest entry instead of 2^-56: the bound is 32 x wider, still the size of an FP64 GEMM's
    accumulation error and four orders of magnitude inside the 1e-9 tolerance."""
    n, L = 257, 400
    G = synth.genotypes(n, L, seed=5)
    _, mt = write_pair(tmp_path, G, "xp")
    rng = np.random.default_rng(4)
    d = 2.0 ** rng.integers(-20, 21, n)
    A = rng.standard_normal((n, n))
    S = ((A + A.T) / np.sqrt(n) + 2 * np.eye(n)) * d[:, None] * d[None, :]
    B = rng.standard_normal((n, n))
    V = (B + B.T) / np.sqrt(n) - 0.5 * np.eye(n)                   # indefinite: var(a) sums cancel
    a = rng.standard_normal(n)
    prev, prev_d = api.get_scan_mode(), api.get_scan_digits()
    api.set_scan_mode(1)
    api.set_scan_digits(digits)
    try:
        got = api.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    finally:
        api.set_scan_mode(prev)
        api.set_scan_digits(prev_d)
    ld = np.longdouble
    Ml = (G.T.astype(ld) - 1)
    Wl = S.astype(ld) @ (V.astype(ld) @ S.astype(ld))
    vx = np.einsum("ij,ij->i", Ml @ Wl, Ml)
    ax = Ml @ (S.astype(ld) @ a.astype(ld))
    ref64 = npo.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    _, cv = scan_conds(G, S, V, a)
    e_gpu = np.abs(got["vara"].reshape(-1).astype(ld) - vx).astype(np.float64) / cv
    e_f64 = np.abs(ref64["vara"].reshape(-1).astype(ld) - vx).astype(np.float64) / cv
    print(f"digits {digits}: max error / cond  {e_gpu.max():.3e}   (FP64 restatement {e_f64.max():.3e}, n eps {n * EPS:.3e})")
    if digits == 7:
        assert e_gpu.max() <= 8 * EPS * n                            # a few ulps of the sum of absolute terms
        assert e_gpu.max() <= 4 * max(e_f64.max(), EPS)
    else:
        assert e_gpu.max() <= 32 * 8 * EPS * n                       # 2^-48 instead of 2^-53 per entry
        assert (np.abs(got["vara"].reshape(-1) - ref64["vara"].reshape(-1)) <= 1e-9 * np.abs(ref64["vara"].reshape(-1))
                + 4 * (n + 10) * EPS * cv).all()
    ea = np.abs(got["a"].reshape(-1).astype(ld) - ax).astype(np.float64)
    ca, _ = scan_conds(G, S, V, a)
    assert (ea <= 8 * EPS * n * ca).all()


def test_scan_identical_and_mirrored_markers_are_bit_identical(tmp_path, scan_mode):
    """Tie hazard (SURVEY.md section 4): duplicates / mirror images anywhere in the file must give
    bit-identical tsq, so that the first index wins exactly as in the reference."""
    n, L = 300, 2000
    G = synth.genotypes(n, L, seed=99)
    dup = [(5, 6), (5, 127), (5, 128), (5, 1999), (700, 1413)]
    for src, dst in dup:
        G[:, dst] = G[:, src]
    G[:, 300] = 2 - G[:, 5]  # mirror image: m -> -m
    _, mt = write_pair(tmp_path, G, "dup")
    S, V, a = synth.scan_inputs(n, 1)
    r = api.calculate_a_and_vara_rcpp(mt, [NA], S, V, 8, (L, n), a)
    av, vv = r["a"][:, 0], r["vara"][:, 0]
    for src, dst in dup:
        assert av[src] == av[dst] and vv[src] == vv[dst]
    assert av[300] == -av[5] and vv[300] == vv[5]
    tsq = av ** 2 / vv
    assert tsq[300] == tsq[5] == tsq[1999]


def test_reduced_a_and_extract(synth_small):
    s = synth_small
    rng = np.random.default_rng(5)
    P, y = rng.standard_normal((s["n"], s["n"])), rng.standard_normal(s["n"])
    for sel in ([NA], [10.0, 11.0]):
        got = api.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), sel)
        ref = eo.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), sel)
        assert got.shape == (s["L"], 1)
        cond = 1.7 * (np.abs(s["G"].T.astype(np.float64) - 1) @ (np.abs(P) @ np.abs(y)))
        assert_close(got, ref, cond, s["n"], "ar")
    for col in (0, 1234, s["L"] - 1):
        got = api.extract_geno_rcpp(s["M"], 8, col, (s["n"], s["L"]))
        assert got.dtype == np.int32 and np.array_equal(got, eo.extract_geno_rcpp(s["M"], 8, col, (s["n"], s["L"])))
    with pytest.raises(_lib.EagleGpuError):
        api.extract_geno_rcpp(s["M"], 8, s["L"], (s["n"], s["L"]))


# ------------------------------------------------------------------------------- end to end
def test_forward_search_matches_oracle(demo, scan_mode):
    """Full multi-locus AM() forward search with the GPU library plugged into the restated driver:
    identical selected-QTL sequence, extBIC trace and per-iteration scores."""
    z = demo["z"]
    r = am.AM(api, demo["geno"], z["trait1"], keep_trace=True)
    assert r["selected"] == list(z["am1_selected"]) and r["all_picked"] == list(z["am1_all_picked"])
    np.testing.assert_allclose(r["extBIC"], z["am1_extBIC"], rtol=1e-9)
    ro = am.AM(eo, demo["geno"], z["trait1"], keep_trace=True)
    for tg, to in zip(r["trace"], ro["trace"]):
        assert tg["picked"] == to["picked"]
        ca, cv = scan_conds(demo["G"], to["S"], to["V"], to["hat_a"])
        assert_close(tg["a"], to["a"], ca, demo["n"], "a")
        assert_close(tg["vara"], to["vara"], cv, demo["n"], "vara")
    X0 = np.column_stack([np.ones(demo["n"]), z["pc1"], z["pc2"]])
    r2 = am.AM(api, demo["geno"], z["trait2"], X0=X0)
    assert r2["selected"] == [] and r2["all_picked"] == [1200]


def test_forward_search_synthetic(synth_small, scan_mode):
    s = synth_small
    y, qtl = synth.phenotype(s["G"])
    rg = am.AM(api, s["geno"], y, maxit=6)
    ro = am.AM(eo, s["geno"], y, maxit=6)
    assert rg["all_picked"] == ro["all_picked"] and rg["selected"] == ro["selected"]
    np.testing.assert_allclose(rg["extBIC"], ro["extBIC"], rtol=1e-9)


# ------------------------------------------------------------------------------- stores / shards
def test_store_shards_sum_to_full_and_transpose(synth_small, scan_mode):
    from eagleeverything_b200 import dist as egd
    s = synth_small
    img = synth.ascii_image(s["G"])
    full = api.GenotypeStore.from_host_ascii(img, s["n"], s["L"])
    ref = eo.calculateMMt_rcpp(s["M"], 8, 1, [NA], (s["n"], s["L"]))
    assert np.array_equal(full.mmt(), ref)
    acc = np.zeros_like(ref)
    S, V, a = synth.scan_inputs(s["n"], 3)
    ra, rv = full.transpose().a_and_vara(S, V, a)
    for world in (3,):
        pa, pv = [], []
        for r in range(world):
            c0, c1 = egd.shard_range(s["L"], world, r)
            sh = api.GenotypeStore.from_host_ascii(img, s["n"], s["L"], c0, c1)
            assert sh.info()["cols"] == c1 - c0
            acc += sh.mmt()
            x, v = sh.transpose().a_and_vara(S, V, a)
            pa.append(x)
            pv.append(v)
        assert np.array_equal(acc, ref)
        # marker scores do not depend on the shard a marker lives in: bit-identical
        assert np.array_equal(np.concatenate(pa), ra) and np.array_equal(np.concatenate(pv), rv)
    # Mt decoded from Mt.ascii rows == transpose of the M store
    mt_img = synth.ascii_image(s["G"].T)
    rows = api.GenotypeStore.from_host_rows(mt_img, s["L"], s["n"], 1000, 2000)
    xa, xv = rows.a_and_vara(S, V, a)
    assert np.array_equal(xa, ra[1000:2000]) and np.array_equal(xv, rv[1000:2000])
    assert np.array_equal(full.extract_col(77), s["G"][:, 77].astype(np.int32) - 1)


def test_recycled_device_buffers_are_reused_and_released(synth_small):
    """Freed stores go to an exact-size recycling list (capi.cu pool_alloc): the next store of the same shape gets the same
    block back, and eg_cache_clear hands everything to the driver again."""
    import torch
    n, L = 1500, 40000
    img = synth.ascii_image(synth.genotypes(n, L, seed=3))
    api.cache_clear()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    a = api.GenotypeStore.from_host_ascii(img, n, L)
    pa = a.info()["device_ptr"]
    want = a.mmt()
    a.free()
    b = api.GenotypeStore.from_host_ascii(img, n, L)
    assert b.info()["device_ptr"] == pa
    assert np.array_equal(b.mmt(), want)                      # a recycled (dirty) block decodes to the same store
    bt = b.transpose()
    b.free(); bt.free()
    api.cache_clear()
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info()[0] >= free0 - (64 << 20)


def test_path_cache_sees_a_rewrite_with_the_same_size_and_mtime(tmp_path):
    """Resident stores are keyed by (path, size, mtime, a hash of the first and last 4 KB, dims): a file rewritten in place
    with identical size and timestamp is decoded again, not served from the stale store."""
    import os
    n, L = 40, 300
    G1, G2 = synth.genotypes(n, L, seed=1), synth.genotypes(n, L, seed=2)
    m = str(tmp_path / "M.ascii")
    npo.write_ascii(m, G1)
    st = os.stat(m)
    K1 = api.calculateMMt_rcpp(m, 8, 1, [NA], (n, L))
    npo.write_ascii(m, G2)
    os.utime(m, ns=(st.st_atime_ns, st.st_mtime_ns))
    assert os.stat(m).st_mtime_ns == st.st_mtime_ns and os.stat(m).st_size == st.st_size
    K2 = api.calculateMMt_rcpp(m, 8, 1, [NA], (n, L))
    assert np.array_equal(K2, eo.calculateMMt_rcpp(m, 8, 1, [NA], (n, L))) and not np.array_equal(K1, K2)
