"""CPU tests: the oracle against the golden fixtures and against itself (two independent
restatements, both branches of every blocked function, a higher-precision bound)."""
import hashlib

import numpy as np
import pytest

from oracle import am_driver as am
from oracle import eagle_oracle as eo
from oracle import np_oracle as npo

NA = eo.NA_REAL


def test_demo_mmt_golden(demo):
    z = demo["z"]
    MMt = eo.calculateMMt_rcpp(demo["M"], 8, 2, [NA], (demo["n"], demo["L"]))
    assert hashlib.sha256(MMt.astype("<i4").tobytes()).hexdigest() == str(z["mmt_sha256"])
    assert np.array_equal(MMt[:4, :4], z["mmt_corner"])
    assert np.trace(MMt) == z["mmt_trace"] == 551356
    assert MMt.sum() == z["mmt_sum"] == 50562338 and MMt.max() == 3815 and MMt.min() == 1950
    assert list(MMt[0, :4]) == [3643, 2351, 2386, 2314]
    assert np.array_equal(MMt, MMt.T)
    # independent numpy restatement gives the same bits (exact integer arithmetic)
    assert np.array_equal(MMt, npo.calculateMMt_rcpp(demo["M"], 8, 2, [NA], (demo["n"], demo["L"])))
    # trace = number of non-heterozygous genotypes
    assert np.trace(MMt) == np.count_nonzero(demo["G"] != 1)


def test_mmt_blocked_branch_and_selected_loci(synth_small):
    s = synth_small
    dims = (s["n"], s["L"])
    full, br0 = eo.calculateMMt_rcpp(s["M"], 8, 2, [NA], dims, return_branch=True)
    blk, br1 = eo.calculateMMt_rcpp(s["M"], 0.0021, 2, [NA], dims, return_branch=True)
    assert (br0, br1) == (0, 1)
    assert np.array_equal(full, blk)
    sel = [5.0, 17.0, 2999.0]
    z0 = eo.calculateMMt_rcpp(s["M"], 8, 2, sel, dims)
    z1 = eo.calculateMMt_rcpp(s["M"], 0.0021, 2, sel, dims)
    G = s["G"].astype(np.float64) - 1
    G[:, [5, 17, 2999]] = 0
    assert np.array_equal(z0, G @ G.T) and np.array_equal(z1, z0)
    assert np.array_equal(z0, npo.calculateMMt_rcpp(s["M"], 8, 2, sel, dims))


def test_readblock_and_extract(synth_small):
    s = synth_small
    B = eo.ReadBlock(s["M"], 7, s["L"], 50)
    assert B.flags.f_contiguous and np.array_equal(B, s["G"][7:57].astype(np.float64) - 1)
    assert np.array_equal(B, npo.ReadBlock(s["M"], 7, s["L"], 50))
    B2 = eo.ReadBlock(s["Mt"], 100, 60, 9)  # fewer columns than the line holds
    assert np.array_equal(B2, s["G"].T[100:109, :60].astype(np.float64) - 1)
    with pytest.raises(eo.OracleError, match="Could not open"):
        eo.ReadBlock(s["M"] + ".missing", 0, 3, 3)
    for col in (0, 1234, s["L"] - 1):
        c0, b0 = eo.extract_geno_rcpp(s["M"], 8, col, (s["n"], s["L"]), return_branch=True)
        c1, b1 = eo.extract_geno_rcpp(s["M"], 0.0005, col, (s["n"], s["L"]), return_branch=True)
        assert (b0, b1) == (0, 1)
        ref = s["G"][:, col].astype(np.int32) - 1
        assert np.array_equal(c0, ref) and np.array_equal(c1, ref)
        assert np.array_equal(npo.extract_geno_rcpp(s["M"], 8, col, (s["n"], s["L"])), ref)


def _scan_inputs(n, seed=3):
    from eagleeverything_b200 import synth
    return synth.scan_inputs(n, seed)


def test_scan_branches_agree_and_match_numpy(synth_small, tmp_path):
    s = synth_small
    S, V, a = _scan_inputs(s["n"])
    dims = (s["L"], s["n"])
    r0, b0 = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 8, dims, a, return_branch=True)
    assert b0 == 0
    rn = npo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 8, dims, a)
    for k in ("a", "vara"):
        assert r0[k].shape == (s["L"], 1)
        np.testing.assert_allclose(r0[k], rn[k], rtol=1e-12, atol=1e-12 * np.abs(rn[k]).max())
    # 4*n*L*8/1e9 truncates to 0 GB here (integer division, :65), so only availmem <= 0 leaves the
    # in-memory branch: negative -> soft failure List(a=0, vara=0) (:133-142); zero -> division by zero
    rneg, b1 = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, -1.0, dims, a, return_branch=True)
    assert b1 == 1 and rneg == {"a": 0, "vara": 0}
    with pytest.raises(eo.OracleError, match="block size 0"):
        eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 0.0, dims, a)


def test_scan_blocked_branch(tmp_path):
    """The blocked branch (:117-234) needs floor(32*n*L/1e9) >= 1: n=120, L=270000, availmem=0.5 -> 3 blocks."""
    from eagleeverything_b200 import synth
    n, L = 120, 270000
    G = synth.genotypes(n, L, seed=11)
    mt = str(tmp_path / "Mt.ascii")
    npo.write_ascii(mt, G.T)
    S, V, a = _scan_inputs(n)
    sel = [5.0, 130208.0, 269999.0]  # one selected row in each block (block = 130208 rows)
    rb, b = eo.calculate_a_and_vara_rcpp(mt, sel, S, V, 0.5, (L, n), a, return_branch=True)
    ri, bi = eo.calculate_a_and_vara_rcpp(mt, sel, S, V, 8, (L, n), a, return_branch=True)
    assert (b, bi) == (1, 0)
    for k in ("a", "vara"):
        np.testing.assert_allclose(rb[k], ri[k], rtol=1e-13, atol=0)
        assert all(rb[k][int(r), 0] == 0 for r in sel)


def test_scan_selected_rows_zeroed(synth_small):
    s = synth_small
    S, V, a = _scan_inputs(s["n"])
    r = eo.calculate_a_and_vara_rcpp(s["Mt"], [3.0, 2500.0], S, V, 8, (s["L"], s["n"]), a)
    assert r["a"][3, 0] == 0 and r["vara"][3, 0] == 0 and r["a"][2500, 0] == 0 and r["vara"][2500, 0] == 0
    r0 = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 8, (s["L"], s["n"]), a)
    keep = np.ones(s["L"], bool)
    keep[[3, 2500]] = False
    assert np.array_equal(r["a"][keep], r0["a"][keep]) and np.array_equal(r["vara"][keep], r0["vara"][keep])


def test_scan_against_longdouble(synth_small):
    s = synth_small
    S, V, a = _scan_inputs(s["n"])
    r = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, 8, (s["L"], s["n"]), a)
    rows = [0, 1, 77, 1500, s["L"] - 1]
    Mt = (s["G"].T.astype(np.int8) - 1)
    la, lv = npo.a_and_vara_longdouble(Mt, S, V, a, rows)
    np.testing.assert_allclose(r["a"][rows, 0], la.astype(np.float64), rtol=1e-11)
    np.testing.assert_allclose(r["vara"][rows, 0], lv.astype(np.float64), rtol=1e-11)


def test_reduced_a_equals_direct_form(synth_small):
    s = synth_small
    rng = np.random.default_rng(5)
    P = rng.standard_normal((s["n"], s["n"]))
    y = rng.standard_normal(s["n"])
    ar = eo.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), [NA])
    Mt = s["G"].T.astype(np.float64) - 1
    np.testing.assert_allclose(ar[:, 0], 1.7 * (Mt @ (P @ y)), rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(ar, npo.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), [NA]),
                               rtol=1e-12, atol=1e-10)
    arz = eo.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), [10.0])
    assert arz[10, 0] == 0 and np.array_equal(np.delete(arz, 10, 0), np.delete(ar, 10, 0))


def test_am_forward_search_golden(demo):
    z = demo["z"]
    r = am.AM(eo, demo["geno"], z["trait1"], keep_trace=True)
    assert r["selected"] == list(z["am1_selected"]) == [2207, 4503, 873]
    assert r["all_picked"] == list(z["am1_all_picked"]) == [2207, 4503, 873, 2874]
    np.testing.assert_allclose(r["extBIC"], z["am1_extBIC"], rtol=1e-9)
    np.testing.assert_allclose(r["extBIC"], [925.742, 887.799, 886.762, 885.097, 889.442], atol=2e-3)
    t0 = r["trace"][0]
    np.testing.assert_allclose(t0["a"], z["it1_a"], rtol=1e-9, atol=1e-9)
    # The n x n algebra before the scan runs through numpy's multi-threaded LAPACK / BLAS, so S and V carry rounding that
    # depends on the host's thread count.  The scan itself is reproducible: at the stored first-iteration inputs it
    # must give the stored a / var(a); the search's own var(a) may differ from them by what its S, V differences
    # propagate (|m|' |W - W_stored| |m|) plus the contraction's rounding -- var(a) of monomorphic markers is 0 up to
    # exactly that noise.
    n, L = demo["n"], demo["L"]
    S0, V0, h0 = z["it1_S"], z["it1_V"], z["it1_hat_a"]
    scan0 = eo.calculate_a_and_vara_rcpp(demo["Mt"], [NA], S0, V0, 8, (L, n), h0)
    np.testing.assert_allclose(scan0["a"][:, 0], z["it1_a"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(scan0["vara"][:, 0], z["it1_vara"], rtol=1e-9, atol=1e-9)
    for k in ("S", "V", "hat_a"):
        np.testing.assert_allclose(t0[k], z["it1_" + k], rtol=0, atol=1e-9 * np.abs(z["it1_" + k]).max())
    Mabs = np.abs(demo["G"].astype(np.float64) - 1)
    W, W0 = t0["S"] @ t0["V"] @ t0["S"], S0 @ V0 @ S0
    drift = np.einsum("ij,ij->j", Mabs, np.abs(W - W0) @ Mabs)
    rounding = 4 * (n + 10) * np.finfo(np.float64).eps * np.einsum("ij,ij->j", Mabs, np.abs(W) @ Mabs)
    assert (np.abs(t0["vara"] - z["it1_vara"]) <= 1e-9 * np.abs(z["it1_vara"]) + 1e-9 + drift + rounding).all()
    np.testing.assert_allclose(t0["a"][:3], [28.8059, -12.3227, -40.3413], atol=1e-3)
    # the tie hazard: demo columns 2207 and 2209 are identical, their tsq tie and the first wins
    assert np.array_equal(demo["G"][:, 2206], demo["G"][:, 2208])
    assert t0["tsq"][2206] == t0["tsq"][2208] == np.nanmax(t0["tsq"])


def test_am_covariates_golden(demo):
    z = demo["z"]
    X0 = np.column_stack([np.ones(demo["n"]), z["pc1"], z["pc2"]])
    r = am.AM(eo, demo["geno"], z["trait2"], X0=X0)
    assert r["selected"] == [] and r["all_picked"] == [1200]
    np.testing.assert_allclose(r["extBIC"], z["am2_extBIC"], rtol=1e-9)


def test_pick_locus_semantics():
    a = np.array([1.0, 2.0, 2.0, np.nan, 0.0])
    v = np.array([1.0, 1.0, 1.0, 1.0, 0.0])  # last: 0/0 = NaN, ignored
    idx, tsq = am.pick_locus(a, v)
    assert idx == 2 and np.isnan(tsq[3]) and np.isnan(tsq[4])
    idx, _ = am.pick_locus(np.array([1.0, 3.0]), np.array([1.0, 0.0]))  # +Inf is kept by max(na.rm=TRUE)
    assert idx == 2
