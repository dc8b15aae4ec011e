"""CPU tests: oracle/eagle_oracle.c against the REFERENCE'S OWN hot-path sources.  Their answers are recorded in
tests/golden/reference_calls.json (see tests/reference_record.py); where the sources are compiled (oracle/refshim ->
oracle/_ref/libeagle_ref.so, which build() makes when EAGLE_REFERENCE_SRC names the package's src/ directory) they are
also computed live and checked against the records."""
import numpy as np
import pytest
from reference_record import Approx, close, error_message, fingerprint, reference  # noqa: F401  (fixture)

from eagleeverything_b200 import synth
from oracle import eagle_oracle as eo
from oracle import np_oracle as npo

NA = eo.NA_REAL


def fp(x):
    return fingerprint(x, "")


def scan(*a, keep=()):
    res, br = eo.calculate_a_and_vara_rcpp(*a, return_branch=True)
    return {k: Approx(res[k], keep) for k in ("a", "vara")}, br


def test_readblock_identical(synth_small, reference):
    s = synth_small
    for args in [(s["M"], 0, s["L"], s["n"]), (s["M"], 7, s["L"], 50), (s["Mt"], 100, 60, 9), (s["Mt"], 2999, s["n"], 2)]:
        assert fp(eo.ReadBlock(*args)) == reference(lambda: eo.ReadBlock(*args))
    msg = reference(lambda: error_message(eo.ReadBlock, s["M"] + ".missing", 0, 3, 3))
    assert msg is not None and "ERROR: Could not open" in msg


def test_mmt_identical_in_both_branches(demo, synth_small, reference):
    for d, mems in [(demo, (8, 0.004)), (synth_small, (8, 0.0021))]:
        dims = (d["n"], d["L"])
        for mem in mems:
            for sel in ([NA], [5.0, 17.0, 2999.0]):
                mine, bm = eo.calculateMMt_rcpp(d["M"], mem, 2, sel, dims, return_branch=True)
                ref, br = reference(lambda: eo.calculateMMt_rcpp(d["M"], mem, 2, sel, dims, return_branch=True))
                assert bm == br == (0 if mem == 8 else 1)
                assert fp(mine) == ref, (mem, sel)


def test_scan_matches_reference_code(synth_small, reference):
    s = synth_small
    S, V, a = synth.scan_inputs(s["n"], 3)
    dims = (s["L"], s["n"])
    for sel in ([NA], [3.0, 2500.0]):
        mine, bm = eo.calculate_a_and_vara_rcpp(s["Mt"], sel, S, V, 8, dims, a, return_branch=True)
        ref, br = reference(lambda: scan(s["Mt"], sel, S, V, 8, dims, a))
        assert bm == br == 0
        for k in ("a", "vara"):
            close(mine[k], ref[k], rtol=1e-12, atol=1e-12 * ref[k]["absmax"])
    # negative availmemGb: the reference's in-band soft failure List(a=0, vara=0) (:133-142)
    mine = eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, -1.0, dims, a)
    assert mine == reference(lambda: eo.calculate_a_and_vara_rcpp(s["Mt"], [NA], S, V, -1.0, dims, a)) == {"a": 0, "vara": 0}


def test_scan_blocked_branch_matches_reference_code(tmp_path, reference):
    n, L = 120, 270000  # floor(32 n L / 1e9) = 1 GB "needed" > 0.5 -> 3 row blocks
    G = synth.genotypes(n, L, seed=11)
    mt = str(tmp_path / "Mt.ascii")
    npo.write_ascii(mt, G.T)
    S, V, a = synth.scan_inputs(n, 3)
    sel = [5.0, 130208.0, 269999.0]
    mine, bm = eo.calculate_a_and_vara_rcpp(mt, sel, S, V, 0.5, (L, n), a, return_branch=True)
    ref, br = reference(lambda: scan(mt, sel, S, V, 0.5, (L, n), a, keep=sel))
    assert bm == br == 1
    for k in ("a", "vara"):
        close(mine[k], ref[k], rtol=1e-12, atol=1e-12 * ref[k]["absmax"])
        assert all(ref[k]["values"][ref[k]["idx"].index(int(r))] == 0 for r in sel)


def test_reduced_a_and_extract_match_reference_code(synth_small, reference):
    s = synth_small
    rng = np.random.default_rng(5)
    P, y = rng.standard_normal((s["n"], s["n"])), rng.standard_normal(s["n"])
    for sel in ([NA], [10.0]):
        mine = eo.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), sel)
        ref = reference(lambda: Approx(eo.calculate_reduced_a_rcpp(s["Mt"], 1.7, P, y, 8, (s["n"], s["L"]), sel)))
        close(mine, ref, rtol=1e-12, atol=1e-10)
    for mem in (8, 0.0005):
        for col in (0, 1234, s["L"] - 1):
            mine = eo.extract_geno_rcpp(s["M"], mem, col, (s["n"], s["L"]), return_branch=True)
            assert fp(mine) == reference(lambda: eo.extract_geno_rcpp(s["M"], mem, col, (s["n"], s["L"]), return_branch=True))


@pytest.mark.skipif(not eo.reference_available(), reason="oracle/_ref/libeagle_ref.so not built (build() with EAGLE_REFERENCE_SRC set)")
def test_demo_forward_search_through_reference_code(demo):
    """The restated AM() driver on top of the compiled reference sources reproduces the golden trace."""
    from oracle import am_driver as am
    z = demo["z"]
    with eo.use_reference():
        r = am.AM(eo, demo["geno"], z["trait1"])
    assert r["selected"] == list(z["am1_selected"]) and r["all_picked"] == list(z["am1_all_picked"])
    np.testing.assert_allclose(r["extBIC"], z["am1_extBIC"], rtol=1e-9)
