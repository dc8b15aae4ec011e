"""Ingest side (SURVEY.md section 8(f) rank 3): createM_ASCII_rcpp (text files -> no-space ASCII, reference
src/createM_ASCII_rcpp.cpp:19-106 + src/CreateASCIInospace.cpp:17-164) and createMt_ASCII_rcpp (M.ascii -> Mt.ascii,
src/createMt_ASCII_rcpp.cpp:15-245).

CPU tests: oracle/eagle_oracle.c against the reference's own sources (file bytes, return value and every message), as
recorded in tests/golden/reference_calls.json and, where they are compiled through oracle/refshim, live.  GPU tests:
the device tokeniser / encoder through the C ABI against the oracle, byte for byte."""
import hashlib
import os

import numpy as np
import pytest

from eagleeverything_b200 import synth
from oracle import eagle_oracle as eo
from oracle import np_oracle as npo
from reference_record import error_message, fingerprint, reference  # noqa: F401  (fixture)


def write_text(path, G, codes=("0", "1", "2"), missing=None, miss_at=(), style=0, final_newline=True, seed=0):
    """A marker text file the way users write them: tokens separated by whitespace.  style 0: single spaces;
    1: tabs; 2: ragged runs of blanks/tabs with leading and trailing blanks; 3: CR LF line ends."""
    rng = np.random.default_rng(seed)
    miss = set(miss_at)
    lines = []
    for r in range(G.shape[0]):
        toks = [missing if (r, c) in miss else codes[int(g)] for c, g in enumerate(G[r])]
        if style == 0:
            line = " ".join(toks)
        elif style == 1:
            line = "\t".join(toks)
        elif style == 2:
            seps = [" ", "  ", "\t", " \t ", "   "]
            line = seps[r % 5] + "".join(t + seps[int(rng.integers(5))] for t in toks)
        else:
            line = " ".join(toks) + "\r"
        lines.append(line)
    text = "\n".join(lines) + ("\n" if final_newline else "")
    with open(path, "wb") as f:
        f.write(text.encode())
    return text


def cases(tmp):
    """(name, input path, dims, AA, AB, BB, missing, expect_ok, expected image or None)"""
    out = []

    def add(name, G, ok=True, mutate=None, dims=None, AA="0", AB="1", BB="2", missing="NA", **kw):
        p = os.path.join(tmp, name + ".txt")
        codes = (AA, AB if AB != "NA" else "1", BB)
        write_text(p, G, codes=codes, missing=missing, **kw)
        if mutate:
            b = bytearray(open(p, "rb").read())
            b = mutate(b)
            open(p, "wb").write(bytes(b))
        want = G.copy()
        for (r, c) in kw.get("miss_at", ()):
            want[r, c] = 1
        out.append((name, p, dims or G.shape, AA, AB, BB, missing, ok, synth.ascii_image(want) if ok else None))

    G = synth.genotypes(23, 157, seed=3)
    add("plain", G)
    add("tabs", G, style=1)
    add("ragged_blanks", G, style=2, seed=5)
    add("crlf", G, style=3)
    add("no_final_newline", G, final_newline=False)
    add("letters", G, AA="AA", AB="AB", BB="BB", missing="-")
    add("letters_missing", G, AA="AA", AB="AB", BB="BB", missing="-", miss_at=[(0, 0), (7, 100), (22, 156)], style=2)
    add("long_codes", G, AA="homA", AB="het", BB="homozygousB", missing="NA", miss_at=[(3, 3)])
    add("prefix_codes", G, AA="A", AB="AB", BB="ABB", missing="ABBA", miss_at=[(1, 1), (2, 2)])   # codes that prefix each other
    add("no_het_code", synth.genotypes(9, 40, seed=4) // 2 * 2, AB="NA", missing="NA")           # inbreds: AB = NA
    add("one_column", synth.genotypes(40, 1, seed=6))
    add("one_row", synth.genotypes(1, 300, seed=7), final_newline=False)
    big = synth.genotypes(37, 9000, seed=8)                                                        # > 16 chunks of 32 KB
    add("many_chunks", big, style=2, seed=9)
    # ---- failures the reference reports in-band
    add("bad_token_first", G, ok=False, mutate=lambda b: b.replace(b"0", b"7", 1))
    add("bad_token_late", big, ok=False, mutate=lambda b: b[:-2000] + b[-2000:].replace(b"1", b"x", 1))
    add("bad_token_joined", G, ok=False, mutate=lambda b: b.replace(b"0 1", b"01", 1))           # "01": no such code
    add("bad_token_no_het", synth.genotypes(9, 40, seed=4) // 2 * 2, ok=False, AB="NA",
        mutate=lambda b: b[:60] + b[60:].replace(b"0", b"Q", 1))
    add("short_row", G, ok=False, mutate=lambda b: b[:b.index(b"\n", 2000) - 2] + b[b.index(b"\n", 2000):])
    add("long_row", G, ok=False, mutate=lambda b: b[:b.index(b"\n", 900)] + b" 2" + b[b.index(b"\n", 900):])
    add("empty_line", G, ok=False, mutate=lambda b: b[:b.index(b"\n", 1200)] + b"\n" + b[b.index(b"\n", 1200):])
    add("blank_tail", G, ok=False, mutate=lambda b: b + b"  ")                                    # getline returns "  ": 0 columns
    add("short_last_row_unterminated", G, ok=False, final_newline=False, mutate=lambda b: b[:-2])
    add("wrong_dims", G, ok=False, dims=(23, 156))
    add("bad_token_before_short_row", G, ok=False,
        mutate=lambda b: (b[:b.index(b"\n", 1500) - 6] + b"Z" + b[b.index(b"\n", 1500) - 5: b.index(b"\n", 1500) - 2] +
                          b[b.index(b"\n", 1500):]))
    return out


@pytest.fixture(scope="module")
def ingest_cases(tmp_path_factory):
    return cases(str(tmp_path_factory.mktemp("ingest")))


def run_oracle(case, out_path, quiet=False):
    name, p, dims, AA, AB, BB, missing, ok, want = case
    got_ok, msgs = eo.createM_ASCII_rcpp(p, out_path, "text", AA, AB, BB, 8.0, dims, quiet, missing)
    return got_ok, msgs, open(out_path, "rb").read()


def test_oracle_tokeniser_known_answers(ingest_cases, tmp_path):
    for case in ingest_cases:
        ok, msgs, data = run_oracle(case, str(tmp_path / "o.ascii"))
        assert ok == case[7], case[0]
        if ok:
            assert data == case[8].tobytes(), case[0]
            assert msgs[0] == " A text file is being assumed as the input data file type. "
            assert msgs[-1 - min(5, case[2][0])].startswith(" First ")
    by = {c[0]: c for c in ingest_cases}
    ok, msgs, data = run_oracle(by["short_row"], str(tmp_path / "o.ascii"), quiet=True)
    row = open(by["short_row"][1], "rb").read()[:2000].count(b"\n") + 1
    assert msgs[2] == f"        The error has occurred at row {row} which contains 156 but " and len(data) == (row - 1) * 158
    ok, msgs, _ = run_oracle(by["bad_token_first"], str(tmp_path / "o.ascii"), quiet=True)
    assert msgs[1] == " For example , 7 in row 1" and "AA=0 AB=1 BB=2" in msgs[0]
    ok, msgs, _ = run_oracle(by["bad_token_no_het"], str(tmp_path / "o.ascii"), quiet=True)
    assert msgs[0].endswith("different to AA=0 BB=2")
    ok, msgs = eo.createM_ASCII_rcpp(str(tmp_path / "absent.txt"), str(tmp_path / "o.ascii"), "text", "0", "1", "2", 8, (3, 3), True, "NA")
    assert not ok and msgs == ["ERROR: Text file could not be opened with filename  " + str(tmp_path / "absent.txt") + "\n"]


def test_oracle_ingest_matches_reference_code(ingest_cases, tmp_path, demo, reference):
    tmp = reference.tmp
    for case in ingest_cases:
        for quiet in (False, True):
            mine = fingerprint(run_oracle(case, str(tmp_path / "mine.ascii"), quiet), tmp)
            if case[0] == "long_row":      # the reference writes beyond its row buffer here (CreateASCIInospace.cpp:85): same
                ref = reference(lambda: run_oracle(case, str(tmp_path / "ref.ascii"), quiet)[:2])
                assert mine[:2] == ref     # verdict and messages, file content undefined
                continue
            assert mine == reference(lambda: run_oracle(case, str(tmp_path / "ref.ascii"), quiet)), (case[0], quiet)
    # createMt: both situations of the reference write the same bytes; messages but for the two formatted doubles
    for d, mems in ((demo, (8.0, 0.002)), ):
        dims = (d["n"], d["L"])
        for mem in mems:
            for quiet in (False, True):
                m1 = eo.createMt_ASCII_rcpp(d["M"], str(tmp_path / "mine.Mt"), "text", mem, dims, quiet)
                m2, ref_bytes = reference(lambda: (eo.createMt_ASCII_rcpp(d["M"], str(tmp_path / "ref.Mt"), "text", mem, dims, quiet),
                                                   open(tmp_path / "ref.Mt", "rb").read()))
                assert fingerprint(open(tmp_path / "mine.Mt", "rb").read(), tmp) == ref_bytes == fingerprint(open(d["Mt"], "rb").read(), tmp)
                assert fingerprint(m1, tmp) == m2, (mem, quiet)
                assert (len(m1) > 10) == (mem < 1 and not quiet)   # the block situation announces itself


# ---------------------------------------------------------------------------------------------------- PLINK ped files
def write_ped(path, A, sep=" ", final_newline=True, crlf=False):
    """A: (rows, nsnp, 2) array of single-character alleles; six leading ped fields per line."""
    lines = []
    for r in range(A.shape[0]):
        head = [f"FAM{r // 3}", f"ind{r}", "0", "0", str(1 + r % 2), f"{r * 0.5:.1f}"]
        lines.append(sep.join(head + [chr(c) for c in A[r].reshape(-1)]) + ("\r" if crlf else ""))
    with open(path, "wb") as f:
        f.write(("\n".join(lines) + ("\n" if final_newline else "")).encode())


def ped_alleles(rows, nsnp, seed, missing=0.0, mono=0.1):
    rng = np.random.default_rng(seed)
    pairs = [(a, b) for a in "ACGT12" for b in "ACGT12" if a != b]
    A = np.empty((rows, nsnp, 2), np.uint8)
    for i in range(nsnp):
        a, b = pairs[int(rng.integers(len(pairs)))]
        if rng.random() < mono:
            b = a
        f = 0.1 + 0.8 * rng.random()
        A[:, i, :] = np.where(rng.random((rows, 2)) < f, ord(a), ord(b))
    if missing:
        m = rng.random((rows, nsnp)) < missing
        kind = rng.integers(4, size=(rows, nsnp))
        A[:, :, 0] = np.where(m & (kind != 1), np.where(kind == 3, ord("-"), ord("0")), A[:, :, 0])
        A[:, :, 1] = np.where(m & (kind != 0), np.where(kind == 3, ord("-"), ord("0")), A[:, :, 1])
    return A


def ped_cases(tmp):
    out = []

    def add(name, A, ok=True, mutate=None, dims=None, **kw):
        p = os.path.join(tmp, name + ".ped")
        write_ped(p, A, **kw)
        if mutate:
            b = mutate(bytearray(open(p, "rb").read()))
            open(p, "wb").write(bytes(b))
        out.append((name, p, dims or (A.shape[0], 6 + 2 * A.shape[1]), ok))

    def third(A, row, snp, later=()):
        B = A.copy()
        B[row, snp, 1] = ord("Z")
        for (r, s_) in later:
            B[r, s_, 0] = ord("Y")
        return B

    A = ped_alleles(31, 211, 1)
    add("ped_plain", A)
    add("ped_tabs_crlf", A, sep="\t", crlf=True)
    add("ped_no_final_newline", A, final_newline=False)
    add("ped_missing", ped_alleles(31, 211, 2, missing=0.05))
    first_missing = ped_alleles(17, 64, 3, missing=0.02)
    first_missing[0, :20, :] = ord("0")                        # the first row initialises the allele table with 'I'
    first_missing[1, :10, 0] = ord("-")
    add("ped_first_rows_missing", first_missing)
    indel = ped_alleles(12, 40, 4)
    indel[:, 5, :] = np.where(np.random.default_rng(0).random((12, 2)) < 0.5, ord("I"), ord("D"))   # 'I' is the missing mark
    add("ped_indel_I_allele", indel)
    add("ped_one_snp", ped_alleles(9, 1, 5))
    wide = ped_alleles(40, 9000, 6, missing=0.01)              # 36 KB per line: lines span tokeniser chunks
    add("ped_wide", wide)
    mono_then_new = ped_alleles(10, 8, 7, mono=1.0)
    mono_then_new[6:, 3, :] = ord("T") if mono_then_new[0, 3, 0] != ord("T") else ord("G")           # second allele appears late
    add("ped_late_second_allele", mono_then_new)
    # ---- failures
    full = ped_alleles(31, 211, 8, mono=0.0)
    add("ped_third_allele", third(full, 20, 100, later=[(20, 150), (25, 3)]), ok=False)
    add("ped_third_allele_row0", third(full, 0, 0), ok=False)          # A B in row 0, then Z: needs a row where both are known
    add("ped_third_allele_after_missing", third(ped_alleles(31, 211, 9, missing=0.05, mono=0.0), 29, 210), ok=False)
    add("ped_short_row", full, ok=False, mutate=lambda b: b[:b.index(b"\n", 6000) - 2] + b[b.index(b"\n", 6000):])
    add("ped_short_row_after_third_allele", third(full, 3, 7), ok=False,
        mutate=lambda b: b[:b.index(b"\n", 6000) - 2] + b[b.index(b"\n", 6000):])
    add("ped_third_allele_after_short_row", third(full, 30, 7), ok=False,
        mutate=lambda b: b[:b.index(b"\n", 6000) - 2] + b[b.index(b"\n", 6000):])
    add("ped_empty_line", full, ok=False, mutate=lambda b: b[:b.index(b"\n", 3000)] + b"\n" + b[b.index(b"\n", 3000):])
    add("ped_wrong_dims", full, ok=False, dims=(31, 6 + 2 * 210))
    return out


@pytest.fixture(scope="module")
def plink_cases(tmp_path_factory):
    return ped_cases(str(tmp_path_factory.mktemp("ped")))


def run_oracle_ped(case, out_path, quiet=False):
    name, p, dims, ok = case
    got_ok, msgs = eo.createM_ASCII_rcpp(p, out_path, "PLINK", "", "", "", 8.0, dims, quiet, "")
    return got_ok, msgs, open(out_path, "rb").read()


def test_oracle_plink_known_answers(plink_cases, tmp_path):
    by = {c[0]: c for c in plink_cases}
    for case in plink_cases:
        ok, msgs, data = run_oracle_ped(case, str(tmp_path / "o.ascii"))
        assert ok == case[3], case[0]
    # a hand-checked file: SNP 1 A/G, SNP 2 monomorphic then a new allele, SNP 3 with a missing call
    p = str(tmp_path / "tiny.ped")
    open(p, "w").write("f i1 0 0 1 0  A A  C C  T T\nf i2 0 0 1 0  A G  C C  0 T\nf i3 0 0 1 0  G G  T T  G G\n")
    ok, msgs, data = run_oracle_ped(("tiny", p, (3, 12), True), str(tmp_path / "o.ascii"))
    assert ok and data == b"000\n101\n222\n" and any("missing alleles" in m for m in msgs)
    ok, msgs, data = run_oracle_ped(by["ped_third_allele"], str(tmp_path / "o.ascii"))
    assert "        The error has occurred at snp locus 101 for individual 21" in msgs and len(data) == 20 * 212
    ok, msgs, data = run_oracle_ped(by["ped_short_row_after_third_allele"], str(tmp_path / "o.ascii"))
    assert "        The error has occurred at snp locus 8 for individual 4" in msgs
    ok, msgs, data = run_oracle_ped(by["ped_third_allele_after_short_row"], str(tmp_path / "o.ascii"))
    assert any("unequal number of columns" in m for m in msgs) and not any("more than two alleles" in m for m in msgs)


def test_oracle_plink_matches_reference_code(plink_cases, tmp_path, reference):
    tmp = reference.tmp
    for case in plink_cases:
        mine = run_oracle_ped(case, str(tmp_path / "mine.ascii"))
        assert fingerprint(mine, tmp) == reference(lambda: run_oracle_ped(case, str(tmp_path / "ref.ascii"))), case[0]
    # multi-character allele tokens: the reference reads them character by character; so does the restatement
    p = str(tmp_path / "multi.ped")
    open(p, "w").write("f i1 0 0 1 0 AC G T T\nf i2 0 0 1 0 A C GT T\n")
    case = ("multi", p, (2, 10), True)
    mine = run_oracle_ped(case, str(tmp_path / "mine.ascii"))
    assert fingerprint(mine, tmp) == reference(lambda: run_oracle_ped(case, str(tmp_path / "ref.ascii")))
    mine = eo.createM_ASCII_rcpp(str(tmp_path / "absent.ped"), str(tmp_path / "o"), "PLINK", "", "", "", 8, (2, 10), True, "")
    ref = reference(lambda: eo.createM_ASCII_rcpp(str(tmp_path / "absent.ped"), str(tmp_path / "o"), "PLINK", "", "", "", 8, (2, 10), True, ""))
    assert fingerprint(mine, tmp) == ref and not mine[0] and len(mine[1]) == 2


# ---------------------------------------------------------------------------------------------------- ReshapeM, getRowColumn
RESHAPE_CASES = [[], [5], [202], [0], [150, 77, 3], [202, 201, 0], [7, 7], [3, 77, 150], [10, 10, 9]]   # the last three: not decreasing


def _reshape_files(tmp_path, synth_small, tag):
    import shutil
    m, mt = str(tmp_path / f"M{tag}.ascii"), str(tmp_path / f"Mt{tag}.ascii")
    shutil.copy(synth_small["M"], m)
    shutil.copy(synth_small["Mt"], mt)
    return m, mt


def test_oracle_reshape_and_rowcolumn_known_answers(synth_small, tmp_path, ingest_cases):
    s = synth_small
    m, mt = _reshape_files(tmp_path, s, "o")
    assert eo.ReshapeM_rcpp(m, mt, [150, 77, 3], (s["n"], s["L"])) == [s["n"] - 3, s["L"]]
    keep = [i for i in range(s["n"]) if i not in (3, 77, 150)]
    assert open(m + "tmp", "rb").read() == synth.ascii_image(s["G"][keep]).tobytes()
    assert open(mt + "tmp", "rb").read() == synth.ascii_image(s["G"][keep].T.copy()).tobytes()
    by = {c[0]: c for c in ingest_cases}
    assert eo.getRowColumn(by["plain"][1]) == [23, 157] and eo.getRowColumn(by["no_final_newline"][1]) == [23, 157]
    assert eo.getRowColumn(by["ragged_blanks"][1]) == [23, 157] and eo.getRowColumn(by["blank_tail"][1]) == [24, 157]
    assert eo.getRowColumn(s["M"]) == [s["n"], 1]


def test_oracle_reshape_and_rowcolumn_match_reference_code(synth_small, tmp_path, ingest_cases, plink_cases, reference):
    s = synth_small
    for k, idx in enumerate(RESHAPE_CASES):
        m1, mt1 = _reshape_files(tmp_path, s, f"a{k}")
        m2, mt2 = _reshape_files(tmp_path, s, f"b{k}")
        mine = reshape_and_read(m1, mt1, idx, (s["n"], s["L"]))
        assert fingerprint(mine, "") == reference(lambda: reshape_and_read(m2, mt2, idx, (s["n"], s["L"]))), idx
    for case in list(ingest_cases) + list(plink_cases):
        assert eo.getRowColumn(case[1]) == reference(lambda: eo.getRowColumn(case[1])), case[0]
    msg = reference(lambda: error_message(eo.getRowColumn, str(tmp_path / "absent")))
    assert msg is not None and "ERROR: Could not open" in msg


def reshape_and_read(m, mt, idx, dims):
    """ReshapeM_rcpp's return value and the two files it writes."""
    return eo.ReshapeM_rcpp(m, mt, idx, dims), open(m + "tmp", "rb").read(), open(mt + "tmp", "rb").read()


@pytest.mark.gpu
def test_gpu_reshape_and_rowcolumn_match_oracle(api, synth_small, tmp_path, ingest_cases, plink_cases, monkeypatch):
    s = synth_small
    dims = (s["n"], s["L"])
    for k, idx in enumerate(RESHAPE_CASES):
        m1, mt1 = _reshape_files(tmp_path, s, f"g{k}")
        m2, mt2 = _reshape_files(tmp_path, s, f"r{k}")
        assert api.ReshapeM_rcpp(m1, mt1, idx, dims) == eo.ReshapeM_rcpp(m2, mt2, idx, dims), idx
        assert open(m1 + "tmp", "rb").read() == open(m2 + "tmp", "rb").read(), idx
        assert open(mt1 + "tmp", "rb").read() == open(mt2 + "tmp", "rb").read(), idx
    # the reshaped stores serve the calls AM() makes on the two new files (R/AM.R:353-370)
    n1 = s["n"] - 3
    m, mt = _reshape_files(tmp_path, s, "chain")
    assert api.ReshapeM_rcpp(m, mt, [150, 77, 3], dims) == [n1, s["L"]]
    assert np.array_equal(api.calculateMMt_rcpp(m + "tmp", 8.0, 1, [api.NA_REAL], (n1, s["L"])),
                          eo.calculateMMt_rcpp(m + "tmp", 8.0, 1, [eo.NA_REAL], (n1, s["L"])))
    S, V, a = synth.scan_inputs(n1, 3)
    got = api.calculate_a_and_vara_rcpp(mt + "tmp", [api.NA_REAL], S, V, 8.0, (s["L"], n1), a)
    want = eo.calculate_a_and_vara_rcpp(mt + "tmp", [eo.NA_REAL], S, V, 8.0, (s["L"], n1), a)
    np.testing.assert_allclose(got["vara"], want["vara"], rtol=1e-9, atol=1e-12 * np.abs(want["vara"]).max())
    np.testing.assert_allclose(got["a"], want["a"], rtol=1e-9, atol=1e-12 * np.abs(want["a"]).max())
    with pytest.raises(Exception, match="Could not open"):
        api.ReshapeM_rcpp(str(tmp_path / "absent"), mt, [1], dims)
    with pytest.raises(Exception, match="beyond a line"):
        api.ReshapeM_rcpp(m, mt, [s["n"] + 5], dims)
    for piece in (None, 1000):
        if piece:
            monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(piece))
        for case in list(ingest_cases) + list(plink_cases):
            assert api.getRowColumn(case[1]) == eo.getRowColumn(case[1]), case[0]
    with pytest.raises(Exception, match="ERROR: Could not open"):
        api.getRowColumn(str(tmp_path / "absent"))


# ---------------------------------------------------------------------------------------------------- seeded fuzz
SEPS = [" ", "  ", "\t", " \t", "\r", "\v", "\f", "   \t  "]


def fuzz_text_case(rng, path):
    """A random marker text file: random codes (1-3 characters, possibly equal or prefixes of each other), random blank runs,
    and -- in half of the cases -- one defect (foreign token, short / long / blank row, missing final newline)."""
    alpha = list("012ABHN-x")
    code = lambda: "".join(rng.choice(alpha, size=int(rng.integers(1, 4))))
    AA, AB, BB, missing = code(), code(), code(), code()
    if rng.random() < 0.15:
        AB = "NA"
    rows, cols = int(rng.integers(1, 30)), int(rng.integers(1, 40))
    lines = []
    for r in range(rows):
        toks = [str(rng.choice([AA, AB if AB != "NA" else AA, BB, missing], p=[0.4, 0.25, 0.25, 0.1])) for _ in range(cols)]
        lead = str(rng.choice(["", " ", "\t "]))
        lines.append(lead + "".join(t + str(rng.choice(SEPS)) for t in toks).rstrip(" ") if rng.random() < 0.5 else
                     lead + str(rng.choice(SEPS[:3])).join(toks))
    defect = rng.random()
    r = int(rng.integers(rows))
    if defect < 0.12:
        lines[r] = lines[r] + " " + str(rng.choice(["zz", "3", AA + BB + "q"]))           # one token too many (maybe foreign)
    elif defect < 0.24:
        parts = lines[r].split()
        lines[r] = " ".join(parts[:-1])                                                   # one token short (maybe empty line)
    elif defect < 0.36:
        parts = lines[r].split()
        parts[int(rng.integers(len(parts)))] = str(rng.choice(["?", "22x", AA + "_"]))
        lines[r] = " ".join(parts)                                                        # a foreign token
    elif defect < 0.42:
        lines.insert(r, "")                                                               # an empty line
    text = "\n".join(lines) + ("" if rng.random() < 0.25 else "\n") + ("  " if rng.random() < 0.05 else "")
    with open(path, "wb") as f:
        f.write(text.encode("latin-1"))
    return (rows, cols), AA, AB, BB, missing


def fuzz_ped_case(rng, path):
    rows, nsnp = int(rng.integers(1, 14)), int(rng.integers(1, 24))
    pool = list("ACGT12")
    lines = []
    al = [(str(rng.choice(pool)), str(rng.choice(pool))) for _ in range(nsnp)]
    for r in range(rows):
        toks = [f"F{r}", f"I{r}", "0", "0", "1", "-9"]
        for i in range(nsnp):
            for _ in range(2):
                u = rng.random()
                toks.append("0" if u < 0.04 else "-" if u < 0.06 else "I" if u < 0.08 else
                            str(rng.choice(pool)) if u < 0.085 else al[i][int(rng.integers(2))])
        sep = str(rng.choice([" ", "\t", "  "]))
        lines.append(sep.join(toks))
    if rng.random() < 0.15:
        r = int(rng.integers(rows))
        lines[r] = lines[r] + " A" if rng.random() < 0.5 else " ".join(lines[r].split()[:-1])
    with open(path, "wb") as f:
        f.write(("\n".join(lines) + ("" if rng.random() < 0.2 else "\n")).encode())
    return (rows, 6 + 2 * nsnp)


def test_oracle_ingest_fuzz_against_reference_code(tmp_path, reference):
    rng = np.random.default_rng(2026)
    p = str(tmp_path / "f.txt")
    n_bad = 0
    read = lambda name: open(tmp_path / name, "rb").read()
    for k in range(300):
        dims, AA, AB, BB, missing = fuzz_text_case(rng, p)
        mine = eo.createM_ASCII_rcpp(p, str(tmp_path / "a"), "text", AA, AB, BB, 8.0, dims, True, missing)
        too_long = not mine[0] and any("which contains" in m and int(m.split("contains")[1].split()[0]) > dims[1] for m in mine[1])
        # beyond dims[1] tokens the reference writes outside its row buffer: file content undefined
        ref = reference(lambda: (eo.createM_ASCII_rcpp(p, str(tmp_path / "b"), "text", AA, AB, BB, 8.0, dims, True, missing),
                                 None if too_long else read("b")), digest=True)
        assert reference.fp((mine, None if too_long else read("a")), digest=True) == ref, (k, open(p, "rb").read())
        n_bad += not mine[0]
        assert eo.getRowColumn(p) == reference(lambda: eo.getRowColumn(p))
    assert 60 < n_bad < 240
    for k in range(200):
        dims = fuzz_ped_case(rng, p)
        mine = eo.createM_ASCII_rcpp(p, str(tmp_path / "a"), "PLINK", "", "", "", 8.0, dims, True, "")
        ref = reference(lambda: (eo.createM_ASCII_rcpp(p, str(tmp_path / "b"), "PLINK", "", "", "", 8.0, dims, True, ""), read("b")),
                        digest=True)
        assert reference.fp((mine, read("a")), digest=True) == ref, (k, open(p, "rb").read())


def test_second_restatement_agrees_with_the_c_oracle_on_the_fuzz_corpus(tmp_path):
    """oracle/np_oracle.py holds an independent plain-Python restatement of what the two ingest routines write and why
    they stop; it must agree with oracle/eagle_oracle.c (files, verdict, row / token / count in the messages)."""
    rng = np.random.default_rng(2026)
    p = str(tmp_path / "f.txt")
    for k in range(300):
        dims, AA, AB, BB, missing = fuzz_text_case(rng, p)
        ok, msgs = eo.createM_ASCII_rcpp(p, str(tmp_path / "a"), "text", AA, AB, BB, 8.0, dims, True, missing)
        ok2, rows2, why = npo.tokenise_text(open(p, "rb").read(), dims[1], AA, AB, BB, missing)
        assert ok == ok2, k
        too_long = why is not None and why[0] == "columns" and why[2] > dims[1]
        if not too_long:
            assert open(tmp_path / "a", "rb").read() == rows2, k
        if why and why[0] == "token":
            assert msgs[1] == f" For example , {why[2]} in row {why[1]}", k
        elif why:
            assert msgs[2] == f"        The error has occurred at row {why[1]} which contains {why[2]} but ", k
    for k in range(200):
        dims = fuzz_ped_case(rng, p)
        ok, msgs = eo.createM_ASCII_rcpp(p, str(tmp_path / "a"), "PLINK", "", "", "", 8.0, dims, True, "")
        ok2, rows2, why, warned = npo.plink_genotypes(open(p, "rb").read(), dims[1])
        assert ok == ok2 and open(tmp_path / "a", "rb").read() == rows2, k
        assert warned == any("missing alleles" in m for m in msgs), k
        if why and why[0] == "alleles":
            assert f"        The error has occurred at snp locus {why[1]} for individual {why[2]}" in msgs, k
        elif why:
            assert f"        The error has occurred at row {why[1]} which contains {why[2]} but " in msgs, k


def fuzz_reshape_case(rng, tmp_path, tag):
    """Random small M.ascii / Mt.ascii pair and a random index list: decreasing (what R passes), or shuffled / with
    repeats (the reference then erases shifted characters from the Mt lines)."""
    n, L = int(rng.integers(2, 40)), int(rng.integers(1, 60))
    G = synth.genotypes(n, L, seed=int(rng.integers(1 << 30)))
    m, mt = str(tmp_path / f"M{tag}.ascii"), str(tmp_path / f"Mt{tag}.ascii")
    npo.write_ascii(m, G)
    npo.write_ascii(mt, G.T)
    k = int(rng.integers(0, min(n - 1, 6) + 1))
    idx = sorted((int(i) for i in rng.choice(n, size=k, replace=False)), reverse=True)
    u = rng.random()
    if u < 0.2 and k > 1:
        rng.shuffle(idx)
    elif u < 0.3 and k > 0 and len(idx) < n - 1:
        idx.append(idx[int(rng.integers(len(idx)))])
    # keep every erase position inside the (shrinking) line: the reference throws otherwise
    size = n
    ok = True
    for i in idx:
        ok &= i <= size
        size -= i < size
    return (m, mt, [int(i) for i in idx], (n, L)) if ok and size > 0 and len(set(idx)) < n else None


def test_oracle_reshape_fuzz_against_reference_code(tmp_path, reference):
    rng = np.random.default_rng(77)
    done = 0
    for k in range(150):
        a = fuzz_reshape_case(rng, tmp_path, "a")
        if a is None:
            continue
        m, mt, idx, dims = a
        import shutil
        m2, mt2 = str(tmp_path / "Mb.ascii"), str(tmp_path / "Mtb.ascii")
        shutil.copy(m, m2); shutil.copy(mt, mt2)
        mine = reshape_and_read(m, mt, idx, dims)
        assert reference.fp(mine, digest=True) == reference(lambda: reshape_and_read(m2, mt2, idx, dims), digest=True), idx
        done += 1
    assert done > 100


@pytest.mark.gpu
def test_gpu_reshape_fuzz_against_oracle(api, tmp_path):
    import shutil
    rng = np.random.default_rng(77)
    done = 0
    for k in range(150):
        a = fuzz_reshape_case(rng, tmp_path, "a")
        if a is None:
            continue
        m, mt, idx, dims = a
        m2, mt2 = str(tmp_path / "Mb.ascii"), str(tmp_path / "Mtb.ascii")
        shutil.copy(m, m2); shutil.copy(mt, mt2)
        api.cache_clear()   # the same two paths are rewritten every round, possibly within one mtime tick of the file system
        assert api.ReshapeM_rcpp(m, mt, idx, dims) == eo.ReshapeM_rcpp(m2, mt2, idx, dims), idx
        assert open(m + "tmp", "rb").read() == open(m2 + "tmp", "rb").read(), (idx, dims)
        assert open(mt + "tmp", "rb").read() == open(mt2 + "tmp", "rb").read(), (idx, dims)
        done += 1
    assert done > 100


@pytest.mark.gpu
def test_gpu_ingest_fuzz_against_oracle(api, tmp_path, monkeypatch):
    rng = np.random.default_rng(2026)
    p = str(tmp_path / "f.txt")
    for k in range(300):
        dims, AA, AB, BB, missing = fuzz_text_case(rng, p)
        monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(int(rng.choice([64, 200, 1000, 1 << 28]))))
        ref = eo.createM_ASCII_rcpp(p, str(tmp_path / "b"), "text", AA, AB, BB, 8.0, dims, True, missing)
        msgs = []
        ok = api.createM_ASCII_rcpp(p, str(tmp_path / "a"), "text", AA, AB, BB, 8.0, dims, True, msgs.append, missing)
        assert (ok, msgs) == ref, (k, open(p, "rb").read())
        too_long = not ok and any("which contains" in m and int(m.split("contains")[1].split()[0]) > dims[1] for m in msgs)
        if not too_long:
            assert open(tmp_path / "a", "rb").read() == open(tmp_path / "b", "rb").read(), k
        assert api.getRowColumn(p) == eo.getRowColumn(p)
    for k in range(200):
        dims = fuzz_ped_case(rng, p)
        monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(int(rng.choice([64, 300, 1 << 28]))))
        ref = eo.createM_ASCII_rcpp(p, str(tmp_path / "b"), "PLINK", "", "", "", 8.0, dims, True, "")
        msgs = []
        ok = api.createM_ASCII_rcpp(p, str(tmp_path / "a"), "PLINK", "", "", "", 8.0, dims, True, msgs.append, "")
        assert (ok, msgs) == ref, (k, open(p, "rb").read())
        assert open(tmp_path / "a", "rb").read() == open(tmp_path / "b", "rb").read(), k


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("piece", [None, 40000, 3000])
def test_gpu_plink_matches_oracle(api, plink_cases, tmp_path, piece, monkeypatch):
    if piece:
        monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(piece))   # the allele table is carried from piece to piece
    for case in plink_cases:
        name, p, dims, ok = case
        ref = run_oracle_ped(case, str(tmp_path / "ref.ascii"))
        msgs = []
        got_ok = api.createM_ASCII_rcpp(p, str(tmp_path / "gpu.ascii"), "PLINK", "", "", "", 8.0, dims, True, msgs.append, "")
        assert got_ok == ref[0] == ok, name
        assert msgs == ref[1], name
        assert open(tmp_path / "gpu.ascii", "rb").read() == ref[2], name
    msgs = []
    assert api.createM_ASCII_rcpp(str(tmp_path / "absent.ped"), str(tmp_path / "g"), "PLINK", "", "", "", 8, (2, 10), True, msgs.append) is False
    assert len(msgs) == 2 and msgs[0].startswith("ERROR: PLINK ped file could not be opened")
    p = str(tmp_path / "multi.ped")
    open(p, "w").write("f i1 0 0 1 0 A G T T\nf i2 0 0 1 0 A C GT T\n")
    with pytest.raises(Exception, match="allele \"GT\" in row 2 is not a single character"):
        api.createM_ASCII_rcpp(p, str(tmp_path / "g"), "PLINK", "", "", "", 8, (2, 10), True, None)


@pytest.fixture(scope="module")
def api():
    from eagleeverything_b200 import api as a
    from eagleeverything_b200 import device
    device.init(0)
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("piece", [None, 4096, 700])
def test_gpu_tokeniser_matches_oracle(api, ingest_cases, tmp_path, piece, monkeypatch):
    if piece:
        monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(piece))   # several pieces of whole lines per file
    for case in ingest_cases:
        name, p, dims, AA, AB, BB, missing, ok, want = case
        for quiet in (False, True):
            ref = run_oracle(case, str(tmp_path / "ref.ascii"), quiet)
            msgs = []
            got_ok = api.createM_ASCII_rcpp(p, str(tmp_path / "gpu.ascii"), "text", AA, AB, BB, 8.0, dims, quiet, msgs.append, missing)
            data = open(tmp_path / "gpu.ascii", "rb").read()
            assert got_ok == ref[0] == ok, name
            assert msgs == ref[1], (name, quiet)
            if name != "long_row":
                assert data == ref[2], name
    msgs = []
    assert api.createM_ASCII_rcpp(str(tmp_path / "absent.txt"), str(tmp_path / "gpu.ascii"), "text", "0", "1", "2", 8, (3, 3), True,
                                  msgs.append) is False
    assert msgs == ["ERROR: Text file could not be opened with filename  " + str(tmp_path / "absent.txt") + "\n"]


@pytest.mark.gpu
def test_gpu_tokeniser_large_file_and_late_errors(api, tmp_path):
    n, L = 300, 40000                                 # 24 MB of text: ~730 chunks, several CTAs per SM
    G = synth.genotypes(n, L, seed=12)
    p = str(tmp_path / "big.txt")
    img = synth.ascii_image(G)
    text = np.full((n, 2 * L), ord(" "), np.uint8)
    text[:, 0::2] = img[:, :L]
    text[:, -1] = ord("\n")
    text.tofile(p)
    assert api.createM_ASCII_rcpp(p, str(tmp_path / "big.ascii"), "text", "0", "1", "2", 8.0, (n, L), True, None) is True
    assert open(tmp_path / "big.ascii", "rb").read() == img.tobytes()
    for row, col in [(299, 39999), (150, 20000), (0, 0)]:
        bad = text.copy()
        bad[row, 2 * col] = ord("5")
        if row + 1 < n:
            bad[row + 1, 2 * 100] = ord("6")           # a later error must not win
        bad.tofile(p)
        msgs = []
        assert api.createM_ASCII_rcpp(p, str(tmp_path / "bad.ascii"), "text", "0", "1", "2", 8.0, (n, L), True, msgs.append) is False
        assert msgs[1] == f" For example , 5 in row {row + 1}", (row, col)
        assert open(tmp_path / "bad.ascii", "rb").read() == img[:row].tobytes()
    short = text.copy()
    short[200, 2 * 777] = ord(" ")                     # one token fewer in row 201
    short.tofile(p)
    msgs = []
    assert api.createM_ASCII_rcpp(p, str(tmp_path / "bad.ascii"), "text", "0", "1", "2", 8.0, (n, L), True, msgs.append) is False
    assert msgs[2] == f"        The error has occurred at row 201 which contains {L - 1} but "


@pytest.mark.gpu
@pytest.mark.parametrize("n,L", [(5, 40), (16, 33), (31, 100), (150, 4998), (203, 3001), (1000, 777)])
def test_gpu_createMt_matches_oracle_and_feeds_the_cache(api, tmp_path, n, L):
    G = synth.genotypes(n, L, seed=n + L)
    m, mt, mt_ref = str(tmp_path / "M.ascii"), str(tmp_path / "Mt.ascii"), str(tmp_path / "Mt.ref")
    npo.write_ascii(m, G)
    ref_msgs = eo.createMt_ASCII_rcpp(m, mt_ref, "text", 8.0, (n, L), True)
    msgs = []
    api.createMt_ASCII_rcpp(m, mt, "text", 8.0, (n, L), True, msgs.append)
    assert open(mt, "rb").read() == open(mt_ref, "rb").read() == synth.ascii_image(G.T.copy()).tobytes()
    assert len(msgs) == len(ref_msgs) == 10
    for a, b in zip(msgs, ref_msgs):
        if "gigabytes" not in a:
            assert a == b
    # the stores left behind serve the hot-path calls on those files
    S, V, a = synth.scan_inputs(n, 3)
    got = api.calculate_a_and_vara_rcpp(mt, [api.NA_REAL], S, V, 8.0, (L, n), a)
    want = eo.calculate_a_and_vara_rcpp(mt, [eo.NA_REAL], S, V, 8.0, (L, n), a)
    scale = np.abs(want["vara"]).max()
    np.testing.assert_allclose(got["vara"], want["vara"], rtol=1e-9, atol=1e-12 * scale)
    assert np.array_equal(api.calculateMMt_rcpp(m, 8.0, 1, [api.NA_REAL], (n, L)), eo.calculateMMt_rcpp(m, 8.0, 1, [eo.NA_REAL], (n, L)))
    with pytest.raises(Exception, match="Could not open"):
        api.createMt_ASCII_rcpp(str(tmp_path / "absent.ascii"), mt, "text", 8.0, (n, L), True, None)


@pytest.mark.gpu
def test_gpu_text_to_scan_chain(api, tmp_path, demo):
    """ReadMarker's chain on the device: text -> M.ascii -> Mt.ascii -> M.Mt, all equal to the golden demo results."""
    G = demo["G"]
    n, L = G.shape
    p = str(tmp_path / "geno.txt")
    write_text(p, G, style=2, seed=1)
    m, mt = str(tmp_path / "M.ascii"), str(tmp_path / "Mt.ascii")
    assert api.createM_ASCII_rcpp(p, m, "text", "0", "1", "2", 8.0, (n, L), True, None)
    api.createMt_ASCII_rcpp(m, mt, "text", 8.0, (n, L), True, None)
    assert open(m, "rb").read() == open(demo["M"], "rb").read() and open(mt, "rb").read() == open(demo["Mt"], "rb").read()
    MMt = api.calculateMMt_rcpp(m, 8.0, 1, [api.NA_REAL], (n, L))
    assert hashlib.sha256(MMt.astype("<i4").tobytes()).hexdigest() == str(demo["z"]["mmt_sha256"])
