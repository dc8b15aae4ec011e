"""Streamed stores (include/eagle_gpu.h, eg_store_stream_*): genotype sets larger than device memory, decoded piece by piece
on every call.  On the CPU: the constructors' checks before any device work.  On the GPU: M.Mt, a / var(a) and extracted
columns bit for bit equal to the resident stores', across sources, piece counts, zeroed markers and compute modes; ASCII
format errors in later pieces; the drop-in exports' fall-back to streaming; the demo forward search on streamed stores."""
import ctypes as C
import os

import numpy as np
import pytest

from eagleeverything_b200 import _lib, synth
from plink_bed import write_bed


def random_genotypes(n, L, seed, p_missing=0.02):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 3, (n, L), dtype=np.uint8), rng.random((n, L)) < p_missing


# ----------------------------------------------------------------------------- checks before any device work
def _stream_bed(path, n, L, snp0=0, snp1=None, kblocked=1):
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.eg_store_stream_bed(os.fsencode(path), n, L, snp0, L if snp1 is None else snp1, kblocked, C.byref(h))
    if rc == _lib.EG_OK:
        lib.eg_store_free(h)
    return rc, lib.eg_last_error().decode()


def _stream_host_bed(data, n, L, snp0=0, snp1=None):
    lib = _lib.load()
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    h = C.c_void_p()
    rc = lib.eg_store_stream_host_bed(buf.ctypes.data_as(C.c_void_p), n, L, snp0, L if snp1 is None else snp1, 0, C.byref(h))
    if rc == _lib.EG_OK:
        lib.eg_store_free(h)
    return rc, lib.eg_last_error().decode()


def _stream_file(path, rows, cols, kblocked=1):
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.eg_store_stream_file(os.fsencode(path), rows, cols, kblocked, C.byref(h))
    if rc == _lib.EG_OK:
        lib.eg_store_free(h)
    return rc, lib.eg_last_error().decode()


@pytest.fixture
def bed_file(tmp_path):
    n, L = 13, 300
    G, miss = random_genotypes(n, L, seed=5)
    data = write_bed(G, missing=miss)

    def write(name, blob):
        p = tmp_path / name
        p.write_bytes(blob)
        return str(p)
    return n, L, G, data, write


def test_constructors_refuse_what_the_resident_ones_refuse(bed_file):
    n, L, G, data, write = bed_file
    rc, msg = _stream_bed(write("magic.bed", b"\x6c\x1c\x01" + data[3:]), n, L)
    assert rc == _lib.EG_ERR_FORMAT and "not a PLINK .bed file" in msg and "6c 1c" in msg
    rc, msg = _stream_bed(write("imaj.bed", b"\x6c\x1b\x00" + data[3:]), n, L)
    assert rc == _lib.EG_ERR_FORMAT and "individual-major" in msg
    rc, msg = _stream_bed(write("short.bed", data[:-1]), n, L)
    assert rc == _lib.EG_ERR_FORMAT and f"has {len(data) - 1} bytes" in msg
    good = write("good.bed", data)
    rc, msg = _stream_bed(good, n, L, 0, L + 1)
    assert rc == _lib.EG_ERR_ARG and "eg_store_stream_bed" in msg and "outside [0, 300)" in msg
    rc, msg = _stream_bed(good, n, L, 10, 10)
    assert rc == _lib.EG_ERR_ARG and "empty" in msg
    rc, msg = _stream_bed(good, n + 4, L)
    assert rc == _lib.EG_ERR_FORMAT and "wrong n / L" in msg
    rc, msg = _stream_bed(os.path.dirname(good) + "/absent.bed", n, L)
    assert rc == _lib.EG_ERR_OPEN and "Could not open" in msg
    rc, msg = _stream_host_bed(b"\x6c\x1b\x00" + data[3:], n, L)
    assert rc == _lib.EG_ERR_FORMAT and "individual-major" in msg
    rc, msg = _stream_host_bed(data, n, L, 0, L + 1)
    assert rc == _lib.EG_ERR_ARG and "eg_store_stream_host_bed" in msg
    # ASCII: check_image_size's messages
    img = synth.ascii_image(G).reshape(-1).tobytes()
    m = write("M.ascii", img)
    rc, msg = _stream_file(m, n, L + 1)
    assert rc == _lib.EG_ERR_FORMAT and "no-space ASCII need" in msg
    rc, msg = _stream_file(write("bad_line.ascii", img[1:] + b"\n"), n, L)
    assert rc == _lib.EG_ERR_FORMAT and "first line is not" in msg
    rc, msg = _stream_file(m, 0, L)
    assert rc == _lib.EG_ERR_ARG
    rc, msg = _stream_file(os.path.dirname(m) + "/absent.ascii", n, L)
    assert rc == _lib.EG_ERR_OPEN


def test_valid_sources_without_gpu_fail_loudly(bed_file):
    lib = _lib.load()
    if lib.eg_device_count() > 0:
        pytest.skip("a GPU is visible")
    n, L, G, data, write = bed_file
    rc, msg = _stream_bed(write("good.bed", data), n, L)
    assert rc == _lib.EG_ERR_CUDA and "no CPU fallback" in msg
    rc, msg = _stream_host_bed(data, n, L)
    assert rc == _lib.EG_ERR_CUDA and "no CPU fallback" in msg
    rc, msg = _stream_file(write("M.ascii", synth.ascii_image(G).reshape(-1).tobytes()), n, L)
    assert rc == _lib.EG_ERR_CUDA and "no CPU fallback" in msg


# ----------------------------------------------------------------------------- on the GPU
@pytest.fixture(scope="module")
def gpu():
    from eagleeverything_b200 import api, device
    device.init(0)
    return api


def _source(api, route, data, tmp_path, n, L, snp0, snp1, kblocked, streamed):
    import torch
    if route == "file":
        p = tmp_path / "g.bed"
        if not p.exists():
            p.write_bytes(data)
        f = api.GenotypeStore.stream_bed if streamed else api.GenotypeStore.from_bed
        return f(str(p), n, L, snp0, snp1, kblocked=kblocked)
    img = np.frombuffer(data, np.uint8).copy()
    if route == "pinned":
        img = torch.from_numpy(img).pin_memory()
    f = api.GenotypeStore.stream_host_bed if streamed else api.GenotypeStore.from_host_bed
    return f(img, n, L, snp0, snp1, kblocked=kblocked)


def _check_equal(api, M, Ms, Mt, Mts, n, w, zero=()):
    assert Ms.info()["device_ptr"] is None and Mts.info()["device_ptr"] is None
    for k in ("rows", "cols", "pitch"):
        assert Ms.info()[k] == M.info()[k] and Mts.info()[k] == Mt.info()[k]
    z = [c for c in zero if c < w]
    assert np.array_equal(Ms.mmt(z), M.mmt(z))
    S, V, a = synth.scan_inputs(n)
    ra, rv = Mt.a_and_vara(S, V, a, z)
    qa, qv = Mts.a_and_vara(S, V, a, z)
    assert np.array_equal(ra, qa) and np.array_equal(rv, qv)
    for c in sorted({0, 127, 128, w // 2, w - 1}):
        if c < w:
            assert np.array_equal(Ms.extract_col(c), M.extract_col(c))


# (piece bytes, expected pieces) at n = 203 (51 bytes per SNP): one piece, two, and many with a ragged last one
PIECES = {"one": 1 << 30, "two": 1600 * 51, "many": 300 * 51}


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["file", "pageable", "pinned"])
@pytest.mark.parametrize("pieces", ["one", "two", "many"])
@pytest.mark.parametrize("snp0,snp1", [(0, 3001), (130, 2777)])
def test_streamed_bed_equals_resident(gpu, route, pieces, snp0, snp1, tmp_path, monkeypatch):
    n, L = 203, 3001
    G, miss = random_genotypes(n, L, seed=11)
    data = write_bed(G, missing=miss)
    M = _source(gpu, route, data, tmp_path, n, L, snp0, snp1, True, False)
    Mt = _source(gpu, route, data, tmp_path, n, L, snp0, snp1, False, False)
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(PIECES[pieces]))
    Ms = _source(gpu, route, data, tmp_path, n, L, snp0, snp1, True, True)
    Mts = _source(gpu, route, data, tmp_path, n, L, snp0, snp1, False, True)
    _check_equal(gpu, M, Ms, Mt, Mts, n, snp1 - snp0, zero=(5, 1500, 2600))


@pytest.mark.gpu
def test_streamed_bed_larger_shape(gpu, monkeypatch):
    n, L = 515, 9001
    G, miss = random_genotypes(n, L, seed=12)
    data = write_bed(G, missing=miss)
    M, Mt = gpu.GenotypeStore.from_host_bed(data, n, L), gpu.GenotypeStore.from_host_bed(data, n, L, kblocked=False)
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(1000 * 129))   # 896 SNPs a piece: 11 pieces, the last one ragged
    Ms, Mts = gpu.GenotypeStore.stream_host_bed(data, n, L), gpu.GenotypeStore.stream_host_bed(data, n, L, kblocked=False)
    _check_equal(gpu, M, Ms, Mt, Mts, n, L, zero=(0, 895, 896, 4000, 9000))


@pytest.mark.gpu
def test_zeroed_markers_in_every_piece_and_at_boundaries(gpu, monkeypatch):
    n, L = 203, 3001
    G, _ = random_genotypes(n, L, seed=13)
    data = write_bed(G)
    M, Mt = gpu.GenotypeStore.from_host_bed(data, n, L), gpu.GenotypeStore.from_host_bed(data, n, L, kblocked=False)
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(300 * 51))   # pieces of 256 SNPs
    Ms, Mts = gpu.GenotypeStore.stream_host_bed(data, n, L), gpu.GenotypeStore.stream_host_bed(data, n, L, kblocked=False)
    S, V, a = synth.scan_inputs(n)
    for z in ([0, 3], [255, 256], [1279, 1280, 1281, 1500], [2815, 2816, 3000], [0, 255, 256, 1500, 1500, 3000]):
        assert np.array_equal(Ms.mmt(z), M.mmt(z)), z
        ra, rv = Mt.a_and_vara(S, V, a, z)
        qa, qv = Mts.a_and_vara(S, V, a, z)
        assert np.array_equal(ra, qa) and np.array_equal(rv, qv), z
        assert (qa[z] == 0).all() and (qv[z] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mmt_mode", ["fp4", "i8"])
@pytest.mark.parametrize("scan_mode", ["i8", "f64"])
def test_compute_modes(gpu, mmt_mode, scan_mode, monkeypatch):
    n, L = 515, 3001
    G, miss = random_genotypes(n, L, seed=14)
    data = write_bed(G, missing=miss)
    if mmt_mode == "i8":
        monkeypatch.setenv("EAGLE_MMT_MODE", "i8")
    old = gpu.get_scan_mode()
    gpu.set_scan_mode(scan_mode)
    try:
        M, Mt = gpu.GenotypeStore.from_host_bed(data, n, L), gpu.GenotypeStore.from_host_bed(data, n, L, kblocked=False)
        monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(500 * 129))
        Ms, Mts = gpu.GenotypeStore.stream_host_bed(data, n, L), gpu.GenotypeStore.stream_host_bed(data, n, L, kblocked=False)
        _check_equal(gpu, M, Ms, Mt, Mts, n, L, zero=(7, 384, 2999))
        ms, ops = C.c_double(), C.c_double()   # the scan kernel's time: the sum over the pieces
        _lib.check(_lib.load().eg_last_scan_kernel(C.byref(ms), C.byref(ops)))
        assert ms.value > 0 and ops.value > 0
    finally:
        gpu.set_scan_mode(old)


@pytest.mark.gpu
def test_streamed_ascii_equals_resident(gpu, tmp_path, monkeypatch):
    from oracle import np_oracle as npo
    n, L = 203, 3001
    G = synth.genotypes(n, L, seed=15)
    m, mt = str(tmp_path / "M.ascii"), str(tmp_path / "Mt.ascii")
    npo.write_ascii(m, G)
    npo.write_ascii(mt, G.T)
    M, Mt = gpu.GenotypeStore.from_file(m, n, L), gpu.GenotypeStore.from_file(m, n, L).transpose()
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(1024 * n))   # M.ascii: 3 pieces of 1024 columns; Mt.ascii: 4 KB
    Ms, Mts = gpu.GenotypeStore.stream_file(m, n, L), gpu.GenotypeStore.stream_file(mt, L, n, kblocked=False)
    _check_equal(gpu, M, Ms, Mt, Mts, n, L, zero=(1023, 1024, 2500))


@pytest.mark.gpu
def test_bad_byte_in_a_later_piece_gives_the_resident_error(gpu, tmp_path, monkeypatch):
    """Same code and text as the resident upload.  The position is the decoder unit's that saw the byte: the same as the
    resident one for Mt.ascii; for M.ascii, whose column pieces go through other decoder units than the resident upload's
    whole rows, a unit inside the piece that holds the byte (at most 16 rows of at most one piece's columns).  The
    resident uploads from pageable memory and files run through the same piece loop in line pieces, so the piece size is
    set before them too: M.ascii in pieces of 128 lines puts the byte in the second piece, Mt.ascii in pieces of 640
    lines in the fourth, and both must still report the byte's absolute row."""
    import re
    from oracle import np_oracle as npo
    n, L = 203, 3001
    G = synth.genotypes(n, L, seed=16)
    m, mt = str(tmp_path / "M.ascii"), str(tmp_path / "Mt.ascii")
    npo.write_ascii(m, G)
    npo.write_ascii(mt, G.T)
    for path, rows, cols, r, c in ((m, n, L, 150, 2500), (mt, L, n, 2500, 150)):
        b = bytearray(open(path, "rb").read())
        b[r * (cols + 1) + c] = ord("7")
        open(path, "wb").write(bytes(b))
        kb = path == m
        monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(128 * (L + 1)) if kb else str(700 * (n + 1)))
        with pytest.raises(_lib.EagleGpuError) as want:   # the resident uploads: K-blocked M, row-major Mt
            if kb:
                gpu.GenotypeStore.from_file(path, rows, cols)
            else:
                gpu.GenotypeStore.from_host_rows(np.frombuffer(bytes(b), np.uint8), rows, cols, 0, rows)
        if kb:
            monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(1024 * n))
        s = gpu.GenotypeStore.stream_file(path, rows, cols, kblocked=kb)
        with pytest.raises(_lib.EagleGpuError) as got:
            if kb:
                s.mmt()
            else:
                S, V, a = synth.scan_inputs(n)
                s.a_and_vara(S, V, a)
        assert got.value.code == want.value.code == _lib.EG_ERR_FORMAT
        pos = re.compile(r"near row (\d+), column (\d+)")
        assert pos.sub("", str(got.value)) == pos.sub("", str(want.value))
        if kb:   # pieces of 1024 columns: the byte is in the third, [2048, 3001)
            row, col = map(int, pos.search(str(got.value)).groups())
            assert row <= r < row + 16 and 2048 <= col <= c, str(got.value)
            row, col = map(int, pos.search(str(want.value)).groups())   # the resident upload: a 16 KB row chunk
            assert row <= r < row + 16 and col <= c < col + 16384, str(want.value)
        else:
            assert str(got.value) == str(want.value)
        monkeypatch.delenv("EAGLE_INGEST_PIECE_BYTES")


# (route, piece bytes) at n = 403, L = 3001: column pieces of 1024 markers (3), line pieces of 128 individuals (4) or of
# 640 markers (5); the default piece size takes each upload in one piece
RESIDENT_PIECES = {"pinned": 1024 * 403, "pageable": 128 * 3002, "pageable_window": 128 * 3002, "file": 128 * 3002,
                   "file_window": 128 * 3002, "rows_window": 700 * 404}


@pytest.mark.gpu
@pytest.mark.parametrize("route", sorted(RESIDENT_PIECES))
def test_resident_ascii_uploads_in_pieces_equal_one_piece(gpu, route, tmp_path, monkeypatch):
    """The resident ASCII uploads run through the piece loop: in several ragged pieces they give the store bytes, K and
    a / var(a) of one piece.  A page-locked image keeps accumulating M.Mt under the copy (no contraction in mmt)."""
    import torch
    from oracle import np_oracle as npo
    n, L, c0, c1 = 403, 3001, 130, 2777
    G = synth.genotypes(n, L, seed=18)
    img = np.concatenate([synth.ascii_image(G).reshape(-1), np.zeros(64, np.uint8)])
    imgT = synth.ascii_image(np.ascontiguousarray(G.T)).reshape(-1)
    pinned = torch.from_numpy(img.copy()).pin_memory()
    m = str(tmp_path / "M.ascii")
    npo.write_ascii(m, G)
    S, V, a = synth.scan_inputs(n)
    kb = route != "rows_window"

    def upload():
        GS = gpu.GenotypeStore
        return {"pinned": lambda: GS.from_host_ptr(pinned.data_ptr(), n, L),
                "pageable": lambda: GS.from_host_ascii(img, n, L),
                "pageable_window": lambda: GS.from_host_ascii(img, n, L, c0, c1),
                "file": lambda: GS.from_file(m, n, L),
                "file_window": lambda: GS.from_file(m, n, L, c0, c1),
                "rows_window": lambda: GS.from_host_rows(imgT, L, n, c0, c1)}[route]()

    def results():
        s = upload()
        i = s.info()
        words = np.empty((i["rows"], (i["cols"] + 31) // 32), np.uint64)
        _lib.check(_lib.load().eg_store_to_host_packed(s._h, words.ctypes.data_as(C.c_void_p)))
        M, Mt = (s, s.transpose()) if kb else (s.transpose(), s)
        K = M.mmt()
        syrk_ms = gpu.last_timing()["syrk_ms"]
        return words, K, syrk_ms, *Mt.a_and_vara(S, V, a)

    one = results()
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(RESIDENT_PIECES[route]))
    several = results()
    for x, y in zip(one[:2] + one[3:], several[:2] + several[3:]):
        assert np.array_equal(x, y)
    assert (one[2] == several[2] == 0.0) == (route == "pinned"), (one[2], several[2])


@pytest.mark.gpu
def test_exports_stream_when_the_store_does_not_fit(gpu, tmp_path, monkeypatch):
    from oracle import np_oracle as npo
    n, L = 203, 3001
    G = synth.genotypes(n, L, seed=17)
    m, mt = str(tmp_path / "M.ascii"), str(tmp_path / "Mt.ascii")
    npo.write_ascii(m, G)
    npo.write_ascii(mt, G.T)
    NA = gpu.NA_REAL
    S, V, a = synth.scan_inputs(n)

    def run():
        gpu.cache_clear()
        out = [gpu.calculateMMt_rcpp(m, 8, 1, sel, (n, L)) for sel in ([NA], [4.0, 1024.0, float(L - 1)])]
        for sel in ([NA], [0.0, 2047.0, 2048.0]):
            r = gpu.calculate_a_and_vara_rcpp(mt, sel, S, V, 8, (L, n), a)
            out += [r["a"], r["vara"]]
        out += [gpu.extract_geno_rcpp(m, 8, c, (n, L)) for c in (0, 1500, L - 1)]
        out2 = str(tmp_path / "Mt_out.ascii")
        gpu.createMt_ASCII_rcpp(m, out2, "text", 8, (n, L))
        out.append(np.frombuffer(open(out2, "rb").read(), np.uint8))
        return out

    want = run()
    monkeypatch.setenv("EAGLE_TEST_FAIL_ALLOC", "1")
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(1024 * n))
    said = []
    gpu.cache_clear()
    gpu.calculateMMt_rcpp(m, 8, 1, [NA], (n, L), quiet=False, message=said.append)
    assert any("streamed from" in s and "3 pieces" in s for s in said), said
    got = run()
    assert len(got) == len(want)
    for x, y in zip(got, want):
        assert np.array_equal(x, y)
    monkeypatch.delenv("EAGLE_TEST_FAIL_ALLOC")
    gpu.cache_clear()


@pytest.mark.gpu
def test_refusals(gpu, monkeypatch):
    n, L = 203, 600
    G, _ = random_genotypes(n, L, seed=18)
    data = write_bed(G)
    Ms, Mts = gpu.GenotypeStore.stream_host_bed(data, n, L), gpu.GenotypeStore.stream_host_bed(data, n, L, kblocked=False)
    lib = _lib.load()
    h = C.c_void_p()
    words = np.empty(n * 19, np.uint64)
    for call, what in ((lambda: lib.eg_store_transpose(Ms._h, C.byref(h)), "eg_store_transpose"),
                       (lambda: lib.eg_store_drop_individuals(Mts._h, (C.c_int64 * 1)(3), 1, 0, C.byref(h)),
                        "eg_store_drop_individuals"),
                       (lambda: lib.eg_store_to_host_packed(Ms._h, words.ctypes.data_as(C.c_void_p)), "eg_store_to_host_packed")):
        assert call() == _lib.EG_ERR_ARG
        msg = lib.eg_last_error().decode()
        assert what in msg and "streamed" in msg
    with pytest.raises(_lib.EagleGpuError):
        Mts.mmt()
    with pytest.raises(_lib.EagleGpuError):   # the scan needs the Mt orientation (its n is the M store's cols here)
        Ms.a_and_vara(*synth.scan_inputs(L))


@pytest.mark.gpu
def test_constructors_refuse_a_multi_gpu_set(tmp_path):
    import subprocess
    import sys
    import textwrap
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = textwrap.dedent(f"""
        import sys, ctypes as C, numpy as np
        sys.path[:0] = [{root!r}, {os.path.join(root, 'tests')!r}]
        from eagleeverything_b200 import _lib
        from plink_bed import write_bed
        lib = _lib.load()
        _lib.check(lib.eg_init_multi(2, None))
        data = np.frombuffer(write_bed(np.zeros((8, 300), np.uint8)), np.uint8).copy()
        open({str(tmp_path / 'g.bed')!r}, 'wb').write(data.tobytes())
        h = C.c_void_p()
        a = lib.eg_store_stream_host_bed(data.ctypes.data_as(C.c_void_p), 8, 300, 0, 300, 1, C.byref(h))
        b = lib.eg_store_stream_bed({str(tmp_path / 'g.bed')!r}.encode(), 8, 300, 0, 300, 1, C.byref(h))
        open({str(tmp_path / 'M.ascii')!r}, 'wb').write(b"0" * 300 + b"\n" + b"1" * 300 + b"\n")
        c = lib.eg_store_stream_file({str(tmp_path / 'M.ascii')!r}.encode(), 2, 300, 1, C.byref(h))
        assert a == b == c == _lib.EG_ERR_ARG and b"one GPU" in lib.eg_last_error(), (a, b, c)
        lib.eg_shutdown()
        print("STREAM_MULTI_OK")
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "STREAM_MULTI_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


@pytest.mark.gpu
def test_demo_forward_search_on_streamed_data(gpu, demo, tmp_path, monkeypatch):
    from eagleeverything_b200 import am
    z, G, n, L = demo["z"], demo["G"], demo["n"], demo["L"]
    bed = tmp_path / "demo.bed"
    bed.write_bytes(write_bed(G))
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(1 << 20))
    geno = am.ResidentGeno(gpu.GenotypeStore.stream_bed(str(bed), n, L),
                           gpu.GenotypeStore.stream_bed(str(bed), n, L, kblocked=False))
    X0 = np.column_stack([np.ones(n), z["pc1"], z["pc2"]])
    routes = [geno, am.FileGeno(demo["M"], demo["Mt"], (n, L))]
    for k, g in enumerate(routes):
        if k == 1:   # the R route: the exports find no room for the stores and stream the files
            gpu.cache_clear()
            monkeypatch.setenv("EAGLE_TEST_FAIL_ALLOC", "1")
        r = am.AM(g, z["trait1"])
        assert r["selected"] == list(z["am1_selected"]) and r["all_picked"] == list(z["am1_all_picked"])
        np.testing.assert_allclose(r["extBIC"], z["am1_extBIC"], rtol=1e-8)
        r2 = am.AM(g, z["trait2"], X0=X0)
        assert r2["selected"] == list(z["am2_selected"]) and r2["all_picked"] == list(z["am2_all_picked"])
        np.testing.assert_allclose(r2["extBIC"], z["am2_extBIC"], rtol=1e-8)
    monkeypatch.delenv("EAGLE_TEST_FAIL_ALLOC")
    gpu.cache_clear()
