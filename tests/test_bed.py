"""PLINK 1 binary genotypes (.bed, SNP-major) straight into the resident stores: the format contract of
include/eagle_gpu.h restated by tests/plink_bed.py (write_bed / read_bed), the argument and format checks that run before
any device work, and on the GPU the decoder against the ASCII route of the same genotypes, byte for byte."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from eagleeverything_b200 import _lib, synth
from oracle import np_oracle as npo
from plink_bed import read_bed, write_bed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_genotypes(n, L, seed, p_missing=0.02):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 3, (n, L), dtype=np.uint8), rng.random((n, L)) < p_missing


def set_pad_bits(bed, n, L):
    """Every bit past individual n-1 in every SNP's last byte set to 1."""
    b = np.frombuffer(bed, dtype=np.uint8).copy()
    bpr = (n + 3) // 4
    if n % 4:
        b[3 + np.arange(L) * bpr + bpr - 1] |= np.uint8((0xFF << (2 * (n % 4))) & 0xFF)
    return b.tobytes()


# ----------------------------------------------------------------------------- the format, on the CPU
def test_hand_example_bytes():
    # n = 5, one SNP: A1/A1, missing, het, A2/A2, A1/A1 -> values 0, 1, 2, 3, 0
    G = np.array([[0], [0], [1], [2], [0]], dtype=np.uint8)
    miss = np.array([[False], [True], [False], [False], [False]])
    data = write_bed(G, missing=miss)
    assert data == b"\x6c\x1b\x01\xe4\x00"
    G2, m2 = read_bed(data, 5, 1)
    assert G2[:, 0].tolist() == [0, 1, 1, 2, 0] and m2[:, 0].tolist() == [False, True, False, False, False]


@pytest.mark.parametrize("n", [1, 3, 4, 5, 15, 16, 17, 203])
def test_write_read_round_trip(n):
    L = 37
    G, miss = random_genotypes(n, L, seed=n)
    data = write_bed(G, missing=miss)
    assert len(data) == 3 + L * ((n + 3) // 4)
    G2, m2 = read_bed(data, n, L)
    assert np.array_equal(m2, miss) and np.array_equal(G2, np.where(miss, 1, G))
    G3, m3 = read_bed(write_bed(G), n, L)
    assert np.array_equal(G3, G) and not m3.any()
    # A1 / A2 swapped on some SNPs: those columns read back as 2 - G
    flip = np.arange(L) % 3 == 1
    G4, _ = read_bed(write_bed(G, flip=flip), n, L)
    assert np.array_equal(G4[:, ~flip], G[:, ~flip]) and np.array_equal(G4[:, flip], 2 - G[:, flip])


@pytest.mark.parametrize("n", [1, 3, 5, 17, 203])
def test_pad_bits_are_ignored_by_read_bed(n):
    G, miss = random_genotypes(n, 11, seed=100 + n)
    data = write_bed(G, missing=miss)
    dirty = set_pad_bits(data, n, 11)
    assert dirty != data
    assert all(np.array_equal(a, b) for a, b in zip(read_bed(dirty, n, 11), read_bed(data, n, 11)))


# ----------------------------------------------------------------------------- checks before any device work
def _from_bed(path, n, L, snp0=0, snp1=None, kblocked=1):
    lib = _lib.load()
    h, miss = C.c_void_p(), C.c_int64()
    rc = lib.eg_store_from_bed(os.fsencode(path), n, L, snp0, L if snp1 is None else snp1, kblocked, C.byref(miss), C.byref(h))
    if rc == _lib.EG_OK:
        lib.eg_store_free(h)
    return rc, lib.eg_last_error().decode()


def _from_host_bed(data, n, L, snp0=0, snp1=None):
    lib = _lib.load()
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    h = C.c_void_p()
    rc = lib.eg_store_from_host_bed(buf.ctypes.data_as(C.c_void_p), n, L, snp0, L if snp1 is None else snp1, 1, None, C.byref(h))
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
    return n, L, data, write


def test_refusals_before_device_work(bed_file):
    n, L, data, write = bed_file
    rc, msg = _from_bed(write("magic.bed", b"\x6c\x1c\x01" + data[3:]), n, L)
    assert rc == _lib.EG_ERR_FORMAT and "not a PLINK .bed file" in msg and "6c 1c" in msg
    rc, msg = _from_bed(write("imaj.bed", b"\x6c\x1b\x00" + data[3:]), n, L)
    assert rc == _lib.EG_ERR_FORMAT and "individual-major" in msg
    rc, msg = _from_bed(write("short.bed", data[:-1]), n, L)
    assert rc == _lib.EG_ERR_FORMAT and f"has {len(data) - 1} bytes" in msg
    rc, msg = _from_bed(write("long.bed", data + b"\x00"), n, L)
    assert rc == _lib.EG_ERR_FORMAT and f"has {len(data) + 1} bytes" in msg
    rc, msg = _from_bed(write("tiny.bed", b"\x6c"), n, L)
    assert rc == _lib.EG_ERR_FORMAT
    good = write("good.bed", data)
    rc, msg = _from_bed(good, n, L, 0, L + 1)
    assert rc == _lib.EG_ERR_ARG and "outside [0, 300)" in msg
    rc, msg = _from_bed(good, n, L, 10, 10)
    assert rc == _lib.EG_ERR_ARG and "empty" in msg
    rc, msg = _from_bed(good, n + 4, L)      # wrong n: the size does not match
    assert rc == _lib.EG_ERR_FORMAT and "wrong n / L" in msg
    rc, msg = _from_bed(str(os.path.dirname(good)) + "/absent.bed", n, L)
    assert rc == _lib.EG_ERR_OPEN and "Could not open" in msg
    rc, msg = _from_host_bed(b"\x6c\x1b\x00" + data[3:], n, L)
    assert rc == _lib.EG_ERR_FORMAT and "individual-major" in msg
    rc, msg = _from_host_bed(b"\x00\x1b\x01" + data[3:], n, L)
    assert rc == _lib.EG_ERR_FORMAT and "magic" in msg
    rc, msg = _from_host_bed(data, n, L, 0, L + 1)
    assert rc == _lib.EG_ERR_ARG
    lib = _lib.load()
    rc = lib.eg_bed_to_ascii(os.fsencode(write("imaj2.bed", b"\x6c\x1b\x00" + data[3:])), n, L, b"M.ascii", b"Mt.ascii")
    assert rc == _lib.EG_ERR_FORMAT


def test_valid_file_without_gpu_fails_loudly(bed_file):
    lib = _lib.load()
    if lib.eg_device_count() > 0:
        pytest.skip("a GPU is visible")
    n, L, data, write = bed_file
    rc, msg = _from_bed(write("good.bed", data), n, L)
    assert rc == _lib.EG_ERR_CUDA and "no CPU fallback" in msg
    rc, msg = _from_host_bed(data, n, L)
    assert rc == _lib.EG_ERR_CUDA and "no CPU fallback" in msg


# ----------------------------------------------------------------------------- the decoder on the GPU
SHAPES = [(1, 1), (3, 5), (4, 128), (5, 129), (17, 300), (127, 1000), (203, 3001), (1000, 4097)]


def _vp(t):
    return C.c_void_p(t.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("n,L", SHAPES)
def test_decode_bed_equals_ascii_decode(n, L):
    import torch
    from eagleeverything_b200 import device
    lib = device.init(0)
    G, miss = random_genotypes(n, L, seed=n * 7919 + L)
    Geff = np.where(miss, 1, G)
    pad = np.zeros(64, np.uint8)
    imgM = torch.from_numpy(np.concatenate([synth.ascii_image(Geff).reshape(-1), pad])).cuda()
    imgT = torch.from_numpy(np.concatenate([synth.ascii_image(np.ascontiguousarray(Geff.T)).reshape(-1), pad])).cuda()
    ref_kb, e1 = device.decode_kb(imgM, L + 1, n, L)
    ref_rm, e2 = device.decode(imgT, n + 1, L, n)
    assert e1[0].item() == 0 and e2[0].item() == 0
    bpr = (n + 3) // 4
    data = write_bed(G, missing=miss)
    for blob in (data, set_pad_bits(data, n, L)):
        bed = torch.from_numpy(np.frombuffer(blob, np.uint8).copy()).cuda()
        for kblocked, ref in ((True, ref_kb), (False, ref_rm)):
            cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
            out = device.decode_bed(bed, n, L, kblocked, out=torch.full_like(ref, 7), missing=cnt)
            assert torch.equal(out, ref), (kblocked, "pads included")
            assert cnt.item() == int(miss.sum())
        # pieces with m0 offsets: any cut for the row-major layout, 128-marker blocks for the K-blocked one
        for kblocked, ref, step in ((False, ref_rm, 37), (False, ref_rm, 129), (True, ref_kb, 128), (True, ref_kb, 256)):
            out = torch.full_like(ref, 7)
            cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
            for m0 in range(0, L, step):
                ns = min(step, L - m0)
                _lib.check(lib.eg_dev_decode_bed(C.c_void_p(bed.data_ptr() + 3 + m0 * bpr), n, ns, _vp(out), L,
                                                 0 if kblocked else out.stride(0), m0, _vp(cnt), None))
            assert torch.equal(out, ref) and cnt.item() == int(miss.sum())
    if L > 128:   # a K-blocked piece that does not start on a block is refused
        out = torch.empty_like(ref_kb)
        assert lib.eg_dev_decode_bed(C.c_void_p(bed.data_ptr() + 3), n, 5, _vp(out), L, 0, 3, None, None) == _lib.EG_ERR_ARG


def _stores_equal(A, B, cols):
    """Two K-blocked M stores: same M.Mt, same extracted columns, same bytes."""
    lib = _lib.load()
    assert np.array_equal(A.mmt(), B.mmt())
    for c in cols:
        assert np.array_equal(A.extract_col(c), B.extract_col(c))
    i = A.info()
    wa, wb = (np.empty((i["rows"], (i["cols"] + 31) // 32), np.uint64) for _ in range(2))
    _lib.check(lib.eg_store_to_host_packed(A._h, wa.ctypes.data_as(C.c_void_p)))
    _lib.check(lib.eg_store_to_host_packed(B._h, wb.ctypes.data_as(C.c_void_p)))
    assert np.array_equal(wa, wb)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["file", "pageable", "pinned"])
@pytest.mark.parametrize("snp0,snp1", [(0, 3001), (130, 2777)])
def test_store_from_bed_equals_ascii_route(route, snp0, snp1, tmp_path, monkeypatch):
    import torch
    from eagleeverything_b200 import api, device
    device.init(0)
    n, L = 203, 3001
    G, miss = random_genotypes(n, L, seed=11)
    Geff = np.where(miss, 1, G)
    data = write_bed(G, missing=miss)
    # 51 bytes per SNP: pieces of 256 SNPs, twelve of them through the staging ring
    monkeypatch.setenv("EAGLE_INGEST_PIECE_BYTES", str(300 * 51))

    def bed_store(kblocked):
        if route == "file":
            p = tmp_path / "g.bed"
            p.write_bytes(data)
            return api.GenotypeStore.from_bed(str(p), n, L, snp0, snp1, kblocked=kblocked)
        img = np.frombuffer(data, np.uint8).copy()
        if route == "pinned":
            img = torch.from_numpy(img).pin_memory()
        return api.GenotypeStore.from_host_bed(img, n, L, snp0, snp1, kblocked=kblocked)

    M = bed_store(True)
    Mt = bed_store(False)
    w = snp1 - snp0
    assert M.n_missing == Mt.n_missing == int(miss[:, snp0:snp1].sum())
    assert M.info()["rows"] == n and M.info()["cols"] == w and Mt.info()["rows"] == w and Mt.info()["cols"] == n
    Ma = api.GenotypeStore.from_host_ascii(synth.ascii_image(Geff), n, L, snp0, snp1)
    Mta = api.GenotypeStore.from_host_rows(synth.ascii_image(np.ascontiguousarray(Geff.T)), L, n, snp0, snp1)
    _stores_equal(M, Ma, [0, 127, 128, w // 2, w - 1])
    S, V, a = synth.scan_inputs(n)
    ra, rv = Mt.a_and_vara(S, V, a)
    qa, qv = Mta.a_and_vara(S, V, a)
    assert np.array_equal(ra, qa) and np.array_equal(rv, qv)
    assert np.array_equal(M.extract_col(w // 3), Geff[:, snp0 + w // 3].astype(np.int32) - 1)
    for s in (M, Mt, Ma, Mta):
        s.free()


@pytest.mark.gpu
def test_hand_example_on_the_device():
    from eagleeverything_b200 import api, device
    device.init(0)
    s = api.GenotypeStore.from_host_bed(b"\x6c\x1b\x01\xe4\x00", 5, 1)
    assert s.extract_col(0).tolist() == [-1, 0, 0, 1, -1] and s.n_missing == 1


@pytest.mark.gpu
def test_allele_flips_negate_a_and_columns_only():
    from eagleeverything_b200 import api, device
    device.init(0)
    n, L = 203, 3001
    G, miss = random_genotypes(n, L, seed=17)
    flip = np.random.default_rng(3).random(L) < 1 / 3
    plain, flipped = write_bed(G, missing=miss), write_bed(G, flip=flip, missing=miss)
    A, B = (api.GenotypeStore.from_host_bed(d, n, L) for d in (plain, flipped))
    At, Bt = (api.GenotypeStore.from_host_bed(d, n, L, kblocked=False) for d in (plain, flipped))
    assert np.array_equal(A.mmt(), B.mmt())
    S, V, a = synth.scan_inputs(n)
    aa, va = At.a_and_vara(S, V, a)
    ab, vb = Bt.a_and_vara(S, V, a)
    assert np.array_equal(va, vb)
    assert np.array_equal(ab[flip], -aa[flip]) and np.array_equal(ab[~flip], aa[~flip])
    for c in [int(np.flatnonzero(flip)[0]), int(np.flatnonzero(~flip)[0]), L - 1]:
        sign = -1 if flip[c] else 1
        assert np.array_equal(B.extract_col(c), sign * A.extract_col(c))
    for s in (A, B, At, Bt):
        s.free()


@pytest.mark.gpu
@pytest.mark.parametrize("flipped", [False, True])
def test_search_on_stores_decoded_from_bed(demo, flipped):
    import torch
    from eagleeverything_b200 import am, device
    device.init(0)
    z, G, n, L = demo["z"], demo["G"], demo["n"], demo["L"]
    flip = (np.arange(L) % 3 == 2) if flipped else None
    bed = torch.from_numpy(np.frombuffer(write_bed(G, flip=flip), np.uint8).copy()).cuda()
    kb = device.decode_bed(bed, n, L, kblocked=True)
    t = device.decode_bed(bed, n, L, kblocked=False)
    r = am.AM_resident(kb, t, n, L, z["trait1"])
    assert r["selected"] == list(z["am1_selected"]) and r["all_picked"] == list(z["am1_all_picked"])
    np.testing.assert_allclose(r["extBIC"], z["am1_extBIC"], rtol=1e-8)
    X0 = np.column_stack([np.ones(n), z["pc1"], z["pc2"]])
    r2 = am.AM_resident(kb, t, n, L, z["trait2"], X0=X0)
    assert r2["selected"] == list(z["am2_selected"]) and r2["all_picked"] == list(z["am2_all_picked"])
    np.testing.assert_allclose(r2["extBIC"], z["am2_extBIC"], rtol=1e-8)


@pytest.mark.gpu
def test_bed_to_ascii_and_the_exports_that_follow(tmp_path):
    from eagleeverything_b200 import api, device
    device.init(0)
    n, L = 203, 3001
    G, miss = random_genotypes(n, L, seed=23)
    Geff = np.where(miss, 1, G)
    bed = tmp_path / "g.bed"
    bed.write_bytes(write_bed(G, missing=miss))
    (tmp_path / "g.fam").write_text("".join(f"F{i} I{i} 0 0 0 -9\n" for i in range(n)))
    (tmp_path / "g.bim").write_text("".join(f"1 rs{j} 0 {j + 1} A C\n" for j in range(L)))
    assert api.plink_dims(str(tmp_path / "g")) == (n, L) == api.plink_dims(str(bed))
    m, mt = str(tmp_path / "M.ascii"), str(tmp_path / "Mt.ascii")
    api.bed_to_ascii(str(bed), n, L, m, mt)
    rm, rmt = str(tmp_path / "ref_M.ascii"), str(tmp_path / "ref_Mt.ascii")
    npo.write_ascii(rm, Geff)
    npo.write_ascii(rmt, Geff.T)
    assert open(m, "rb").read() == open(rm, "rb").read()
    assert open(mt, "rb").read() == open(rmt, "rb").read()
    NA = api.NA_REAL
    for sel in ([NA], [4.0, float(L - 1)]):
        assert np.array_equal(api.calculateMMt_rcpp(m, 8, 1, sel, (n, L)), api.calculateMMt_rcpp(rm, 8, 1, sel, (n, L)))
        S, V, a = synth.scan_inputs(n)
        r1 = api.calculate_a_and_vara_rcpp(mt, sel, S, V, 8, (L, n), a)
        r2 = api.calculate_a_and_vara_rcpp(rmt, sel, S, V, 8, (L, n), a)
        assert np.array_equal(r1["a"], r2["a"]) and np.array_equal(r1["vara"], r2["vara"])
    assert np.array_equal(api.extract_geno_rcpp(m, 8, 1234, (n, L)), Geff[:, 1234].astype(np.int32) - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("ngpu", [2, 4, 8])
def test_sharded_bed_store_equals_one_gpu(ngpu):
    import torch
    if torch.cuda.device_count() < ngpu:
        pytest.skip(f"needs {ngpu} GPUs")
    script = os.path.join(ROOT, "tests", "bed_multi_worker.py")
    r = subprocess.run([sys.executable, script, str(ngpu), "515", "9001"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "BED_MULTI_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
