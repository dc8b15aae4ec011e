"""M * M^T on block-scaled E2M1 tensor cores (syrk_fp4_kernel, the default of eg_dev_syrk_i8 / eg_dev_syrk_i8_kb):
the FP32 accumulator chains give the same integers as the int8 kernel (EAGLE_MMT_MODE=i8) and as numpy."""
import numpy as np
import pytest

from eagleeverything_b200 import api, synth
from oracle import eagle_oracle as eo
from oracle import np_oracle as npo

pytestmark = pytest.mark.gpu

NA = api.NA_REAL
MMT_FP4_CHAIN = 1 << 20   # syrk_i8.cu: longest accumulator chain the library lets the E2M1 kernel run


@pytest.fixture(scope="module")
def dev():
    import torch
    from eagleeverything_b200 import device
    device.init(0)
    return device, torch


def kblocked(torch, M):
    """int8 (n, L) -> K-blocked store (ceil(L/128), n, 128), zero padded, on the device."""
    n, L = M.shape
    kb = (L + 127) // 128
    P = np.zeros((n, kb * 128), np.int8)
    P[:, :L] = M
    return torch.from_numpy(np.ascontiguousarray(P.reshape(n, kb, 128).transpose(1, 0, 2))).cuda()


def rowmajor(torch, M, pitch=None):
    n, L = M.shape
    P = np.zeros((n, pitch or (L + 127) // 128 * 128), np.int8)
    P[:, :L] = M
    return torch.from_numpy(P).cuda()


def exact(M):
    Mf = M.astype(np.float64)   # exact: |sums| < 2^53
    return (Mf @ Mf.T).astype(np.int64)


def mmt(dev, store, n, L, mode, monkeypatch, kblocked_layout=True, C32=None, zero=True, chunk=None):
    device, torch = dev
    if mode == "i8":
        monkeypatch.setenv("EAGLE_MMT_MODE", "i8")
    else:
        monkeypatch.delenv("EAGLE_MMT_MODE", raising=False)
    if chunk:
        monkeypatch.setenv("EAGLE_MMT_FP4_CHUNK", str(chunk))
    else:
        monkeypatch.delenv("EAGLE_MMT_FP4_CHUNK", raising=False)
    f = device.syrk_kb if kblocked_layout else device.syrk
    C = f(store, n, L, C32=C32, zero=zero)
    torch.cuda.synchronize()
    monkeypatch.delenv("EAGLE_MMT_MODE", raising=False)
    monkeypatch.delenv("EAGLE_MMT_FP4_CHUNK", raising=False)
    return C.cpu().numpy().astype(np.int64)


def upper(C):
    return np.triu(C)


def probe_rows(L, seed=0):
    """Adversarial operands for FP32 accumulation of +-1 products."""
    rng = np.random.default_rng(seed)
    k = np.arange(L)
    rows = [np.ones(L), -np.ones(L), np.where(k % 2 == 0, 1, -1),
            np.where(k % 64 == 63, 0, 1),          # 63 per K=64 instruction against row 0: odd partial sums
            np.where(k % 3 == 2, 0, 1),
            np.where(k < L // 2, 1, -1),           # climbs to L/2 then falls back: small steps at large magnitude
            rng.integers(-1, 2, L), rng.choice([-1, 1], L)]
    return np.stack(rows).astype(np.int8)


@pytest.mark.parametrize("L", [2047, 2049, 16383, 16385, (1 << 20) - 1, (1 << 20) + 1, (1 << 24) - 1, (1 << 24) + 257])
def test_exactness_probe_fp32_chains(dev, monkeypatch, L):
    """One accumulator chain of L markers (K split off): bit for bit with the int8 kernel and numpy up to
    MMT_FP4_CHAIN; longer chains are reported, not required (the library never runs them)."""
    device, torch = dev
    M = probe_rows(L)
    n = M.shape[0]
    store = kblocked(torch, M)
    ref = exact(M)
    i8 = upper(mmt(dev, store, n, L, "i8", monkeypatch))
    assert np.array_equal(i8, upper(ref))
    fp4 = upper(mmt(dev, store, n, L, "fp4", monkeypatch, chunk=(L + 255) // 256 * 256))
    bad = np.argwhere(fp4 != i8)
    print(f"\nexactness probe: chain {L} markers: {'exact' if bad.size == 0 else 'INEXACT at ' + str(bad.tolist())}"
          f" (max |K| {int(np.abs(ref).max())})")
    if L <= MMT_FP4_CHAIN:
        assert bad.size == 0
    del store
    torch.cuda.empty_cache()


def test_all_ones_just_above_the_chain_cap(dev, monkeypatch):
    """The default cuts chains at MMT_FP4_CHAIN: all-ones rows with L just above it still give L exactly."""
    device, torch = dev
    L = MMT_FP4_CHAIN + 259
    M = np.ones((6, L), np.int8)
    M[1] = -1
    M[2, ::2] = 0
    store = kblocked(torch, M)
    assert np.array_equal(upper(mmt(dev, store, 6, L, "fp4", monkeypatch)), upper(exact(M)))


def test_demo_bit_identical_to_int8(dev, monkeypatch, demo):
    device, torch = dev
    M = (demo["G"].astype(np.int8) - 1)
    n, L = M.shape
    store = kblocked(torch, M)
    i8 = upper(mmt(dev, store, n, L, "i8", monkeypatch))
    fp4 = upper(mmt(dev, store, n, L, "fp4", monkeypatch))
    assert np.array_equal(fp4, i8)
    assert np.array_equal(fp4, upper(exact(M)))


@pytest.mark.parametrize("n,L", [(203, 3001), (1000, 257), (129, 999), (5, 1000), (1, 1), (2, 255), (224, 512),
                                 (225, 513), (449, 4097)])
@pytest.mark.parametrize("layout", ["kb", "rowmajor"])
def test_ragged_shapes_both_layouts(dev, monkeypatch, n, L, layout):
    device, torch = dev
    M = (synth.genotypes(n, L, seed=n * 131 + L).astype(np.int8) - 1)
    ref = upper(exact(M))
    if layout == "kb":
        got = mmt(dev, kblocked(torch, M), n, L, "fp4", monkeypatch)
    else:
        got = mmt(dev, rowmajor(torch, M, device.store_pitch(L)), n, L, "fp4", monkeypatch, kblocked_layout=False)
    assert np.array_equal(upper(got), ref)


def test_markers_past_kcols_are_ignored(dev, monkeypatch):
    """The packed operand zeroes every marker >= kcols, whatever the store holds there."""
    device, torch = dev
    n, L, kcols = 70, 1000, 777
    M = (synth.genotypes(n, L, seed=3).astype(np.int8) - 1)
    M[:, kcols:] = 1
    ref = upper(exact(M[:, :kcols]))
    assert np.array_equal(upper(mmt(dev, kblocked(torch, M), n, kcols, "fp4", monkeypatch)), ref)
    assert np.array_equal(upper(mmt(dev, rowmajor(torch, M), n, kcols, "fp4", monkeypatch, kblocked_layout=False)), ref)


def test_many_tiles_and_k_split(dev, monkeypatch):
    device, torch = dev
    for n, L, chunk in [(1500, 3000, None), (150, 300000, None), (150, 300000, 4096), (700, 20000, 512)]:
        M = (synth.genotypes(n, L, seed=42).astype(np.int8) - 1)
        store = kblocked(torch, M)
        fp4 = upper(mmt(dev, store, n, L, "fp4", monkeypatch, chunk=chunk))
        assert np.array_equal(fp4, upper(mmt(dev, store, n, L, "i8", monkeypatch))), (n, L, chunk)
        assert np.array_equal(fp4, upper(exact(M))), (n, L, chunk)


def test_accumulates_into_existing_c32(dev, monkeypatch):
    device, torch = dev
    n, L = 300, 5000
    M = (synth.genotypes(n, L, seed=9).astype(np.int8) - 1)
    C0 = np.random.default_rng(1).integers(-1 << 20, 1 << 20, (n, n)).astype(np.int32)
    C32 = torch.from_numpy(C0).cuda()
    got = mmt(dev, kblocked(torch, M), n, L, "fp4", monkeypatch, C32=C32, zero=False)
    assert np.array_equal(upper(got), upper(C0.astype(np.int64) + exact(M)))


def test_selected_loci_both_modes(monkeypatch, synth_small):
    s = synth_small
    dims = (s["n"], s["L"])
    for mode in ("i8", "fp4"):
        api.cache_clear()
        if mode == "i8":
            monkeypatch.setenv("EAGLE_MMT_MODE", "i8")
        else:
            monkeypatch.delenv("EAGLE_MMT_MODE", raising=False)
        for sel in ([NA], [5.0, 17.0, 2999.0]):
            assert np.array_equal(api.calculateMMt_rcpp(s["M"], 8, 1, sel, dims), eo.calculateMMt_rcpp(s["M"], 8, 1, sel, dims))
    api.cache_clear()
    monkeypatch.delenv("EAGLE_MMT_MODE", raising=False)


def test_upload_chunks_and_store_path(tmp_path, monkeypatch):
    """The product accumulated during the upload of a K-blocked store, in both modes."""
    n, L = 260, 9000
    G = synth.genotypes(n, L, seed=77)
    m = str(tmp_path / "M.ascii")
    npo.write_ascii(m, G)
    Gi = G.astype(np.float64) - 1
    ref = Gi @ Gi.T
    for mode in ("i8", "fp4"):
        api.cache_clear()
        if mode == "i8":
            monkeypatch.setenv("EAGLE_MMT_MODE", "i8")
        else:
            monkeypatch.delenv("EAGLE_MMT_MODE", raising=False)
        assert np.array_equal(api.calculateMMt_rcpp(m, 8, 1, [NA], (n, L)), ref), mode
    api.cache_clear()
