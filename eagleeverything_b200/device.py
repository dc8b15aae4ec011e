"""Device-resident pipeline: torch owns the HBM buffers and streams (plumbing), libeaglegpu's
`eg_dev_*` entry points do all of the work.  Used by bench.py (inputs already resident in HBM), by
the multi-GPU layer (dist.py) and by the device-level parity tests.

Nothing here computes on the CPU or with torch ops on the hot path; torch is used for
allocation, the current stream, and (in dist.py) the NCCL all-reduce.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def store_pitch(cols: int) -> int:
    """Row pitch of a genotype store: one spare zero column, rounded to 128 bytes."""
    return (cols + 1 + 127) // 128 * 128


def init(device: int):
    lib = _lib.require_gpu()
    torch.cuda.set_device(device)
    _lib.check(lib.eg_init(int(device)))
    return lib


def synth_ascii(rows, cols, seed, col_offset=0, n_total=None, row_offset=0, device=None):
    """Synthetic M.ascii image in HBM: uint8 tensor of rows*(cols+1) bytes (+64 bytes of slack)."""
    lib = _lib.load()
    img = torch.empty(rows * (cols + 1) + 64, dtype=torch.uint8, device=device or "cuda")
    img[rows * (cols + 1):].zero_()
    _lib.check(lib.eg_dev_synth_ascii(_ptr(img), rows, cols, col_offset, rows if n_total is None else n_total,
                                      row_offset, C.c_uint64(seed), _stream()))
    return img


def decode(img, src_pitch, rows, cols, out=None, err=None, src_offset=0):
    """K1.  img: uint8 tensor holding the ASCII bytes; returns int8 tensor (rows, pitch)."""
    lib = _lib.load()
    pitch = store_pitch(cols)
    if out is None:
        out = torch.empty((rows, pitch), dtype=torch.int8, device=img.device)
    if err is None:
        err = torch.zeros(4, dtype=torch.int32, device=img.device)
    _lib.check(lib.eg_dev_decode(C.c_void_p(img.data_ptr() + src_offset), src_pitch, img.numel() - src_offset, rows, cols,
                                 _ptr(out), out.stride(0), _ptr(err), _stream()))
    return out, err


def decode_kb(img, src_pitch, rows, cols, out=None, err=None, src_offset=0):
    """K1 into the K-blocked layout of M stores: int8 tensor (ceil(cols/128), rows, 128)."""
    lib = _lib.load()
    kb = (cols + 127) // 128
    if out is None:
        out = torch.empty((kb, rows, 128), dtype=torch.int8, device=img.device)
    if err is None:
        err = torch.zeros(4, dtype=torch.int32, device=img.device)
    _lib.check(lib.eg_dev_decode_kb(C.c_void_p(img.data_ptr() + src_offset), src_pitch, img.numel() - src_offset, rows,
                                    cols, _ptr(out), rows, 0, _ptr(err), _stream()))
    return out, err


def decode_bed(bed, n, L, kblocked=True, out=None, missing=None):
    """A SNP-major PLINK .bed file image in HBM (uint8 tensor, header included) -> the K-blocked M store
    (ceil(L/128), n, 128) like decode_kb, or (kblocked=False) the row-major Mt store (L, pitch(n)) like transpose_kb.
    missing: optional one-element int64 tensor that accumulates the number of missing genotypes."""
    lib = _lib.load()
    bpr = (n + 3) // 4
    if bed.numel() != 3 + L * bpr:
        raise ValueError(f"a .bed image of {L} SNPs x {n} individuals has {3 + L * bpr} bytes, not {bed.numel()}")
    head = bytes(bed[:3].cpu().tolist())
    if head != b"\x6c\x1b\x01":
        raise ValueError(f"not a SNP-major PLINK .bed image (header {head.hex()}, expected 6c1b01)")
    if out is None:
        shape = ((L + 127) // 128, n, 128) if kblocked else (L, store_pitch(n))
        out = torch.empty(shape, dtype=torch.int8, device=bed.device)
    _lib.check(lib.eg_dev_decode_bed(C.c_void_p(bed.data_ptr() + 3), n, L, _ptr(out), L, 0 if kblocked else out.stride(0), 0,
                                     None if missing is None else _ptr(missing), _stream()))
    return out


def transpose_kb(store_kb, rows, cols, out=None):
    """K-blocked M store (ceil(cols/128), rows, 128) -> row-major Mt store (cols, pitch(rows))."""
    lib = _lib.load()
    if out is None:
        out = torch.empty((cols, store_pitch(rows)), dtype=torch.int8, device=store_kb.device)
    _lib.check(lib.eg_dev_transpose_kb_i8(_ptr(store_kb), rows, cols, _ptr(out), out.stride(0), _stream()))
    return out


def syrk_kb(store_kb, n, kcols, C32=None, zero=True):
    """K2 on a K-blocked M store."""
    lib = _lib.load()
    if C32 is None:
        C32 = torch.empty((n, n), dtype=torch.int32, device=store_kb.device)
    if zero:
        C32.zero_()
    _lib.check(lib.eg_dev_syrk_i8_kb(_ptr(store_kb), n, kcols, _ptr(C32), C32.stride(0), _stream()))
    return C32


def transpose(store, rows, cols, out=None):
    lib = _lib.load()
    if out is None:
        out = torch.empty((cols, store_pitch(rows)), dtype=torch.int8, device=store.device)
    _lib.check(lib.eg_dev_transpose_i8(_ptr(store), rows, cols, store.stride(0), _ptr(out), out.stride(0), _stream()))
    return out


def syrk(store, n, kcols, C32=None, zero=True):
    """K2.  store: int8 (n, pitch).  Returns int32 (n, n) whose upper triangle holds M*M^T."""
    lib = _lib.load()
    if C32 is None:
        C32 = torch.empty((n, n), dtype=torch.int32, device=store.device)
    if zero:
        C32.zero_()
    _lib.check(lib.eg_dev_syrk_i8(_ptr(store), n, kcols, store.stride(0), _ptr(C32), C32.stride(0), _stream()))
    return C32


def syrk_zero_cols(store, n, zero_cols, C32):
    lib = _lib.load()
    z = np.asarray(list(zero_cols), dtype=np.int64)
    _lib.check(lib.eg_dev_syrk_zero_cols(_ptr(store), n, store.stride(0), z.ctypes.data_as(C.POINTER(C.c_int64)), len(z),
                                         _ptr(C32), C32.stride(0), _stream()))
    return C32


def mmt_finalize(C32, n, out=None):
    lib = _lib.load()
    if out is None:
        out = torch.empty((n, n), dtype=torch.float64, device=C32.device)
    _lib.check(lib.eg_dev_mmt_finalize(_ptr(C32), n, C32.stride(0), _ptr(out), _stream()))
    return out


def scan_prepare(S, V, a, n, Wp=None, tmp=None):
    """Pre-products of K3 (cuBLAS): v = S a, W = S (V S), packed.  S, V: (n, n) column-major content."""
    lib = _lib.load()
    if Wp is None:
        Wp = torch.empty(lib.eg_scan_wp_elems(n), dtype=torch.float64, device=S.device)
    if tmp is None:
        tmp = torch.empty(n * n, dtype=torch.float64, device=S.device)
    _lib.check(lib.eg_dev_scan_prepare(_ptr(S), _ptr(V), _ptr(a), n, _ptr(tmp), _ptr(Wp), _stream()))
    return Wp


def scan_prepare_sharded(S, V, a, n, rank, world, Wp=None, tmp=None):
    """Pre-products with the columns of W = S (V S) split over the ranks (instead of replicated), the blocks
    exchanged with one broadcast per rank (NCCL), then folded on every rank.  With symmetric S, V only the upper
    triangle of W is computed and the column ranges are cut at equal cost."""
    import torch.distributed as dist
    lib = _lib.load()
    Kpad = (n + 31) // 32 * 32
    if Wp is None:
        Wp = torch.empty(lib.eg_scan_wp_elems(n), dtype=torch.float64, device=S.device)
    sym = C.c_int(0)
    _lib.check(lib.eg_dev_inputs_symmetric(_ptr(S), _ptr(V), n, C.byref(sym), _stream()))
    sym = int(sym.value)
    if not (sym and lib.eg_prep_uses_i8(n)):
        # library DGEMMs round differently for different column splits: every rank computes all of W itself, which is
        # bit-identical to the single-GPU evaluation (and negligible at the sizes where this path is taken)
        if tmp is None or tmp.numel() < n * n:
            tmp = torch.empty(n * n, dtype=torch.float64, device=S.device)
        Wp.zero_()
        _lib.check(lib.eg_dev_scan_prepare_cols(_ptr(S), _ptr(V), n, 0, n, sym, _ptr(tmp), _ptr(Wp), _stream()))
        _lib.check(lib.eg_dev_scan_fold(_ptr(S), _ptr(a), n, sym, _ptr(Wp), _stream()))
        return Wp
    if sym:
        # cost of columns [0,c): n*c (V*S) + c^2/2 (upper part of S*tmp)  ->  equal-cost cuts
        cuts = [min(n, int(round(n * ((1.0 + 3.0 * r / world) ** 0.5 - 1.0) / 32.0)) * 32) for r in range(world)] + [n]
    else:
        blk = (n + world - 1) // world
        cuts = [min(r * blk, n) for r in range(world)] + [n]
    c0, c1 = cuts[rank], cuts[rank + 1]
    need = n * max(max(cuts[r + 1] - cuts[r] for r in range(world)), 1)
    if tmp is None or tmp.numel() < need:
        tmp = torch.empty(need, dtype=torch.float64, device=S.device)
    Wp.zero_()
    _lib.check(lib.eg_dev_scan_prepare_cols(_ptr(S), _ptr(V), n, c0, c1, sym, _ptr(tmp), _ptr(Wp), _stream()))
    # ONE collective when its staging buffers are small.  W is symmetric here and only rows 0 .. c1-1 of the columns
    # [c0, c1) were computed (the rest of Wp is zero), so the UPPER TRAPEZOID of every column block is what travels:
    # packed (width x c1 doubles per block, unequal), all-gathered at the size of the largest block and copied into
    # place -- 55 % of the bytes of whole column blocks.  At n = 50,000 the staging buffers would be tens of GB and push
    # the digit slices of the pre-products out of memory: one broadcast per block there.
    Wv = Wp[: (Wp.numel() // Kpad) * Kpad].view(-1, Kpad)          # row r of this view = column r of W
    sizes = [(cuts[r + 1] - cuts[r]) * cuts[r + 1] for r in range(world)]
    smax = max(sizes)
    if (world + 1) * smax * 8 <= (4 << 30):
        mine = torch.zeros(smax, dtype=torch.float64, device=S.device)
        if c1 > c0:
            mine[: sizes[rank]].view(c1 - c0, c1).copy_(Wv[c0:c1, :c1])
        allb = torch.empty(world * smax, dtype=torch.float64, device=S.device)
        dist.all_gather_into_tensor(allb, mine)
        for r in range(world):
            if r != rank and cuts[r + 1] > cuts[r]:
                Wv[cuts[r]:cuts[r + 1], :cuts[r + 1]].copy_(allb[r * smax:r * smax + sizes[r]].view(cuts[r + 1] - cuts[r], cuts[r + 1]))
        del mine, allb
    else:
        for r in range(world):
            if cuts[r + 1] > cuts[r]:
                dist.broadcast(Wp[cuts[r] * Kpad:cuts[r + 1] * Kpad], src=r)
    _lib.check(lib.eg_dev_scan_fold(_ptr(S), _ptr(a), n, sym, _ptr(Wp), _stream()))
    return Wp


def scan(storeT, L, n, Wp, zero_rows=(), out_a=None, out_vara=None):
    """K3.  storeT: int8 (L, pitch >= round_up(n+1,128)) holding Mt."""
    lib = _lib.load()
    if out_a is None:
        out_a = torch.empty(L, dtype=torch.float64, device=storeT.device)
    if out_vara is None:
        out_vara = torch.empty(L, dtype=torch.float64, device=storeT.device)
    z = np.asarray(list(zero_rows), dtype=np.int64)
    _lib.check(lib.eg_dev_scan(_ptr(storeT), L, n, storeT.stride(0), _ptr(Wp), z.ctypes.data_as(C.POINTER(C.c_int64)),
                               len(z), _ptr(out_a), _ptr(out_vara), _stream()))
    return out_a, out_vara


def argmax_tsq(a, vara, out=None):
    """K5.  Returns (best: float64[1], idx: int64[1]) device tensors."""
    lib = _lib.load()
    best = torch.empty(1, dtype=torch.float64, device=a.device)
    idx = torch.empty(1, dtype=torch.int64, device=a.device)
    _lib.check(lib.eg_dev_argmax_tsq(_ptr(a), _ptr(vara), a.numel(), _ptr(best), _ptr(idx), _stream()))
    return best, idx


def gemv_i8(storeT, L, n, x, scale=1.0):
    lib = _lib.load()
    y = torch.empty(L, dtype=torch.float64, device=storeT.device)
    _lib.check(lib.eg_dev_gemv_i8(_ptr(storeT), L, n, storeT.stride(0), _ptr(x), float(scale), _ptr(y), _stream()))
    return y


def extract_col(store, n, col, kblocked=False):
    lib = _lib.load()
    out = torch.empty(n, dtype=torch.int32, device=store.device)
    _lib.check(lib.eg_dev_extract_col(_ptr(store), n, 0 if kblocked else store.stride(0), col, _ptr(out), _stream()))
    return out
