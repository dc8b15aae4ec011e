"""Host-side mirror of the reference's Rcpp exports for the genome-scan hot path.

Same function names, argument order, argument meaning and error behaviour as
/root/reference/MyPackage/Eagle/src/RcppExports.cpp:9, 37, 54, 73, 129 (and the R closures in
R/RcppExports.R:4-38), so that the parity tests read like calls into the R package.  Every
function forwards to the C ABI of libeaglegpu.so (include/eagle_gpu.h); none computes anything
on the CPU.  R is not installed in this image, so this module plays the role the generated
RcppExports glue plays in the package (the real glue is in eagleeverything_b200/rcpp/).
"""
from __future__ import annotations

import ctypes as C
import os
import struct

import numpy as np

from . import _lib

#: R's NA_real_; `selected_loci = [NA_REAL]` means "no selected loci" (R/AM.R:260).
NA_REAL = struct.unpack("<d", struct.pack("<Q", 0x7FF00000000007A2))[0]


def _d(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _dims(dims):
    return (C.c_int64 * 2)(int(dims[0]), int(dims[1]))


def _sel(selected_loci):
    return np.atleast_1d(np.asarray(selected_loci, dtype=np.float64)).copy()


def _msg(message):
    if message is None:
        return _lib.MESSAGE_FN(0), None
    cb = _lib.MESSAGE_FN(lambda ctx, text: message(text.decode("utf-8", "replace")))
    return cb, cb


def ReadBlock(asciifname, start_row, numcols, numrows_in_block):
    """ReadBlock.cpp:16-68 -> float64 (numrows x numcols), column-major, values -1/0/1."""
    lib = _lib.require_gpu()
    out = np.empty((int(numrows_in_block), int(numcols)), dtype=np.float64, order="F")
    _lib.check(lib.eg_ReadBlock(os.fsencode(asciifname), int(start_row), int(numcols), int(numrows_in_block), _d(out)))
    return out


def calculateMMt_rcpp(f_name_ascii, max_memory_in_Gbytes, num_cores, selected_loci, dims, quiet=True, message=None):
    """calculateMMt_rcpp.cpp:19-185; dims = (n, L).  -> float64 (n, n)."""
    lib = _lib.require_gpu()
    n = int(dims[0])
    out = np.empty((n, n), dtype=np.float64, order="F")
    s = _sel(selected_loci)
    cb, keep = _msg(message)
    _lib.check(lib.eg_calculateMMt_rcpp(os.fsencode(f_name_ascii), float(max_memory_in_Gbytes), int(num_cores), _d(s),
                                        len(s), _dims(dims), int(bool(quiet)), cb, None, _d(out)))
    return out


def calculate_a_and_vara_rcpp(f_name_ascii, selected_loci, inv_MMt_sqrt, dim_reduced_vara, max_memory_in_Gbytes,
                              dims, a, quiet=True, message=None):
    """calculate_a_and_vara_rcpp.cpp:22-241; dims = (L, n) of Mt.  -> dict(a=(L,1), vara=(L,1))."""
    lib = _lib.require_gpu()
    L, n = int(dims[0]), int(dims[1])
    S = np.asfortranarray(inv_MMt_sqrt, dtype=np.float64)
    V = np.asfortranarray(dim_reduced_vara, dtype=np.float64)
    av = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1))
    if S.shape != (n, n) or V.shape != (n, n) or av.shape != (n,):
        raise ValueError("inv_MMt_sqrt / dim_reduced_vara must be n x n and a of length n (dims = (L, n))")
    oa = np.empty(L, dtype=np.float64)
    ov = np.empty(L, dtype=np.float64)
    s = _sel(selected_loci)
    cb, keep = _msg(message)
    _lib.check(lib.eg_calculate_a_and_vara_rcpp(os.fsencode(f_name_ascii), _d(s), len(s), _d(S), _d(V),
                                                float(max_memory_in_Gbytes), _dims(dims), _d(av), int(bool(quiet)),
                                                cb, None, _d(oa), _d(ov)))
    return {"a": oa.reshape(L, 1), "vara": ov.reshape(L, 1)}


def calculate_reduced_a_rcpp(f_name_ascii, varG, P, y, max_memory_in_Gbytes, dims, selected_loci, quiet=True,
                             message=None):
    """calculate_reduced_a_rcpp.cpp:20-171; dims = (n, L) of M, file = Mt.ascii.  -> float64 (L, 1)."""
    lib = _lib.require_gpu()
    n, L = int(dims[0]), int(dims[1])
    Pm = np.asfortranarray(P, dtype=np.float64)
    yv = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    if Pm.shape != (n, n) or yv.shape != (n,):
        raise ValueError("P must be n x n and y of length n (dims = (n, L))")
    out = np.empty(L, dtype=np.float64)
    s = _sel(selected_loci)
    cb, keep = _msg(message)
    _lib.check(lib.eg_calculate_reduced_a_rcpp(os.fsencode(f_name_ascii), float(varG), _d(Pm), _d(yv),
                                               float(max_memory_in_Gbytes), _dims(dims), _d(s), len(s),
                                               int(bool(quiet)), cb, None, _d(out)))
    return out.reshape(L, 1)


def extract_geno_rcpp(f_name_ascii, max_memory_in_Gbytes, selected_locus, dims):
    """extract_geno_rcpp.cpp:17-86; dims = (n, L); selected_locus 0-based.  -> int32 (n,)."""
    lib = _lib.require_gpu()
    out = np.empty(int(dims[0]), dtype=np.int32)
    _lib.check(lib.eg_extract_geno_rcpp(os.fsencode(f_name_ascii), float(max_memory_in_Gbytes), int(selected_locus),
                                        _dims(dims), out.ctypes.data_as(C.POINTER(C.c_int32))))
    return out


def createM_ASCII_rcpp(f_name, f_name_ascii, type, AA, AB, BB, max_memory_in_Gbytes, dims, quiet=True, message=None,
                       missing="NA"):
    """createM_ASCII_rcpp.cpp:19-106 (text files: CreateASCIInospace.cpp:17-164, tokenised on the device).
    dims = (rows, columns) of the text file.  -> bool, the reference's return value."""
    lib = _lib.require_gpu()
    cb, keep = _msg(message)
    ok = C.c_int(0)
    _lib.check(lib.eg_createM_ASCII_rcpp(os.fsencode(f_name), os.fsencode(f_name_ascii), str(type).encode(), str(AA).encode(),
                                         str(AB).encode(), str(BB).encode(), float(max_memory_in_Gbytes), _dims(dims),
                                         int(bool(quiet)), cb, None, str(missing).encode(), C.byref(ok)))
    return bool(ok.value)


def createMt_ASCII_rcpp(f_name, f_name_ascii, type, max_memory_in_Gbytes, dims, quiet=True, message=None):
    """createMt_ASCII_rcpp.cpp:15-245: f_name = M.ascii with dims = (n, L); writes Mt.ascii to f_name_ascii."""
    lib = _lib.require_gpu()
    cb, keep = _msg(message)
    _lib.check(lib.eg_createMt_ASCII_rcpp(os.fsencode(f_name), os.fsencode(f_name_ascii), str(type).encode(),
                                          float(max_memory_in_Gbytes), _dims(dims), int(bool(quiet)), cb, None))


def ReshapeM_rcpp(fnameM, fnameMt, indxNA, dims):
    """ReshapeM_rcpp.cpp:16-117: writes fnameM + "tmp" / fnameMt + "tmp" without the individuals indxNA (0-based, decreasing
    as R passes them); dims = (n, L).  -> [rows kept, L]."""
    lib = _lib.require_gpu()
    idx = np.asarray(list(indxNA), dtype=np.int64)
    out = (C.c_int64 * 2)()
    _lib.check(lib.eg_ReshapeM_rcpp(os.fsencode(fnameM), os.fsencode(fnameMt), idx.ctypes.data_as(C.POINTER(C.c_int64)), len(idx),
                                    _dims(dims), out))
    return [int(out[0]), int(out[1])]


def getRowColumn(fname):
    """getRowColumn.cpp:19-72 -> [rows, columns] of a marker text file."""
    lib = _lib.require_gpu()
    out = (C.c_int64 * 2)()
    _lib.check(lib.eg_getRowColumn(os.fsencode(fname), out))
    return [int(out[0]), int(out[1])]


def plink_dims(prefix):
    """(n, L) of a PLINK 1 binary data set: the lines of <prefix>.fam (one per individual) and of <prefix>.bim (one per
    SNP), counted by eg_getRowColumn.  `prefix` may also be the path of the .bed file."""
    prefix = os.fspath(prefix)
    if prefix.endswith(".bed"):
        prefix = prefix[:-4]
    return getRowColumn(prefix + ".fam")[0], getRowColumn(prefix + ".bim")[0]


def bed_to_ascii(bed_path, n, L, M_ascii, Mt_ascii):
    """A SNP-major .bed file -> M.ascii and Mt.ascii as the text readers write them (include/eagle_gpu.h, eg_bed_to_ascii);
    both stores stay resident under the two names for the calculateMMt_rcpp / calculate_a_and_vara_rcpp calls that follow."""
    lib = _lib.require_gpu()
    _lib.check(lib.eg_bed_to_ascii(os.fsencode(bed_path), int(n), int(L), os.fsencode(M_ascii), os.fsencode(Mt_ascii)))


def _bed_bytes(n, L):
    return 3 + int(L) * ((int(n) + 3) // 4)


def _host_bytes(image, who):
    """(object that owns the bytes, size, address) of a .bed image: numpy uint8 array, bytes, or a contiguous CPU tensor."""
    if hasattr(image, "data_ptr"):
        if image.device.type != "cpu" or not image.is_contiguous():
            raise ValueError(f"{who}: a contiguous CPU tensor is needed")
        return image, image.numel() * image.element_size(), image.data_ptr()
    keep = np.ascontiguousarray(np.frombuffer(image, dtype=np.uint8) if isinstance(image, (bytes, bytearray))
                                else image, dtype=np.uint8).reshape(-1)
    return keep, keep.size, keep.ctypes.data


# ------------------------------------------------------------------ resident stores (host buffers in, handles out)
class GenotypeStore:
    """A decoded int8 genotype matrix resident in HBM (eg_store_t)."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)

    @classmethod
    def from_host_ascii(cls, image, rows, cols, col0=0, col1=None):
        lib = _lib.require_gpu()
        img = np.ascontiguousarray(image, dtype=np.uint8).reshape(-1)
        if img.size < rows * (cols + 1) - 1:
            raise ValueError("image is smaller than rows*(cols+1)-1 bytes")
        h = C.c_void_p()
        _lib.check(lib.eg_store_from_host_ascii(img.ctypes.data, rows, cols, col0, cols if col1 is None else col1,
                                                C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_host_ptr(cls, ptr, rows, cols, col0=0, col1=None):
        """`ptr`: address of a (possibly pinned) host buffer holding the ASCII image."""
        lib = _lib.require_gpu()
        h = C.c_void_p()
        _lib.check(lib.eg_store_from_host_ascii(C.c_void_p(ptr), rows, cols, col0, cols if col1 is None else col1,
                                                C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_host_rows(cls, image, rows, cols, row0, row1):
        lib = _lib.require_gpu()
        img = np.ascontiguousarray(image, dtype=np.uint8).reshape(-1)
        h = C.c_void_p()
        _lib.check(lib.eg_store_from_host_ascii_rows(img.ctypes.data, rows, cols, row0, row1, C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_file(cls, path, rows, cols, col0=0, col1=None):
        lib = _lib.require_gpu()
        h = C.c_void_p()
        _lib.check(lib.eg_store_from_file(os.fsencode(path), rows, cols, col0, cols if col1 is None else col1,
                                          C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_bed(cls, path, n, L, snp0=0, snp1=None, kblocked=True):
        """SNPs [snp0, snp1) of a SNP-major PLINK .bed file (n individuals, L SNPs) -> the K-blocked M store (kblocked) or
        the row-major Mt store.  The store's `n_missing` counts the missing genotypes read (stored as heterozygotes)."""
        lib = _lib.require_gpu()
        h, miss = C.c_void_p(), C.c_int64()
        _lib.check(lib.eg_store_from_bed(os.fsencode(path), int(n), int(L), int(snp0), int(L if snp1 is None else snp1),
                                         int(bool(kblocked)), C.byref(miss), C.byref(h)))
        s = cls(h.value)
        s.n_missing = miss.value
        return s

    @classmethod
    def from_host_bed(cls, image, n, L, snp0=0, snp1=None, kblocked=True):
        """As from_bed, from the whole file image in host memory: a numpy uint8 array (or bytes), or a CPU torch tensor --
        page-locked ones (pin_memory()) are copied without staging."""
        lib = _lib.require_gpu()
        keep, size, ptr = _host_bytes(image, "from_host_bed")
        if size != _bed_bytes(n, L):
            raise ValueError(f"a .bed image of {L} SNPs x {n} individuals has {_bed_bytes(n, L)} bytes, not {size}")
        h, miss = C.c_void_p(), C.c_int64()
        _lib.check(lib.eg_store_from_host_bed(C.c_void_p(ptr), int(n), int(L), int(snp0), int(L if snp1 is None else snp1),
                                              int(bool(kblocked)), C.byref(miss), C.byref(h)))
        del keep
        s = cls(h.value)
        s.n_missing = miss.value
        return s

    # -------------------------------------------------------------- streamed stores: data sets larger than device memory
    @classmethod
    def stream_file(cls, path, rows, cols, kblocked=True):
        """A store that leaves the genotypes of a no-space ASCII file on the host: M.ascii (kblocked, rows = n, cols = L) or
        Mt.ascii (rows = L, cols = n).  mmt / extract_col (M) and a_and_vara (Mt) decode the file piece by piece on every
        call, with the resident store's results; transpose and the packed export are refused (include/eagle_gpu.h)."""
        lib = _lib.require_gpu()
        h = C.c_void_p()
        _lib.check(lib.eg_store_stream_file(os.fsencode(path), int(rows), int(cols), int(bool(kblocked)), C.byref(h)))
        return cls(h.value)

    @classmethod
    def stream_bed(cls, path, n, L, snp0=0, snp1=None, kblocked=True):
        """As stream_file, from SNPs [snp0, snp1) of a SNP-major .bed file, in either orientation."""
        lib = _lib.require_gpu()
        h = C.c_void_p()
        _lib.check(lib.eg_store_stream_bed(os.fsencode(path), int(n), int(L), int(snp0), int(L if snp1 is None else snp1),
                                           int(bool(kblocked)), C.byref(h)))
        return cls(h.value)

    @classmethod
    def stream_host_bed(cls, image, n, L, snp0=0, snp1=None, kblocked=True):
        """As stream_bed, from the whole .bed image in host memory (numpy uint8 array, bytes, or a CPU torch tensor; pinned
        ones are copied without staging).  The store keeps a reference to the image: the library reads it on every call."""
        lib = _lib.require_gpu()
        keep, size, ptr = _host_bytes(image, "stream_host_bed")
        if size != _bed_bytes(n, L):
            raise ValueError(f"a .bed image of {L} SNPs x {n} individuals has {_bed_bytes(n, L)} bytes, not {size}")
        h = C.c_void_p()
        _lib.check(lib.eg_store_stream_host_bed(C.c_void_p(ptr), int(n), int(L), int(snp0), int(L if snp1 is None else snp1),
                                                int(bool(kblocked)), C.byref(h)))
        s = cls(h.value)
        s._source = keep
        return s

    def info(self):
        r, c, p = C.c_int64(), C.c_int64(), C.c_int64()
        d = C.c_void_p()
        _lib.check(_lib.load().eg_store_info(self._h, C.byref(r), C.byref(c), C.byref(p), C.byref(d)))
        return dict(rows=r.value, cols=c.value, pitch=p.value, device_ptr=d.value)

    def transpose(self):
        h = C.c_void_p()
        _lib.check(_lib.load().eg_store_transpose(self._h, C.byref(h)))
        return GenotypeStore(h.value)

    def mmt(self, zero_cols=()):
        n = self.info()["rows"]
        out = np.empty((n, n), dtype=np.float64, order="F")
        z = np.asarray(list(zero_cols), dtype=np.int64)
        _lib.check(_lib.load().eg_store_mmt(self._h, z.ctypes.data_as(C.POINTER(C.c_int64)), len(z), _d(out)))
        return out

    def a_and_vara(self, inv_MMt_sqrt, dim_reduced_vara, a, zero_rows=()):
        i = self.info()
        L, n = i["rows"], i["cols"]
        S = np.asfortranarray(inv_MMt_sqrt, dtype=np.float64)
        V = np.asfortranarray(dim_reduced_vara, dtype=np.float64)
        av = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1))
        assert S.shape == (n, n) and V.shape == (n, n) and av.shape == (n,)
        oa, ov = np.empty(L), np.empty(L)
        z = np.asarray(list(zero_rows), dtype=np.int64)
        _lib.check(_lib.load().eg_store_a_and_vara(self._h, z.ctypes.data_as(C.POINTER(C.c_int64)), len(z), _d(S),
                                                   _d(V), _d(av), _d(oa), _d(ov)))
        return oa, ov

    def extract_col(self, col):
        out = np.empty(self.info()["rows"], dtype=np.int32)
        _lib.check(_lib.load().eg_store_extract_col(self._h, int(col), out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def free(self):
        if self._h:
            _lib.load().eg_store_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# ----------------------------------------------------------------------------- SURVEY.md section 8(f) rank 1
# The n x n algebra between two scans: R functions of the same names (R/calculateMMt_sqrt_and_sqrtinv.R,
# R/calculateH.R, R/calculateP.R, R/calculate_reduced_a.R, R/calculate_reduced_vara.R), same argument order;
# `ngpu` is accepted and ignored as in the reference's current R code.
def _f(a):
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


def calculateMMt_sqrt_and_sqrtinv(MMt, checkres=True, quiet=True, ngpu=0, message=None):
    """-> dict(sqrt_MMt=..., inverse_sqrt_MMt=...), or None after the reference's messages when MMt is not
    positive definite (calculateMMt_sqrt_and_sqrtinv.R:14-21)."""
    lib = _lib.require_gpu()
    K = _f(MMt)
    n = K.shape[0]
    sq, inv = np.empty((n, n), order="F"), np.empty((n, n), order="F")
    ok = C.c_int(0)
    cb, keep = _msg(message)
    _lib.check(lib.eg_calculateMMt_sqrt_and_sqrtinv(_d(K), n, int(bool(checkres)), cb, None, _d(sq), _d(inv), C.byref(ok)))
    return dict(sqrt_MMt=sq, inverse_sqrt_MMt=inv) if ok.value else None


def calculateH(MMt, varE, varG, message=None):
    """H = varE * I + varG * MMt (calculateH.R:36); None with the reference's message for a negative variance."""
    lib = _lib.require_gpu()
    K = _f(MMt)
    n = K.shape[0]
    H = np.empty((n, n), order="F")
    ok = C.c_int(0)
    cb, keep = _msg(message)
    _lib.check(lib.eg_calculateH(_d(K), n, float(varE), float(varG), cb, None, _d(H), C.byref(ok)))
    return H if ok.value else None


def calculateP(H, X, ngpu=0, message=None):
    """P = Hinv - Hinv X (X' Hinv X)^-1 X' Hinv (calculateP.R:27-28)."""
    lib = _lib.require_gpu()
    Hf, Xf = _f(H), _f(np.asarray(X, dtype=np.float64).reshape(np.asarray(H).shape[0], -1))
    if Hf.shape[0] != Xf.shape[0]:
        if message:
            message(" The number of rows in H and X are not the same.")
        return None
    n, q = Xf.shape
    P = np.empty((n, n), order="F")
    _lib.check(lib.eg_calculateP(_d(Hf), _d(Xf), n, q, _d(P)))
    return P


def calculate_reduced_a(varG, P, MMtsqrt, y, quiet=True, message=None):
    """varG * MMtsqrt %*% P %*% y (calculate_reduced_a.R:31) -> (n, 1)."""
    lib = _lib.require_gpu()
    Pf, Sf = _f(P), _f(MMtsqrt)
    yv = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    n = Pf.shape[0]
    if n != yv.size:
        if message:
            message(" Error:  there is a problem with the  dimensions of  P, and/or the vector y.")
        return None
    out = np.empty(n)
    _lib.check(lib.eg_calculate_reduced_a(float(varG), _d(Pf), _d(Sf), _d(yv), n, _d(out)))
    return out.reshape(n, 1)


def calculate_reduced_vara(X, varE, varG, invMMt, MMtsqrt, quiet=True, message=None):
    """calculate_reduced_vara.R:21-35 (invMMt only gives the dimension there)."""
    lib = _lib.require_gpu()
    Sf = _f(MMtsqrt)
    n = Sf.shape[0]
    Xf = _f(np.asarray(X, dtype=np.float64).reshape(n, -1))
    V = np.empty((n, n), order="F")
    _lib.check(lib.eg_calculate_reduced_vara(_d(Xf), n, Xf.shape[1], float(varE), float(varG), _d(Sf), _d(V)))
    return V


def emma_eigen_L_wo_Z(K, ngpu=0, vectors=True):
    """emma.eigen.L.wo.Z (emma_eigen_L_wo_Z.R:9): eigen(K, symmetric=TRUE) -> dict(values (decreasing), vectors)."""
    lib = _lib.require_gpu()
    Kf = _f(K)
    n = Kf.shape[0]
    w = np.empty(n)
    U = np.empty((n, n), order="F") if vectors else None
    _lib.check(lib.eg_emma_eigen_L_wo_Z(_d(Kf), n, _d(w), _d(U) if vectors else None))
    return dict(values=w, vectors=U)


def emma_eigen_R_wo_Z(K, X, ngpu=0):
    """emma.eigen.R.wo.Z (emma_eigen_R_wo_Z.R:4-20) -> dict(values (n-q), vectors (n x (n-q)))."""
    lib = _lib.require_gpu()
    Kf = _f(K)
    n = Kf.shape[0]
    Xf = _f(np.asarray(X, dtype=np.float64).reshape(n, -1))
    q = Xf.shape[1]
    w = np.empty(n - q)
    U = np.empty((n, n - q), order="F")
    _lib.check(lib.eg_emma_eigen_R_wo_Z(_d(Kf), _d(Xf), n, q, _d(w), _d(U)))
    return dict(values=w, vectors=U)


def set_scan_mode(mode):
    """'f64' / 0: FP64 tensor cores (DMMA).  'i8' / 1: exact int8 slices on the tcgen05 tensor cores."""
    m = {"f64": 0, "dmma": 0, "i8": 1}.get(mode, mode)
    _lib.check(_lib.load().eg_set_scan_mode(int(m)))


def set_scan_digits(digits):
    """7 (default) or 6 balanced base-256 digits per column of U in the int8 scan (include/eagle_gpu.h)."""
    _lib.check(_lib.load().eg_set_scan_digits(int(digits)))


def get_scan_digits():
    return int(_lib.load().eg_get_scan_digits())


def get_scan_mode():
    return int(_lib.load().eg_get_scan_mode())


def last_timing():
    out = (C.c_double * 8)()
    _lib.check(_lib.load().eg_last_timing(out, 8))
    keys = ["h2d_decode_ms", "syrk_ms", "finalize_ms", "mmt_d2h_ms", "scan_h2d_ms", "prepare_ms", "scan_ms", "scan_d2h_ms"]
    return dict(zip(keys, list(out)))


def cache_clear():
    _lib.load().eg_cache_clear()


def init_multi(ngpu, devs=None):
    """eg_init_multi: the reference's `ngpu` argument (R/AM.R:185-196) made live -- one process, one host thread per GPU,
    stores sharded by markers, NCCL over NVLink for the one exchange of each export.  Every function of this module then
    works unchanged on the sharded stores."""
    lib = _lib.require_gpu()
    arr = None if devs is None else (C.c_int * int(ngpu))(*[int(d) for d in devs])
    _lib.check(lib.eg_init_multi(int(ngpu), arr))
    return int(lib.eg_gpu_count())


def gpu_count():
    return int(_lib.load().eg_gpu_count())


def shutdown():
    _lib.check(_lib.load().eg_shutdown())
