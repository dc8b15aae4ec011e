"""Exact restatements of the digit-slice kernels of the cached-projection search route, in plain numpy / torch.

The projection (scan_i8.cu, eg_dev_project_i8) and the exact matrix-vector product (layout.cu, eg_dev_gemv_i8) write
every column k of their FP64 operand as  U_ik = 2^(e_k - 55) X_ik + r,  X_ik = rint(U_ik 2^(55 - e_k)),  with e_k taken
from the column's largest magnitude, and return  RN(sum_i m_ji X_ik) 2^(e_k - 55):  ONE rounding of an exact integer sum,
then an exact power-of-two scale.  Here the same integer sum is formed with three FP64 GEMMs on 19-bit pieces of X:
every partial sum is an integer below 2^53, so the GEMMs are exact in any summation order, and the one rounding is
applied explicitly.  So the kernels can be held to equality.

tests/test_digits_cpu.py proves these functions against Python integers and fractions.Fraction.
"""
import numpy as np
import torch

BITS = 55                      # scale_k = 2^(e_k - 55): 7 balanced base-256 digits, top digit in [-127, 127]
TOP = 0.9921875                # 127/128: a column maximum whose frexp mantissa reaches this gets e_k + 1
_P19 = float(2 ** 19)
_P38 = float(2 ** 38)


def colscale(U, full=True):
    """(e, scale) per column of U (rows = the contracted index), as si_colscale_kernel / gv_slice_kernel compute them:
    e with  max_i |U_ik| 2^-e  in [0.5, 127/128)  (frexp, bumped by one at >= 127/128 so the top digit stays <= 127),
    scale = 2^(e - 55).  A zero column gives e = 0, scale = 0; a column holding NaN or Inf gives scale = NaN.  A column
    whose largest magnitude is below 2^-1020 (e < -1019) gets scale = ldexp(1, e - 55) = 0: its products flush to zero.
    full=False: only rows i <= k count (the scan's triangular U).  U: numpy array or torch tensor, 2-D."""
    if isinstance(U, torch.Tensor):
        m = np.zeros(U.shape[1])
        for c0 in range(0, U.shape[1] if U.shape[0] else 0, 2048):     # column blocks: no full-size temporary
            A = U[:, c0:c0 + 2048].abs()
            if not full:
                A = torch.triu(A, diagonal=c0)
            m[c0:c0 + A.shape[1]] = A.amax(dim=0).double().cpu().numpy()
    else:
        A = np.abs(np.asarray(U, dtype=np.float64))
        if not full:
            A = np.triu(A)
        m = A.max(axis=0) if A.shape[0] else np.zeros(A.shape[1])
    mant, e = np.frexp(m)
    e = np.where(mant >= TOP, e + 1, e).astype(np.int64)
    bad = ~np.isfinite(m)
    zero = m == 0
    e[bad | zero] = 0
    scale = np.ldexp(1.0, e - BITS)
    scale[zero] = 0.0
    scale[bad] = np.nan
    return e, scale


def _pow2_t(k, device):
    """2^k as float64 tensors, exact for integer k in [-1022, 1023]"""
    k = torch.as_tensor(np.asarray(k, dtype=np.int64), device=device)
    return ((k + 1023) << 52).view(torch.float64)


def integer_digits(U, e):
    """X = rint(U 2^(55 - e)) per column (float64 holding integers, |X| <= 127 2^48); non-finite entries give 0 like the
    kernels' `fabs(v) < 3.6e16 ? rint(v) : 0`.  The scaling is exact: up-scaling never rounds, and a down-scaling
    exponent (e > 55) stays inside the normal range."""
    if isinstance(U, torch.Tensor):
        k = BITS - np.asarray(e, dtype=np.int64)
        h1 = np.where(k > 0, k // 2, k)
        v = U * _pow2_t(h1, U.device) * _pow2_t(k - h1, U.device)
        return torch.where(v.abs() < 3.6e16, torch.round(v), torch.zeros((), dtype=v.dtype, device=v.device))
    v = np.ldexp(np.asarray(U, dtype=np.float64), BITS - np.asarray(e, dtype=np.int64))
    with np.errstate(invalid="ignore"):
        return np.where(np.abs(v) < 3.6e16, np.rint(v), 0.0)


def balanced_digits(X):
    """the 7 balanced base-256 digits the slice kernels store for an integer X (Python int), most significant first:
    X = sum_s q_s 256^(6-s), q_1..q_6 in [-128, 127]"""
    q = []
    for _ in range(6):
        d = ((X & 0xFF) ^ 0x80) - 0x80
        q.append(d)
        X = (X - d) >> 8
    return [X] + q[::-1]


def _exact_sum_rounded(Mf, X):
    """RN(Mf @ X) for Mf with entries in {-1, 0, 1} and integer X (|X| < 2^55), both float64 tensors of one device"""
    Xa = torch.floor(X / _P38)
    r = X - Xa * _P38                      # [0, 2^38)
    Xb = torch.floor(r / _P19)
    Xc = r - Xb * _P19                     # [0, 2^19)
    Sa, Sb, Sc = Mf @ Xa, Mf @ Xb, Mf @ Xc   # integers below n 2^19: exact in any order
    h = Sa * _P19 + Sb                     # exact for n < 2^17
    return h * _P19 + Sc                   # the one rounding


def digits_exact_product(Mt, U, col_block=2048):
    """B_ref = RN(sum_i m_ji X_ik) 2^(e_k - 55): what eg_dev_project_i8 returns for B = Mt U, bit for bit.
    Mt: int8 torch tensor (L, >= n), the first n columns are the store's values; U: float64 torch tensor (n, m) on the
    same device.  Column blocks keep the GEMM operands small (n = 65,537 fits next to U)."""
    n = U.shape[0]
    assert n < 2 ** 17
    e, scale = colscale(U)
    Mf = Mt[:, :n].to(torch.float64)
    out = torch.empty((Mt.shape[0], U.shape[1]), dtype=torch.float64, device=U.device)
    sc = torch.from_numpy(scale).to(U.device)
    for c0 in range(0, U.shape[1], col_block):
        c1 = min(c0 + col_block, U.shape[1])
        X = integer_digits(U[:, c0:c1], e[c0:c1])
        out[:, c0:c1] = _exact_sum_rounded(Mf, X) * sc[c0:c1]     # power-of-two scale: exact
        del X
    return out


def gemv_exact(Mt, x, scale):
    """y = (-scale) (RN(sum_i m_ji X_i) 2^(e - 55)): eg_dev_gemv_i8 on its default path, bit for bit.  The negation
    mirrors the entry point (the store holds the negated genotypes); the product with -scale is the second rounding."""
    n = x.shape[0]
    e, sc = colscale(x.reshape(n, 1))
    X = integer_digits(x.reshape(n, 1), e)
    v = _exact_sum_rounded(Mt[:, :n].to(torch.float64), X)[:, 0]
    return (-float(scale)) * (v * float(sc[0]))


def same(a, b):
    """equal values, NaN where the other is NaN (zeros compare equal whatever their sign)"""
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())
