"""numpy restatement of PLINK 1 binary genotype files (.bed, SNP-major): the bytes the .bed decoder eats, written and
read back independently of the library.  TEST INFRASTRUCTURE ONLY.

Format (include/eagle_gpu.h): header 6c 1b 01; SNP j in bytes 3 + j*ceil(n/4) .. 3 + (j+1)*ceil(n/4) - 1; individual i of
it in bits 2(i%4), 2(i%4)+1 of byte i//4; values 0 = A1/A1, 1 = missing, 2 = het, 3 = A2/A2; pad bits ignored."""
import numpy as np

BED_MAGIC = b"\x6c\x1b\x01"


def write_bed(G012, flip=None, missing=None):
    """The bytes of a SNP-major .bed file holding G012 ((n, L) codes 0 = AA, 1 = AB, 2 = BB, M orientation).
    flip: L booleans, SNPs whose .bim lists the alleles the other way round (AA written as A2/A2, BB as A1/A1);
    missing: (n, L) booleans written as missing (value 1) whatever G012 says.  Pad bits are zero."""
    G = np.asarray(G012, dtype=np.uint8)
    n, L = G.shape
    v = np.array([0, 2, 3], dtype=np.uint8)[G]
    if flip is not None:
        f = np.asarray(flip, dtype=bool)
        v[:, f] = np.array([3, 2, 0], dtype=np.uint8)[G[:, f]]
    if missing is not None:
        v[np.asarray(missing, dtype=bool)] = 1
    bpr = (n + 3) // 4
    vt = np.zeros((L, 4 * bpr), dtype=np.uint8)
    vt[:, :n] = v.T
    vt = vt.reshape(L, bpr, 4)
    rows = vt[:, :, 0] | (vt[:, :, 1] << 2) | (vt[:, :, 2] << 4) | (vt[:, :, 3] << 6)
    return BED_MAGIC + rows.astype(np.uint8).tobytes()


def read_bed(data, n, L):
    """Inverse of write_bed up to allele orientation -> (G012 (n, L) with missing read as 1, the way the text readers read
    missing genotypes; missing (n, L) booleans).  Pad bits past individual n-1 are ignored."""
    data = bytes(data)
    bpr = (n + 3) // 4
    if data[:3] != BED_MAGIC:
        raise ValueError("not a SNP-major .bed file")
    if len(data) != 3 + L * bpr:
        raise ValueError(f"{len(data)} bytes; {L} SNPs x {n} individuals need {3 + L * bpr}")
    rows = np.frombuffer(data, dtype=np.uint8, offset=3).reshape(L, bpr)
    v = ((rows[:, :, None] >> (2 * np.arange(4, dtype=np.uint8))) & 3).reshape(L, 4 * bpr)[:, :n].T
    return np.array([0, 1, 1, 2], dtype=np.uint8)[v], v == 1
