// SURVEY.md section 8(f), rank 2 -- a packed 2-bit genotype container in place of the ASCII files for transport.
//
// Format: the one the pre-CRAN code wrote (reference: MyPackage/RcppFunctions.cpp.gpu:224-345, CreatePackedBinary):
// every row is ceil(cols/32) little-endian 64-bit words; genotype k of the row sits in bits 2(k mod 32), 2(k mod 32)+1
// of word k/32 with the code of the ASCII file (0 = AA, 1 = AB / missing, 2 = BB); a row starts on a fresh word and the
// unused bits of its last word are zero.  4 genotypes per byte: the 10 GB ASCII image of config 3 becomes 2.5 GB, which
// is what matters once the kernels are fast and the PCIe transfer is the longest stage of an end-to-end step.
//
// Both kernels are pure bandwidth kernels: one thread = one 64-bit word = 32 genotypes = two aligned 16-byte vectors of
// the int8 store (row-major, or the K-blocked layout of M stores in which 32 consecutive markers of a row stay
// contiguous because 128 is a multiple of 32).
#include "codes2.cuh"
#include "common.cuh"

namespace eg {

__global__ void __launch_bounds__(256) pack2_kernel(const int8_t* __restrict__ store, int64_t rows, int64_t cols, int64_t pitch,
                                                    uint64_t* __restrict__ words, int64_t wpr) {
    // K-blocked stores: 4 consecutive threads take the 4 words of one row inside one 128-marker block (a contiguous
    // 128-byte line of the store), then the next ROW of that block
    const int64_t wq = (wpr + 3) / 4;
    const int64_t total = pitch ? rows * wpr : rows * wq * 4;
    for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (int64_t)gridDim.x * 256) {
        int64_t r, w;
        if (pitch) { r = t / wpr; w = t - r * wpr; }
        else { r = (t >> 2) % rows; w = ((t >> 2) / rows) * 4 + (t & 3); if (w >= wpr) continue; }
        const int8_t* src = store + store_off(r, 32 * w, rows, pitch);
        uint4 a = *reinterpret_cast<const uint4*>(src), b = *reinterpret_cast<const uint4*>(src + 16);
        const int64_t left = cols - 32 * w;  // genotypes of this word that exist; the store's pad is zero = code 1: mask it
        uint64_t v = (uint64_t)pack16(a) | ((uint64_t)pack16(b) << 32);
        if (left < 32) v &= (left <= 0) ? 0ull : (~0ull >> (64 - 2 * left));
        words[r * wpr + w] = v;
    }
}

__global__ void __launch_bounds__(256) unpack2_kernel(const uint64_t* __restrict__ words, int64_t wpr, int64_t rows, int64_t cols,
                                                      int8_t* __restrict__ store, int64_t pitch, int64_t words_out,
                                                      int32_t* __restrict__ err) {
    // words_out >= wpr: word columns written per row, so that the store's zero pad is (re)written too
    const int64_t total = rows * words_out;
    uint32_t bad = 0;
    for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (int64_t)gridDim.x * 256) {
        int64_t r, w;
        if (pitch) { r = t / words_out; w = t - r * words_out; }
        else { r = (t >> 2) % rows; w = ((t >> 2) / rows) * 4 + (t & 3); }  // words_out is a multiple of 4 here
        uint64_t v = w < wpr ? words[r * wpr + w] : 0x5555555555555555ull;  // code 1 -> genotype 0 in the pad
        const int64_t left = cols - 32 * w;
        if (left < 32) {
            const uint64_t keep = left <= 0 ? 0ull : (~0ull >> (64 - 2 * left));
            if (v & ~keep & (w < wpr ? ~0ull : 0ull)) bad |= 2u;  // bits set beyond the last genotype of the row
            v = (v & keep) | (0x5555555555555555ull & ~keep);
        }
        int8_t* dst = store + store_off(r, 32 * w, rows, pitch);
        *reinterpret_cast<uint4*>(dst) = unpack16((uint32_t)v, bad);
        *reinterpret_cast<uint4*>(dst + 16) = unpack16((uint32_t)(v >> 32), bad);
        if (bad && !err[0]) {
            if (atomicExch(&err[0], 1) == 0) {
                err[1] = (int32_t)(r & 0x7FFFFFFF);
                err[2] = (int32_t)((32 * w) & 0x7FFFFFFF);
                err[3] = (int32_t)(r >> 31);
            }
        }
    }
}

}  // namespace eg

using namespace eg;

extern "C" int64_t eg_packed_words_per_row(int64_t cols) { return (cols + 31) / 32; }

// store: int8 genotypes, row-major with `pitch` bytes per row (multiple of 32, pad zero) or K-blocked (pitch == 0)
extern "C" int eg_dev_pack_2bit(const int8_t* d_store, int64_t rows, int64_t cols, int64_t pitch, uint64_t* d_words, void* stream) {
    if (!d_store || !d_words || rows <= 0 || cols <= 0 || (pitch && ((pitch & 31) || pitch < ((cols + 31) / 32) * 32)))
        return set_error(EG_ERR_ARG, "eg_dev_pack_2bit: bad argument");
    const int64_t wpr = (cols + 31) / 32, total = pitch ? rows * wpr : rows * ((wpr + 3) / 4) * 4;
    const int64_t cap = (int64_t)num_sms() * 32, nb = (total + 255) / 256;
    pack2_kernel<<<(unsigned)(nb < cap ? nb : cap), 256, 0, (cudaStream_t)stream>>>(d_store, rows, cols, pitch, d_words, wpr);
    return check_launch("pack2_kernel");
}
// d_err: 4 x int32, zeroed by the caller; err[0] != 0 after the kernel: a code 3 or stray bits near (row, column) = (err[1], err[2])
extern "C" int eg_dev_unpack_2bit(const uint64_t* d_words, int64_t rows, int64_t cols, int8_t* d_store, int64_t pitch,
                                  int32_t* d_err, void* stream) {
    if (!d_store || !d_words || !d_err || rows <= 0 || cols <= 0 || (pitch && ((pitch & 31) || pitch < ((cols + 31) / 32) * 32)))
        return set_error(EG_ERR_ARG, "eg_dev_unpack_2bit: bad argument");
    const int64_t wpr = (cols + 31) / 32;
    const int64_t words_out = pitch ? pitch / 32 : round_up(cols, 128) / 32;  // the whole padded row of the store
    const int64_t total = rows * words_out;
    const int64_t cap = (int64_t)num_sms() * 32, nb = (total + 255) / 256;
    unpack2_kernel<<<(unsigned)(nb < cap ? nb : cap), 256, 0, (cudaStream_t)stream>>>(d_words, wpr, rows, cols, d_store, pitch,
                                                                                   words_out, d_err);
    return check_launch("unpack2_kernel");
}
