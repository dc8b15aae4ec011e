// PLINK 1 binary genotypes (.bed, SNP-major) -> int8 store, on the device.  The format contract is in include/eagle_gpu.h.
//
// A .bed SNP row is ceil(n/4) bytes, individual i in bits 2(i%4), 2(i%4)+1 of byte i/4 -- the bit order of the packed
// container (pack2.cu), with other values: 0 = A1/A1, 1 = missing, 2 = het, 3 = A2/A2.  Per 2-bit field
// c = v - ((v >> 1) & 1) maps them to the ASCII file's codes 0, 1, 1, 2 (missing -> het, the policy of the text readers)
// without a borrow between fields, so unpack16 (codes2.cuh) writes the store bytes.  Missing genotypes are
// v & ~(v >> 1) & 0x55..: counted per thread, summed per block, one atomic per block.
//
// Both kernels are bound by HBM: 1/4 byte read + 1 byte written per genotype (n = 10,000, L = 1,000,000: 2.5 GB in,
// 10 GB out per layout).  SNP rows start at any byte (ceil(n/4) need not be a multiple of 4, and a file image puts a
// 3-byte header in front), so sources are read bytewise; the reads of a warp stay contiguous, the writes are aligned
// 16-byte vectors.
#include "codes2.cuh"
#include "common.cuh"

namespace eg {

__device__ __forceinline__ uint32_t bed_codes(uint32_t v) { return v - ((v >> 1) & 0x55555555u); }
__device__ __forceinline__ uint32_t bed_missing(uint32_t v) { return v & ~(v >> 1) & 0x55555555u; }
constexpr uint32_t BED_HET4 = 0xAAu;   // four heterozygotes: what stands in for bytes past a row or block (store value 0)

// sum of every thread's count into *missing, one atomic per block; every thread of the block calls it
__device__ void block_add_missing(uint64_t mine, unsigned long long* missing) {
    __shared__ unsigned long long part[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += part[w];
        if (s && missing) atomicAdd(missing, s);
    }
}

// Row-major (Mt) store: one thread = 16 individuals of one SNP = 4 source bytes -> one 16-byte vector of the store row,
// the row's zero pad up to `pitch` included.
__global__ void __launch_bounds__(256) bed_rows_kernel(const uint8_t* __restrict__ snps, int64_t n, int64_t bpr, int64_t nsnp,
                                                       int8_t* __restrict__ dst, int64_t pitch, unsigned long long* missing) {
    const int64_t gpr = pitch >> 4, total = nsnp * gpr;
    uint64_t miss = 0;
    uint32_t unused = 0;
    for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (int64_t)gridDim.x * 256) {
        const int64_t j = t / gpr, g = t - j * gpr;
        const uint8_t* row = snps + j * bpr;
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t c = 4 * g + k;
            v |= (c < bpr ? (uint32_t)row[c] : BED_HET4) << (8 * k);
        }
        const int64_t left = n - 16 * g;   // individuals of this group that exist: the pad bits past n are ignored
        if (left < 16) {
            const uint32_t keep = left <= 0 ? 0u : (0xFFFFFFFFu >> (32 - 2 * left));
            v = (v & keep) | (0xAAAAAAAAu & ~keep);
        }
        miss += __popc(bed_missing(v));
        *reinterpret_cast<uint4*>(dst + j * pitch + 16 * g) = unpack16(bed_codes(v), unused);
    }
    block_add_missing(miss, missing);
}

// K-blocked (M) store [L/128][n][128]: a 2-bit -> int8 transpose.  A tile is one 128-SNP block x 256 individuals: 128
// source rows of 64 bytes into shared memory, then 256 store rows of 128 bytes out.  Row stride 65 in shared memory: the
// 8 lanes of a warp that read the same byte column of 8 different 16-SNP groups hit 8 different banks.
constexpr int BT_IND = 256, BT_COLS = BT_IND / 4, BT_ROWB = BT_COLS + 1;

__global__ void __launch_bounds__(256) bed_kb_kernel(const uint8_t* __restrict__ snps, int64_t n, int64_t bpr, int64_t nsnp,
                                                     int8_t* __restrict__ dst, unsigned long long* missing) {
    __shared__ uint8_t tile[128 * BT_ROWB];
    const int64_t nblk = (nsnp + 127) / 128, bands = (n + BT_IND - 1) / BT_IND;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane & 7;
    uint64_t miss = 0;
    uint32_t unused = 0;
    for (int64_t u = blockIdx.x; u < nblk * bands; u += gridDim.x) {
        const int64_t blk = u / bands, band = u - blk * bands;   // bands fastest: CTAs running together write one block
        const int64_t s0 = blk * 128, c0 = band * BT_COLS;
        __syncthreads();   // the previous tile has been written out
        for (int e = threadIdx.x; e < 128 * BT_COLS; e += 256) {
            const int s = e / BT_COLS, c = e - s * BT_COLS;
            const int64_t snp = s0 + s, byte = c0 + c;
            uint32_t b = BED_HET4;   // SNPs past the last one: the zero tail of the last marker block
            if (snp < nsnp && byte < bpr) {
                b = snps[snp * bpr + byte];
                const int64_t left = n - 4 * byte;
                if (left < 4) {
                    const uint32_t keep = (1u << (2 * left)) - 1u;
                    b = (b & keep) | (BED_HET4 & ~keep);
                }
                miss += __popc(bed_missing(b));
            }
            tile[s * BT_ROWB + c] = (uint8_t)b;
        }
        __syncthreads();
        // lane -> 16 SNPs (16 g .. 16 g + 15) x one byte column (4 individuals): four 16-byte vectors; the 8 lanes of a
        // byte column write whole 128-byte store rows
        for (int cc = warp * 4 + (lane >> 3); cc < BT_COLS; cc += 32) {
            const int64_t r = 4 * (c0 + cc);
            if (r >= n) break;
            uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int s = 0; s < 16; s++) {
                const uint32_t b = tile[(16 * g + s) * BT_ROWB + cc];
#pragma unroll
                for (int q = 0; q < 4; q++) w[q] |= ((b >> (2 * q)) & 3u) << (2 * s);
            }
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (r + q < n) *reinterpret_cast<uint4*>(dst + ((blk * n) + r + q) * 128 + 16 * g) = unpack16(bed_codes(w[q]), unused);
        }
    }
    block_add_missing(miss, missing);
}

}  // namespace eg

using namespace eg;

extern "C" int eg_dev_decode_bed(const uint8_t* d_snps, int64_t n, int64_t nsnp, int8_t* d_dst, int64_t dst_rows_or_L,
                                 int64_t dst_pitch, int64_t m0, uint64_t* d_missing, void* stream) {
    if (!d_snps || !d_dst || n <= 0 || nsnp < 0 || m0 < 0 || dst_pitch < 0 || ((uintptr_t)d_dst & 15))
        return set_error(EG_ERR_ARG, "eg_dev_decode_bed: bad argument");
    if (m0 + nsnp > dst_rows_or_L)
        return set_error(EG_ERR_ARG, "eg_dev_decode_bed: markers [%lld, %lld) outside the store's %lld", (long long)m0,
                         (long long)(m0 + nsnp), (long long)dst_rows_or_L);
    if (nsnp == 0) return EG_OK;
    const int64_t bpr = (n + 3) / 4, cap = (int64_t)num_sms() * 8;
    unsigned long long* miss = reinterpret_cast<unsigned long long*>(d_missing);
    if (dst_pitch) {
        if ((dst_pitch & 127) || dst_pitch < n) return set_error(EG_ERR_ARG, "eg_dev_decode_bed: pitch must be a multiple of 128 and >= n");
        const int64_t nb = (nsnp * (dst_pitch >> 4) + 255) / 256;
        bed_rows_kernel<<<(unsigned)(nb < cap ? nb : cap), 256, 0, (cudaStream_t)stream>>>(d_snps, n, bpr, nsnp, d_dst + m0 * dst_pitch,
                                                                                          dst_pitch, miss);
        return check_launch("bed_rows_kernel");
    }
    // K-blocked: a piece fills whole 128-marker blocks; only the store's last block may be partial (its tail is zeroed)
    if ((m0 & 127) || ((nsnp & 127) && m0 + nsnp != dst_rows_or_L))
        return set_error(EG_ERR_ARG, "eg_dev_decode_bed: K-blocked pieces start on a 128-marker block and end on one or at L");
    const int64_t units = ((nsnp + 127) / 128) * ((n + BT_IND - 1) / BT_IND);
    bed_kb_kernel<<<(unsigned)(units < cap ? units : cap), 256, 0, (cudaStream_t)stream>>>(d_snps, n, bpr, nsnp,
                                                                                          d_dst + (m0 >> 7) * n * 128, miss);
    return check_launch("bed_kb_kernel");
}
