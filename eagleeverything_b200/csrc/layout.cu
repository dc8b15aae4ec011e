// Small bandwidth-bound kernels around the two tensor-core kernels:
//   transpose_i8      M (n x L int8) -> Mt (L x n int8)        replaces createMt_ASCII_rcpp.cpp:99-118
//   mmt_finalize      int32 upper triangle -> symmetric double  (Rcpp::wrap of MMt, calculateMMt_rcpp.cpp:183)
//   syrk_zero_cols    rank-k correction for zeroed loci         calculateMMt_rcpp.cpp:88-92
//   extract_col       one marker column of M as int32           extract_geno_rcpp.cpp:46-48
//   argmax_tsq        tsq = a^2/vara, first index of the max    R/find_qtl.R:71-80
//   gemv_i8           y = scale * Mt * x                        calculate_reduced_a_rcpp.cpp:83-84
#include <cmath>
#include <vector>

#include <cstdlib>

#include "common.cuh"

namespace eg {

// ------------------------------------------------------------------ transpose (64 x 64 byte tiles)
constexpr int TR_TILE = 64;
// in: row-major (in_pitch) when in_kb == 0, else K-blocked [col/128][rows][128]
__global__ void __launch_bounds__(256) transpose_i8_kernel(const int8_t* __restrict__ in, int64_t rows, int64_t cols,
                                                           int64_t in_pitch, int in_kb, int8_t* __restrict__ out,
                                                           int64_t out_pitch, int64_t tiles_c) {
    __shared__ __align__(16) uint8_t tile[TR_TILE][TR_TILE + 16];
    const int t = threadIdx.x;
    for (int64_t tix = blockIdx.x; ; tix += gridDim.x) {
        const int64_t tr = tix / tiles_c, tc = tix - tr * tiles_c;
        if (tr * TR_TILE >= out_pitch) break;
        const int64_t r0 = tr * TR_TILE, c0 = tc * TR_TILE;
        __syncthreads();
        {   // load 64 rows x 64 bytes: thread -> (row t/4, 16-byte segment t%4); pitch padding is readable
            const int r = t >> 2, sgm = t & 3;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (r0 + r < rows && c0 + sgm * 16 < in_pitch) {
                const int64_t c = c0 + sgm * 16;
                v = in_kb ? *reinterpret_cast<const uint4*>(in + ((c >> 7) * rows + r0 + r) * 128 + (c & 127))
                          : *reinterpret_cast<const uint4*>(in + (r0 + r) * in_pitch + c);
            }
            *reinterpret_cast<uint4*>(&tile[r][sgm * 16]) = v;
        }
        __syncthreads();
        {   // store: out row = input column c0 + t/4, 16 consecutive input rows per thread
            const int c = t >> 2, sgm = t & 3;
            if (c0 + c < cols) {
                uint32_t w[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int rb = sgm * 16 + k * 4;
                    w[k] = (uint32_t)tile[rb][c] | ((uint32_t)tile[rb + 1][c] << 8) | ((uint32_t)tile[rb + 2][c] << 16) |
                           ((uint32_t)tile[rb + 3][c] << 24);
                }
                // rows beyond `rows` were loaded as 0, so the output pad stays zero
                if (r0 + sgm * 16 < out_pitch)
                    *reinterpret_cast<uint4*>(out + (c0 + c) * out_pitch + r0 + sgm * 16) =
                        make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
}

// ------------------------------------------------------------------ finalize: mirror + int32 -> double
__global__ void __launch_bounds__(256) mmt_finalize_kernel(const int32_t* __restrict__ C, int64_t n, int64_t ldc,
                                                           double* __restrict__ out) {
    // block (bx, by) with bx >= by handles the 32x32 tile rows by*32.., cols bx*32.. of the upper
    // triangle and writes both out[r][c] and out[c][r] (out is symmetric: row- == column-major).
    __shared__ int32_t tile[32][33];
    const int bx = blockIdx.x, by = blockIdx.y;
    if (bx < by) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const int64_t r0 = (int64_t)by * 32, c0 = (int64_t)bx * 32;
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = r0 + i, c = c0 + tx;
        int32_t v = 0;
        if (r < n && c < n) v = (c >= r) ? C[r * ldc + c] : C[c * ldc + r];
        tile[i][tx] = v;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = r0 + i, c = c0 + tx;
        if (r < n && c < n) out[r * n + c] = (double)tile[i][tx];
    }
    if (bx != by) {
        for (int i = ty; i < 32; i += 8) {
            const int64_t r = c0 + i, c = r0 + tx;  // transposed tile
            if (r < n && c < n) out[r * n + c] = (double)tile[tx][i];
        }
    }
}

// ------------------------------------------------------------------ zeroed loci as a rank-k update
// element (i, c) of an M store: row-major (pitch > 0) or K-blocked (pitch == 0)
__device__ __forceinline__ int8_t store_at(const int8_t* M, int64_t n, int64_t pitch, int64_t i, int64_t c) {
    return pitch ? M[i * pitch + c] : M[((c >> 7) * n + i) * 128 + (c & 127)];
}
__global__ void gather_cols_kernel(const int8_t* __restrict__ M, int64_t n, int64_t pitch,
                                   const int64_t* __restrict__ cols, int ncols, int8_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int s = 0; s < ncols; s++) out[i * ncols + s] = store_at(M, n, pitch, i, cols[s]);
}
__global__ void __launch_bounds__(256) syrk_zero_cols_kernel(const int8_t* __restrict__ G, int64_t n, int ncols,
                                                             int32_t* __restrict__ C, int64_t ldc) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t r = blockIdx.y;
    if (c >= n || c < r) return;
    int32_t acc = 0;
    for (int s = 0; s < ncols; s++) acc += (int32_t)G[r * ncols + s] * (int32_t)G[c * ncols + s];
    if (acc) C[r * ldc + c] -= acc;
}

// ------------------------------------------------------------------ extract one marker column
__global__ void extract_col_kernel(const int8_t* __restrict__ M, int64_t n, int64_t pitch, int64_t col,
                                   int32_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = -(int32_t)store_at(M, n, pitch, i, col);  // stores hold the negated value (decode.cu)
}

// ------------------------------------------------------------------ tsq argmax
struct Best {
    double v;
    int64_t i;
};
__device__ __forceinline__ Best better(Best a, Best b) {
    // larger value wins; ties -> lower index (which(tsq == max)[1]); i < 0 marks "nothing yet"
    if (b.i < 0) return a;
    if (a.i < 0) return b;
    if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
    return a;
}
__device__ __forceinline__ Best warp_best(Best x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Best y;
        y.v = __shfl_xor_sync(0xffffffffu, x.v, o);
        y.i = __shfl_xor_sync(0xffffffffu, x.i, o);
        x = better(x, y);
    }
    return x;
}
__global__ void __launch_bounds__(256) argmax_tsq_kernel(const double* __restrict__ a, const double* __restrict__ vara,
                                                         int64_t L, Best* __restrict__ partial) {
    Best b;
    b.v = 0.0;
    b.i = -1;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < L; j += (int64_t)gridDim.x * blockDim.x) {
        const double av = a[j];
        const double t = (av * av) / vara[j];  // a**2/vara, IEEE division as in R
        if (t == t) {                          // max(tsq, na.rm=TRUE): NaN ignored, +-Inf kept
            Best c;
            c.v = t;
            c.i = j;
            b = better(b, c);
        }
    }
    __shared__ Best sh[8];
    b = warp_best(b);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = b;
    __syncthreads();
    if (threadIdx.x < 32) {
        Best c;
        c.v = 0.0;
        c.i = -1;
        if (threadIdx.x < 8) c = sh[threadIdx.x];
        c = warp_best(c);
        if (threadIdx.x == 0) partial[blockIdx.x] = c;
    }
}
__global__ void argmax_final_kernel(const Best* __restrict__ partial, int nparts, double* best, int64_t* best_idx) {
    Best b;
    b.v = 0.0;
    b.i = -1;
    for (int k = threadIdx.x; k < nparts; k += 32) b = better(b, partial[k]);
    b = warp_best(b);
    if (threadIdx.x == 0) {
        *best = b.i >= 0 ? b.v : nan("");
        *best_idx = b.i;
    }
}

// ------------------------------------------------------------------ y = scale * Mt * x
// HBM-bound: reads the Mt store once.  x is staged in shared memory chunk by chunk, transposed so
// that the 32 lanes of a warp (each holding one 16-genotype vector) read consecutive doubles
// (conflict-free).  A warp owns 8 marker rows; per row the reduction order is fixed (lane-private
// sums in vector order, then a shuffle tree), so identical rows give bit-identical results.
constexpr int GV_CHUNK_VEC = 256;                  // 16-genotype vectors per x chunk (4096 doubles, 32 KB)
constexpr int GV_ROWS_PER_WARP = 8;
constexpr int GV_ROWS_PER_BLOCK = 8 * GV_ROWS_PER_WARP;
__device__ __forceinline__ double gv_s8_to_f64(uint32_t w, int b) {  // byte b of w in {-1,0,1} -> double, integer ops only
    const uint32_t g = (uint32_t)((int32_t)(w << (24 - 8 * b)) >> 24);
    const uint32_t hi = (g & 0x80000000u) | ((g & 1u) * 0x3FF00000u);
    return __hiloint2double((int)hi, 0);
}
__global__ void __launch_bounds__(256) gemv_i8_kernel(const int8_t* __restrict__ Mt, int64_t L, int64_t n,
                                                      int64_t pitch, const double* __restrict__ x, double scale,
                                                      double* __restrict__ y) {
    __shared__ double xs[16 * GV_CHUNK_VEC];  // xs[k * GV_CHUNK_VEC + v] = x[chunk0 + 16 v + k]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t nvec = (n + 15) >> 4;
    for (int64_t rb = (int64_t)blockIdx.x * GV_ROWS_PER_BLOCK; rb < L; rb += (int64_t)gridDim.x * GV_ROWS_PER_BLOCK) {
        const int64_t r0 = rb + warp * GV_ROWS_PER_WARP;
        double acc[GV_ROWS_PER_WARP];
#pragma unroll
        for (int r = 0; r < GV_ROWS_PER_WARP; r++) acc[r] = 0.0;
        for (int64_t v0 = 0; v0 < nvec; v0 += GV_CHUNK_VEC) {
            __syncthreads();
            for (int e = threadIdx.x; e < 16 * GV_CHUNK_VEC; e += 256) {
                const int64_t i = v0 * 16 + e;
                xs[(e & 15) * GV_CHUNK_VEC + (e >> 4)] = i < n ? x[i] : 0.0;  // zero beyond n: no bounds checks below
            }
            __syncthreads();
            const int nv = (int)((nvec - v0) < GV_CHUNK_VEC ? (nvec - v0) : GV_CHUNK_VEC);
#pragma unroll
            for (int r = 0; r < GV_ROWS_PER_WARP; r++) {
                if (r0 + r >= L) break;
                const uint4* row = reinterpret_cast<const uint4*>(Mt + (r0 + r) * pitch) + v0;
                double a = acc[r];
                for (int v = lane; v < nv; v += 32) {
                    const uint4 q = row[v];
                    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                    for (int k = 0; k < 16; k++) a += gv_s8_to_f64(w[k >> 2], k & 3) * xs[k * GV_CHUNK_VEC + v];
                }
                acc[r] = a;
            }
        }
#pragma unroll
        for (int r = 0; r < GV_ROWS_PER_WARP; r++) {
            double a = acc[r];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0 && r0 + r < L) y[r0 + r] = scale * a;
        }
    }
}

// K-blocked input [col/128][rows][128] -> Mt rows, 128 x 128 byte tiles.  The 64 x 64 kernel above keeps 16 bytes
// per thread in flight, moves 64-byte pieces and gathers bytes one LDS.U8 at a time (measured 2.9 TB/s at n = 10k).
// Here a tile is one contiguous 16 KB range of the input (four independent 16-byte loads per thread); it is
// transposed as 4 x 4 byte blocks in registers (LDS.32 + PRMT) into a second, XOR-swizzled tile (word w of output
// row c sits at w ^ (c >> 2): both the 4-byte scatter and the 16-byte read-out are bank-conflict free) and leaves
// as 128 full 128-byte lines; tiles run along the rows first so that neighbouring CTAs extend each other's lines.
__global__ void __launch_bounds__(256) transpose_kb128_kernel(const int8_t* __restrict__ in, int64_t rows, int64_t cols,
                                                              int8_t* __restrict__ out, int64_t out_pitch, int64_t tiles_r,
                                                              int64_t total) {
    __shared__ __align__(16) uint32_t tin[128][36];   // [input row][word of 4 columns], 16 B of padding per row
    __shared__ __align__(16) uint32_t tout[128][32];  // [output row = column][word of 4 input rows, swizzled]
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int64_t tix = blockIdx.x; tix < total; tix += gridDim.x) {
        const int64_t kb = tix / tiles_r, tr = tix - kb * tiles_r;
        const int64_t r0 = tr * 128;
        {
            const int seg = t & 7;
            uint4 v[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int r = (t >> 3) + 32 * k;
                v[k] = make_uint4(0, 0, 0, 0);  // rows beyond `rows` read as 0: the output pad stays zero
                if (r0 + r < rows) v[k] = *reinterpret_cast<const uint4*>(in + (kb * rows + r0 + r) * 128 + seg * 16);
            }
            __syncthreads();  // the previous tile has left tin / tout
#pragma unroll
            for (int k = 0; k < 4; k++) *reinterpret_cast<uint4*>(&tin[(t >> 3) + 32 * k][seg * 4]) = v[k];
        }
        __syncthreads();
        // thread (lane = 4 columns, warp = 16 input rows): 4 blocks of 4 x 4 bytes
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const int rb = warp * 16 + m * 4;
            const uint32_t a0 = tin[rb][lane], a1 = tin[rb + 1][lane], a2 = tin[rb + 2][lane], a3 = tin[rb + 3][lane];
            const uint32_t p0 = __byte_perm(a0, a1, 0x5140), p1 = __byte_perm(a0, a1, 0x7362);  // a0.0 a1.0 a0.1 a1.1 | .2 .3
            const uint32_t q0 = __byte_perm(a2, a3, 0x5140), q1 = __byte_perm(a2, a3, 0x7362);
            const uint32_t b[4] = {__byte_perm(p0, q0, 0x5410), __byte_perm(p0, q0, 0x7632), __byte_perm(p1, q1, 0x5410),
                                   __byte_perm(p1, q1, 0x7632)};  // b[j] = column j of the block, rows rb..rb+3
            const int w = warp * 4 + m;  // word (4 input rows) inside the output row
#pragma unroll
            for (int j = 0; j < 4; j++) tout[lane * 4 + j][w ^ lane] = b[j];
        }
        __syncthreads();
        {
            const int g = t & 7;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int c = (t >> 3) + 32 * k;
                const int cg = c >> 2;
                const uint4 x = *reinterpret_cast<const uint4*>(&tout[c][(g ^ (cg >> 2)) * 4]);
                uint32_t w0 = x.x, w1 = x.y, w2 = x.z, w3 = x.w, s;
                if (cg & 1) { s = w0; w0 = w1; w1 = s; s = w2; w2 = w3; w3 = s; }
                if (cg & 2) { s = w0; w0 = w2; w2 = s; s = w1; w1 = w3; w3 = s; }
                if (kb * 128 + c < cols)
                    *reinterpret_cast<uint4*>(out + (kb * 128 + c) * out_pitch + r0 + g * 16) = make_uint4(w0, w1, w2, w3);
            }
        }
    }
}

// ------------------------------------------------------------------ y = alpha * Mt * x, exact on the integer pipe
// FP64 FMAs outside the tensor cores retire a few per clock per SM on B200: the FP64 kernel above spends 5 ms on
// the 10^10 FMAs of config 3 where reading Mt takes 1.7 ms.  Same digit scheme as scan_i8.cu instead: x is written
// as 2^(e-55) * sum_s q_s 256^(6-s) with 7 balanced int8 digits (|residual| <= 2^(e-56), e from max |x|), the seven
// integer dot products  A_s(j) = sum_i m_ji q_s(i)  are exact (DP4A, int32) in any order, and they are recombined
// with ONE rounding.  Identical rows give bit-identical results wherever they sit.  An x whose largest magnitude is below
// 2^-1020 (e < -1019) gets the scale ldexp(1, e - 55) = 0, so y = 0: the vectors of the search (E_c, v) are far above it.
constexpr int GD_KW = 4096;           // words (4 genotypes each) of x digits staged per pass: 7 x 16 KB of shared memory
constexpr int GD_ROWS_PER_WARP = 8;
constexpr int GD_SMEM_BYTES = 7 * GD_KW * 4;

__global__ void __launch_bounds__(1024) gv_slice_kernel(const double* __restrict__ x, int64_t n, int64_t Kw,
                                                        uint32_t* __restrict__ xs, double* __restrict__ xscale) {
    __shared__ unsigned long long sh[32];
    __shared__ int s_e;
    unsigned long long m = 0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) {
        const unsigned long long b = (unsigned long long)__double_as_longlong(x[i]) & 0x7FFFFFFFFFFFFFFFull;
        m = b > m ? b : m;   // |x| bit patterns order like integers; NaN > Inf > finite
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
        m = t > m ? t : m;
    }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; w++) m = sh[w] > m ? sh[w] : m;
        int e = 0;
        double sc = 0.0;
        if (m >= 0x7FF0000000000000ull) sc = __longlong_as_double(0x7FF8000000000000LL);  // NaN / Inf in x poisons y
        else if (m) {
            if (frexp(__longlong_as_double((long long)m), &e) >= 0.9921875) e++;
            sc = ldexp(1.0, e - 55);
        }
        s_e = e;
        *xscale = sc;
    }
    __syncthreads();
    const int e = s_e;
    for (int64_t w = threadIdx.x; w < Kw; w += 1024) {
        uint32_t out[7] = {0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int d = 0; d < 4; d++) {
            const int64_t i = 4 * w + d;
            if (i < n) {
                const double v = ldexp(x[i], 55 - e);
                long long X = fabs(v) < 3.6e16 ? __double2ll_rn(v) : 0;
#pragma unroll
                for (int sidx = 6; sidx > 0; sidx--) {
                    const int q = (int)(int8_t)(X & 0xFF);
                    out[sidx] |= ((uint32_t)q & 0xFFu) << (8 * d);
                    X = (X - q) >> 8;
                }
                out[0] |= ((uint32_t)(int)X & 0xFFu) << (8 * d);
            }
        }
#pragma unroll
        for (int sidx = 0; sidx < 7; sidx++) xs[sidx * Kw + w] = out[sidx];
    }
}

__global__ void __launch_bounds__(256) gemv_i8_dp4a_kernel(const int8_t* __restrict__ Mt, int64_t L, int64_t pitch,
                                                           const uint32_t* __restrict__ xs, int64_t Kw,
                                                           const double* __restrict__ xscale, double alpha,
                                                           double* __restrict__ y) {
    extern __shared__ __align__(16) uint32_t sx[];  // [7][GD_KW]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t groups = (L + 8 * GD_ROWS_PER_WARP - 1) / (8 * GD_ROWS_PER_WARP);
    const double sc = *xscale;
    int64_t staged = -1;
    for (int64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
        const int64_t row0 = (grp * 8 + warp) * GD_ROWS_PER_WARP;
        int acc[GD_ROWS_PER_WARP][7];
#pragma unroll
        for (int r = 0; r < GD_ROWS_PER_WARP; r++)
#pragma unroll
            for (int q = 0; q < 7; q++) acc[r][q] = 0;
        for (int64_t k0 = 0; k0 < Kw; k0 += GD_KW) {
            const int kw = (int)(Kw - k0 < GD_KW ? Kw - k0 : GD_KW);
            if (staged != k0) {   // one pass when the whole of x fits (n <= 16384): staged once per CTA
                __syncthreads();
                for (int q = 0; q < 7; q++)
                    for (int w = threadIdx.x; w < kw; w += 256) sx[q * GD_KW + w] = xs[q * Kw + k0 + w];
                __syncthreads();
                staged = k0;
            }
            for (int w4 = lane; w4 < (kw >> 2); w4 += 32) {  // 16 genotypes per lane and row: 4 KB per warp in flight
                uint4 m[GD_ROWS_PER_WARP];
#pragma unroll
                for (int r = 0; r < GD_ROWS_PER_WARP; r++) {
                    const int64_t row = row0 + r < L ? row0 + r : L - 1;
                    m[r] = *reinterpret_cast<const uint4*>(Mt + row * pitch + 4 * k0 + 16 * (int64_t)w4);
                }
#pragma unroll
                for (int q = 0; q < 7; q++) {
                    const uint4 d = *reinterpret_cast<const uint4*>(&sx[q * GD_KW + 4 * w4]);
#pragma unroll
                    for (int r = 0; r < GD_ROWS_PER_WARP; r++) {
                        int a = acc[r][q];
                        a = __dp4a((int)m[r].x, (int)d.x, a);
                        a = __dp4a((int)m[r].y, (int)d.y, a);
                        a = __dp4a((int)m[r].z, (int)d.z, a);
                        a = __dp4a((int)m[r].w, (int)d.w, a);
                        acc[r][q] = a;
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < GD_ROWS_PER_WARP; r++) {
#pragma unroll
            for (int q = 0; q < 7; q++)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc[r][q] += __shfl_xor_sync(0xffffffffu, acc[r][q], o);  // exact: any order
            if (lane == r && row0 + r < L) {
                const long long hi = (((long long)acc[r][0] * 256 + acc[r][1]) * 256 + acc[r][2]) * 256 + acc[r][3];
                const long long lo = ((long long)acc[r][4] * 256 + acc[r][5]) * 256 + acc[r][6];
                const double v = fma((double)hi, 16777216.0, (double)lo);  // the one rounding of the recombination
                y[row0 + r] = alpha * (v * sc);                             // power-of-two scale: exact
            }
        }
    }
}

// ------------------------------------------------------------------ ReshapeM as a device row / column mask
// (reference: src/ReshapeM_rcpp.cpp:59-109 rewrites M.ascii without the rows of individuals whose trait is NA and
// Mt.ascii without the matching columns).  map[new] = old index of the individuals that stay.
// rows: one thread = one 16-byte vector of an output row; both layouts (pitch == 0: K-blocked [c/128][rows][128])
__global__ void __launch_bounds__(256) gather_rows_kernel(const int8_t* __restrict__ in, int64_t in_rows, int64_t in_pitch,
                                                          const int64_t* __restrict__ map, int64_t out_rows, int64_t out_pitch,
                                                          int64_t vec_per_row, int8_t* __restrict__ out) {
    const int64_t total = out_rows * vec_per_row;
    for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (int64_t)gridDim.x * 256) {
        int64_t r, v;
        if (in_pitch) { r = t / vec_per_row; v = t - r * vec_per_row; }
        else { r = (t >> 3) % out_rows; v = ((t >> 3) / out_rows) * 8 + (t & 7); }  // 8 vectors = one 128-byte line
        const int64_t c = 16 * v, ro = map[r];
        const int64_t src = in_pitch ? ro * in_pitch + c : ((c >> 7) * in_rows + ro) * 128 + (c & 127);
        const int64_t dst = out_pitch ? r * out_pitch + c : ((c >> 7) * out_rows + r) * 128 + (c & 127);
        *reinterpret_cast<uint4*>(out + dst) = *reinterpret_cast<const uint4*>(in + src);
    }
}
// columns of a row-major store (Mt: columns = individuals): one thread = 4 output bytes; the output pad is zero
__global__ void __launch_bounds__(256) gather_cols_kernel(const int8_t* __restrict__ in, int64_t rows, int64_t in_pitch,
                                                          const int64_t* __restrict__ map, int64_t out_cols, int64_t out_pitch,
                                                          int8_t* __restrict__ out) {
    const int64_t wpr = out_pitch / 4, total = rows * wpr;
    for (int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (int64_t)gridDim.x * 256) {
        const int64_t r = t / wpr, w = t - r * wpr;
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int64_t c = 4 * w + b;
            if (c < out_cols) v |= (uint32_t)(uint8_t)in[r * in_pitch + map[c]] << (8 * b);
        }
        *reinterpret_cast<uint32_t*>(out + r * out_pitch + 4 * w) = v;
    }
}

}  // namespace eg

using namespace eg;

static int transpose_launch(const int8_t* d_in, int64_t rows, int64_t cols, int64_t in_pitch, int in_kb, int8_t* d_out,
                            int64_t out_pitch, void* stream) {
    if (!d_in || !d_out || rows < 0 || cols < 0 || (in_pitch & 15) || (out_pitch & 63) || in_pitch < cols ||
        out_pitch < rows)
        return set_error(EG_ERR_ARG, "eg_dev_transpose_i8: bad argument");
    if (rows == 0 || cols == 0) return EG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (in_kb && (out_pitch & 127) == 0 && !(getenv("EAGLE_TRANSPOSE_128") && getenv("EAGLE_TRANSPOSE_128")[0] == '0')) {
        const int64_t tiles_r = out_pitch / 128, total = tiles_r * ((cols + 127) / 128);
        const int64_t cap = (int64_t)num_sms() * 8;
        transpose_kb128_kernel<<<(unsigned)(total < cap ? total : cap), 256, 0, st>>>(d_in, rows, cols, d_out, out_pitch, tiles_r,
                                                                                  total);
        return check_launch("transpose_kb128_kernel");
    }
    // tiles run over the whole output pitch: input rows >= `rows` are read as 0, which zero-fills the pad
    const int64_t tiles_r = (out_pitch + TR_TILE - 1) / TR_TILE, tiles_c = (cols + TR_TILE - 1) / TR_TILE;
    const int64_t total = tiles_r * tiles_c;
    const int64_t cap = (int64_t)num_sms() * 16;
    transpose_i8_kernel<<<(unsigned)(total < cap ? total : cap), 256, 0, st>>>(d_in, rows, cols, in_pitch, in_kb, d_out,
                                                                              out_pitch, tiles_c);
    return check_launch("transpose_i8_kernel");
}
extern "C" int eg_dev_transpose_i8(const int8_t* d_in, int64_t rows, int64_t cols, int64_t in_pitch, int8_t* d_out,
                                   int64_t out_pitch, void* stream) {
    return transpose_launch(d_in, rows, cols, in_pitch, 0, d_out, out_pitch, stream);
}
// input in the K-blocked layout [ceil(cols/128)][rows][128]
extern "C" int eg_dev_transpose_kb_i8(const int8_t* d_in_kb, int64_t rows, int64_t cols, int8_t* d_out,
                                      int64_t out_pitch, void* stream) {
    return transpose_launch(d_in_kb, rows, cols, round_up(cols, 128), 1, d_out, out_pitch, stream);
}

extern "C" int eg_dev_mmt_finalize(const int32_t* d_C, int64_t n, int64_t ldc, double* d_out, void* stream) {
    if (!d_C || !d_out || n <= 0 || ldc < n) return set_error(EG_ERR_ARG, "eg_dev_mmt_finalize: bad argument");
    const unsigned nb = (unsigned)((n + 31) / 32);
    mmt_finalize_kernel<<<dim3(nb, nb), 256, 0, (cudaStream_t)stream>>>(d_C, n, ldc, d_out);
    return check_launch("mmt_finalize_kernel");
}

extern "C" int eg_dev_syrk_zero_cols(const int8_t* d_M, int64_t n, int64_t pitch, const int64_t* h_zero_cols,
                                     int64_t n_zero, int32_t* d_C, int64_t ldc, void* stream) {
    if (n_zero <= 0) return EG_OK;
    if (!d_M || !d_C || !h_zero_cols) return set_error(EG_ERR_ARG, "eg_dev_syrk_zero_cols: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    // a locus listed twice must only be removed once (setZero is idempotent in the reference)
    std::vector<int64_t> uniq;
    for (int64_t i = 0; i < n_zero; i++) {
        bool seen = false;
        for (int64_t u : uniq) seen |= (u == h_zero_cols[i]);
        if (!seen) uniq.push_back(h_zero_cols[i]);
    }
    const int k = (int)uniq.size();
    int64_t* d_cols = nullptr;
    int8_t* d_G = nullptr;
    EG_CUDA(cudaMalloc(&d_cols, k * sizeof(int64_t)));
    if (malloc_retry((void**)&d_G, (size_t)n * k) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d_cols);
        return set_error(EG_ERR_ALLOC, "eg_dev_syrk_zero_cols: out of device memory");
    }
    int rc = check_cuda(cudaMemcpyAsync(d_cols, uniq.data(), k * sizeof(int64_t), cudaMemcpyHostToDevice, st), "memcpy");
    if (rc == EG_OK) {
        gather_cols_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_M, n, pitch, d_cols, k, d_G);
        syrk_zero_cols_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)n), 256, 0, st>>>(d_G, n, k, d_C, ldc);
        rc = check_launch("syrk_zero_cols_kernel");
    }
    cudaStreamSynchronize(st);
    cudaFree(d_cols);
    cudaFree(d_G);
    return rc;
}

extern "C" int eg_dev_extract_col(const int8_t* d_M, int64_t n, int64_t pitch, int64_t col, int32_t* d_out,
                                  void* stream) {
    if (!d_M || !d_out || n <= 0 || col < 0 || (pitch && col >= pitch))  // pitch == 0: K-blocked store
        return set_error(EG_ERR_ARG, "eg_dev_extract_col: bad argument");
    extract_col_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_M, n, pitch, col, d_out);
    return check_launch("extract_col_kernel");
}

extern "C" int eg_dev_argmax_tsq(const double* d_a, const double* d_vara, int64_t L, double* d_best,
                                 int64_t* d_best_idx, void* stream) {
    if (!d_a || !d_vara || !d_best || !d_best_idx || L <= 0)
        return set_error(EG_ERR_ARG, "eg_dev_argmax_tsq: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local Best* d_partial = nullptr;
    static thread_local int d_partial_dev = -1;
    int dev = 0;
    EG_CUDA(cudaGetDevice(&dev));
    const int maxblocks = 1024;
    if (!d_partial || d_partial_dev != dev) {
        EG_CUDA(cudaMalloc(&d_partial, maxblocks * sizeof(Best)));
        d_partial_dev = dev;
    }
    int64_t nb = (L + 255) / 256;
    if (nb > maxblocks) nb = maxblocks;
    argmax_tsq_kernel<<<(unsigned)nb, 256, 0, st>>>(d_a, d_vara, L, d_partial);
    argmax_final_kernel<<<1, 32, 0, st>>>(d_partial, (int)nb, d_best, d_best_idx);
    return check_launch("argmax_tsq_kernel");
}

extern "C" int eg_dev_gemv_i8(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_x,
                              double scale, double* d_y, void* stream) {
    if (!d_Mt || !d_x || !d_y || L <= 0 || n <= 0 || (pitch & 15) || pitch < n)
        return set_error(EG_ERR_ARG, "eg_dev_gemv_i8: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    scale = -scale;  // the store holds the negated genotype values (decode.cu): y = scale * (M_true x)
    const char* env = getenv("EAGLE_GEMV_MODE");
    if (!(env && env[0] == 'f')) {
        // exact integer evaluation (DP4A); workspace: 7 digit planes of x + its scale
        static thread_local uint32_t* d_xs = nullptr;
        static thread_local size_t xs_cap = 0;
        static thread_local int xs_dev = -1;
        int dev = 0;
        EG_CUDA(cudaGetDevice(&dev));
        const int64_t Kw = round_up(n, 16) / 4;
        const size_t need = (size_t)7 * Kw + 2;
        if (xs_dev != dev || need > xs_cap) {
            if (d_xs && xs_dev == dev) cudaFree(d_xs);
            d_xs = nullptr;
            EG_CUDA(cudaMalloc(&d_xs, need * sizeof(uint32_t)));
            xs_cap = need;
            xs_dev = dev;
        }
        double* d_scale = reinterpret_cast<double*>(d_xs + (((size_t)7 * Kw + 1) & ~(size_t)1));
        gv_slice_kernel<<<1, 1024, 0, st>>>(d_x, n, Kw, d_xs, d_scale);
        EG_TRY(check_launch("gv_slice_kernel"));
        EG_CUDA(cudaFuncSetAttribute(gemv_i8_dp4a_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GD_SMEM_BYTES));
        const int64_t groups = (L + 8 * GD_ROWS_PER_WARP - 1) / (8 * GD_ROWS_PER_WARP);
        const int64_t capb = (int64_t)num_sms() * 2;
        gemv_i8_dp4a_kernel<<<(unsigned)(groups < capb ? groups : capb), 256, GD_SMEM_BYTES, st>>>(d_Mt, L, pitch, d_xs, Kw,
                                                                                               d_scale, scale, d_y);
        return check_launch("gemv_i8_dp4a_kernel");
    }
    int64_t nb = (L + GV_ROWS_PER_BLOCK - 1) / GV_ROWS_PER_BLOCK;
    const int64_t cap = (int64_t)num_sms() * 6;
    if (nb > cap) nb = cap;
    gemv_i8_kernel<<<(unsigned)nb, 256, 0, st>>>(d_Mt, L, n, pitch, d_x, scale, d_y);
    return check_launch("gemv_i8_kernel");
}

// in/out: stores of the given geometry (pitch 0 = K-blocked); d_map: kept individuals, new index -> old index
extern "C" int eg_dev_gather_rows(const int8_t* d_in, int64_t in_rows, int64_t cols, int64_t in_pitch, const int64_t* d_map,
                                  int64_t out_rows, int8_t* d_out, int64_t out_pitch, void* stream) {
    if (!d_in || !d_out || !d_map || out_rows <= 0 || cols <= 0 || (in_pitch == 0) != (out_pitch == 0) || (in_pitch & 15) ||
        (out_pitch & 15) || (in_pitch && out_pitch > in_pitch))
        return set_error(EG_ERR_ARG, "eg_dev_gather_rows: bad argument");
    const int64_t vec = in_pitch ? out_pitch / 16 : round_up(cols, 128) / 16, total = out_rows * vec;
    const int64_t cap = (int64_t)num_sms() * 32, nb = (total + 255) / 256;
    gather_rows_kernel<<<(unsigned)(nb < cap ? nb : cap), 256, 0, (cudaStream_t)stream>>>(d_in, in_rows, in_pitch, d_map, out_rows,
                                                                                       out_pitch, vec, d_out);
    return check_launch("gather_rows_kernel");
}
extern "C" int eg_dev_gather_cols(const int8_t* d_in, int64_t rows, int64_t in_pitch, const int64_t* d_map, int64_t out_cols,
                                  int8_t* d_out, int64_t out_pitch, void* stream) {
    if (!d_in || !d_out || !d_map || rows <= 0 || out_cols <= 0 || (out_pitch & 3) || out_pitch < out_cols || in_pitch <= 0)
        return set_error(EG_ERR_ARG, "eg_dev_gather_cols: bad argument");
    const int64_t total = rows * (out_pitch / 4);
    const int64_t cap = (int64_t)num_sms() * 32, nb = (total + 255) / 256;
    gather_cols_kernel<<<(unsigned)(nb < cap ? nb : cap), 256, 0, (cudaStream_t)stream>>>(d_in, rows, in_pitch, d_map, out_cols,
                                                                                       out_pitch, d_out);
    return check_launch("gather_cols_kernel");
}

