// K3 -- per-marker BLUP and variance scan on the FP64 tensor cores.
//
// Replaces, for all markers j (rows of Mt), reference src/calculate_a_and_vara_rcpp.cpp:
//     a_j    = Mt_j . v              v = inv_MMt_sqrt * a_hat                     (:90-91)
//     T      = Mt * W                W = inv_MMt_sqrt * (dim_reduced_vara * inv_MMt_sqrt) (:97-98, :103)
//     vara_j = T_j . Mt_j                                                          (:107-112)
// without ever materialising T (L x n doubles in the reference).
//
// Symmetric half.  vara_j = m_j^T W m_j is a quadratic form: it only sees the symmetric part of W,
// for ANY W.  eg_dev_scan_prepare therefore folds W into U = diag(W) + strict_upper(W + W^T) (lower
// triangle zero), so that  vara_j = sum_k ( sum_{i<=k} m_ij U_ik ) m_kj  and the contraction for
// column k stops at row k: half the FP64 work of the reference's full T = Mt*W, identical in real
// arithmetic, ~1 ulp of W apart in floating point (tolerance 1e-9).  a_j = Mt_j . v is a separate
// bandwidth-bound pass (gemv_i8_kernel, layout.cu) over the same store.
//
// Wp layout (built by eg_dev_scan_prepare): Npad columns x Kpad rows, column-major, ld = Kpad,
// Kpad = round_up(n,32), Npad = round_up(n+1,128); columns 0..n-1 hold U, column n holds v, rest zero.
// Mt: int8 store, L x n, row-major, pitch >= Npad, zero padded (so pad columns add exact zeros).
//
// One CTA owns a block of 64 markers and sweeps all column panels of Wp (128 wide) in the
// same order on every CTA, so the panels are shared through L2.  Inside: 8 warps (2 x 4), warp
// tile 32 x 32, two CTAs per SM, DMMA.8x8x4 (mma.sync.m8n8k4.f64), int8 -> f64 conversion with integer ops
// only, done one stage ahead into a swizzled FP64 shared-memory tile, 4-stage cp.async ring.  The row-dot is fused into the panel epilogue with
// a fixed reduction order (registers -> 4-lane shuffle -> 4 warps through shared memory ->
// panel order), so a marker's a/vara depend only on its genotypes, never on its position,
// tile or GPU: identical marker rows give bit-identical results (tie rule of find_qtl.R:76-80).
#include "common.cuh"
#include "ptx.cuh"

namespace eg {

constexpr int SC_BM = 64;                  // markers per CTA tile
constexpr int SC_BN = 128;                 // columns of Wp per panel
constexpr int SC_BK = 16;                  // k-tile: one 128-byte segment of doubles per row / column
constexpr int SC_THREADS = 256;            // 8 warps = 2 (markers) x 4 (columns), warp tile 32 x 32
constexpr int SC_CTAS_PER_SM = 2;          // independent barrier domains keep the DMMA pipe fed
constexpr int SC_BSTAGES = 4;              // ring of W tiles and raw Mt tiles (cp.async)
constexpr int SC_B_BYTES = SC_BN * 128;    // 16 KB per W k-tile
constexpr int SC_A64_BYTES = SC_BM * 128;  // 8 KB per converted Mt k-tile
constexpr int SC_RAW_BYTES = SC_BM * SC_BK;  // 1 KB per raw int8 Mt k-tile
constexpr int SC_OFF_A64 = SC_BSTAGES * SC_B_BYTES;
constexpr int SC_OFF_RAW = SC_OFF_A64 + 2 * SC_A64_BYTES;
constexpr int SC_OFF_RED = SC_OFF_RAW + SC_BSTAGES * SC_RAW_BYTES;
constexpr int SC_SMEM_BYTES = SC_OFF_RED + 4 * SC_BM * 8;

struct ScanParams {
    const int8_t* Mt;
    int64_t L, n, pitch;
    const double* Wp;
    int64_t Kpad;
    int32_t NP;        // column panels
    int32_t KT;        // k tiles covering all n rows
    int32_t total_steps;  // sum over panels of the k tiles each needs
    const int64_t* zero_rows;
    int32_t n_zero;
    double* out_vara;
    int64_t num_blocks;
};

// genotype byte b (0..3) of w in {-1,0,1} as an IEEE double: integer pipe only
template <int B>
__device__ __forceinline__ double s8_byte_to_f64(uint32_t w) {
    constexpr uint32_t sel = (uint32_t)B | ((8u | B) << 4) | ((8u | B) << 8) | ((8u | B) << 12);
    const uint32_t g = __byte_perm(w, 0u, sel);  // sign-extended byte
    const uint32_t hi = (g & 0x80000000u) | ((g & 1u) * 0x3FF00000u);
    return __hiloint2double((int)hi, 0);
}
__device__ __forceinline__ double s8_to_f64(int g) {  // g in {-1,0,1}
    const uint32_t hi = ((uint32_t)g & 0x80000000u) | (((uint32_t)g & 1u) * 0x3FF00000u);
    return __hiloint2double((int)hi, 0);
}

// Shared-memory tiles.  Both operands are staged as doubles, one 128-byte segment (16 k values) per
// row / column, 16-byte chunks XOR-swizzled with (row & 7) (the SWIZZLE_128B pattern):
//   W tile   : cp.async from the column-major Wp, chunk c of column j at  j*128 + ((c ^ (j&7)) * 16)
//   Mt tile  : raw int8 via cp.async, converted ONE STAGE AHEAD by all threads into the same layout,
// so the DMMA stream contains only LDS.128 and DMMA.  (Microbenchmarks, scripts/microbench: DMMA.8x8x4
// peaks at 37.1 TFLOP/s with >= 8 warps/SM; independent ALU work beside it is free.)
// K permutation: lane lc (= lane & 3) supplies k = 4*lc + 2*p + e for MMA steps (p,e) in {0,1}^2 --
// the same bijection for A and B, so the product is unchanged; each lane's operands become two
// 16-byte chunks (2*lc, 2*lc+1), and chunk ^ (row&7) spreads a quarter-warp over all 8 bank groups.
// Two CTAs share an SM: while one sits at its per-k-tile barrier the other keeps issuing DMMAs.
__global__ void __launch_bounds__(SC_THREADS, SC_CTAS_PER_SM) scan_f64_kernel(const ScanParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    double* red = reinterpret_cast<double*>(smem + SC_OFF_RED);  // [4][SC_BM]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp & 1, wn = warp >> 1;
    const int lr = lane >> 2, lc = lane & 3;
    // panel q only needs k-tiles up to its last column: rows i > k of U are zero
    auto ktiles_of = [&](int q) { const int kt = (q + 1) * (SC_BN / SC_BK); return kt < p.KT ? kt : p.KT; };
    const int total_steps = p.total_steps;

    // fragment offsets (bytes): row/col = base + 8*tile + lr  ->  (row & 7) == lr
    const int fa0 = (wm * 32 + lr) * 128 + (((2 * lc) ^ lr) * 16);      // A, p = 0 ; + mt*1024
    const int fa1 = (wm * 32 + lr) * 128 + (((2 * lc + 1) ^ lr) * 16);  // A, p = 1
    const int fb0 = (wn * 32 + lr) * 128 + (((2 * lc) ^ lr) * 16);      // B, p = 0 ; + t*1024
    const int fb1 = (wn * 32 + lr) * 128 + (((2 * lc + 1) ^ lr) * 16);  // B, p = 1

    // loader roles
    const int ld_c = tid >> 1, ld_h = tid & 1;       // W: column, 64-byte half (chunks 4*ld_h .. +3)
    const int cv_r = tid >> 2, cv_q = tid & 3;       // convert: row, 4 genotypes (chunks 2*cv_q, 2*cv_q+1)

    for (int64_t mb = blockIdx.x; mb < p.num_blocks; mb += gridDim.x) {
        const int64_t j0 = mb * SC_BM;
        int64_t jrow = j0 + tid;                      // raw Mt loader row (threads 0..63)
        if (jrow >= p.L) jrow = p.L - 1;              // tail block: duplicate a valid row, result discarded
        const int8_t* mt_row = p.Mt + jrow * p.pitch;

        int ld_pnl = 0, ld_kt = 0, ld_slot = 0;       // position of the next k-tile to load
        auto load_next = [&]() {
            const uint8_t* src = reinterpret_cast<const uint8_t*>(
                p.Wp + ((int64_t)ld_pnl * SC_BN + ld_c) * p.Kpad + (int64_t)ld_kt * SC_BK) + ld_h * 64;
            uint8_t* dst = smem + ld_slot * SC_B_BYTES + ld_c * 128;
#pragma unroll
            for (int i = 0; i < 4; i++) ptx::cp_async_16(dst + (((ld_h * 4 + i) ^ (ld_c & 7)) * 16), src + i * 16);
            if (tid < SC_BM)
                ptx::cp_async_16(smem + SC_OFF_RAW + ld_slot * SC_RAW_BYTES + tid * SC_BK, mt_row + (int64_t)ld_kt * SC_BK);
            if (++ld_kt == ktiles_of(ld_pnl)) { ld_kt = 0; ld_pnl++; }
            if (++ld_slot == SC_BSTAGES) ld_slot = 0;
        };
        // int8 -> f64 of k-tile in raw slot `slot` into A64[buf]
        auto convert = [&](int slot, int buf) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(smem + SC_OFF_RAW + slot * SC_RAW_BYTES + cv_r * SC_BK + cv_q * 4);
            uint8_t* dst = smem + SC_OFF_A64 + buf * SC_A64_BYTES + cv_r * 128;
            *reinterpret_cast<double2*>(dst + (((2 * cv_q) ^ (cv_r & 7)) * 16)) = make_double2(s8_byte_to_f64<0>(w), s8_byte_to_f64<1>(w));
            *reinterpret_cast<double2*>(dst + (((2 * cv_q + 1) ^ (cv_r & 7)) * 16)) = make_double2(s8_byte_to_f64<2>(w), s8_byte_to_f64<3>(w));
        };

        double acc[4][4][2];
#pragma unroll
        for (int mt = 0; mt < 4; mt++)
#pragma unroll
            for (int t = 0; t < 4; t++) acc[mt][t][0] = acc[mt][t][1] = 0.0;
        double vara_run = 0.0;  // threads 0..63: running vara of marker row tid

        __syncthreads();  // previous marker block fully done with shared memory
        for (int s = 0; s < SC_BSTAGES - 1; s++) {  // groups 0,1,2
            if (s < total_steps) load_next();
            ptx::cp_async_commit();
        }
        ptx::cp_async_wait<SC_BSTAGES - 2>();  // group 0 landed
        __syncthreads();
        convert(0, 0);

        int slot = 0, kt = 0, pnl = 0;
        for (int s = 0; s < total_steps; s++) {
            ptx::cp_async_wait<SC_BSTAGES - 3>();  // groups <= s+1 landed (W(s), raw Mt(s+1))
            __syncthreads();                       // ... for everybody; A64(s) written; tile s-1 fully consumed

            const uint8_t* sB = smem + slot * SC_B_BYTES;
            const uint8_t* sA = smem + SC_OFF_A64 + (s & 1) * SC_A64_BYTES;
            double2 a[4], b[4];
            // ---- MMA step p = 0 first: the pipe refills right after the barrier
#pragma unroll
            for (int mt = 0; mt < 4; mt++) a[mt] = *reinterpret_cast<const double2*>(sA + fa0 + mt * 1024);
#pragma unroll
            for (int t = 0; t < 4; t++) b[t] = *reinterpret_cast<const double2*>(sB + fb0 + t * 1024);
#pragma unroll
            for (int mt = 0; mt < 4; mt++)
#pragma unroll
                for (int t = 0; t < 4; t++) ptx::dmma_884(acc[mt][t][0], acc[mt][t][1], a[mt].x, b[t].x);
            // ---- asynchronous work for later tiles, issued in the shadow of the DMMAs above
            if (s + SC_BSTAGES - 1 < total_steps) load_next();
            ptx::cp_async_commit();
            if (s + 1 < total_steps) convert(slot + 1 == SC_BSTAGES ? 0 : slot + 1, (s + 1) & 1);
#pragma unroll
            for (int mt = 0; mt < 4; mt++)
#pragma unroll
                for (int t = 0; t < 4; t++) ptx::dmma_884(acc[mt][t][0], acc[mt][t][1], a[mt].y, b[t].y);
            // ---- MMA step p = 1
#pragma unroll
            for (int mt = 0; mt < 4; mt++) a[mt] = *reinterpret_cast<const double2*>(sA + fa1 + mt * 1024);
#pragma unroll
            for (int t = 0; t < 4; t++) b[t] = *reinterpret_cast<const double2*>(sB + fb1 + t * 1024);
#pragma unroll
            for (int mt = 0; mt < 4; mt++)
#pragma unroll
                for (int t = 0; t < 4; t++) ptx::dmma_884(acc[mt][t][0], acc[mt][t][1], a[mt].x, b[t].x);
#pragma unroll
            for (int mt = 0; mt < 4; mt++)
#pragma unroll
                for (int t = 0; t < 4; t++) ptx::dmma_884(acc[mt][t][0], acc[mt][t][1], a[mt].y, b[t].y);

            if (++slot == SC_BSTAGES) slot = 0;
            if (++kt == ktiles_of(pnl)) {
                kt = 0;
                // ---------------- panel epilogue: fused row-dot with the marker's own genotypes
                const int64_t cbase = (int64_t)pnl * SC_BN + wn * 32 + lc * 2;
#pragma unroll
                for (int mt = 0; mt < 4; mt++) {
                    const int row = wm * 32 + mt * 8 + lr;
                    int64_t j = j0 + row;
                    if (j >= p.L) j = p.L - 1;
                    const int8_t* mrow = p.Mt + j * p.pitch + cbase;
                    double sum = 0.0;
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                        const short two = *reinterpret_cast<const short*>(mrow + t * 8);
                        const int m0 = (int)(int8_t)(two & 0xFF), m1 = (int)(int8_t)((two >> 8) & 0xFF);
                        sum += acc[mt][t][0] * s8_to_f64(m0);
                        sum += acc[mt][t][1] * s8_to_f64(m1);
                    }
                    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                    if (lc == 0) red[wn * SC_BM + row] = sum;
#pragma unroll
                    for (int t = 0; t < 4; t++) acc[mt][t][0] = acc[mt][t][1] = 0.0;
                }
                __syncthreads();
                if (tid < SC_BM)
                    vara_run += (red[tid] + red[SC_BM + tid]) + (red[2 * SC_BM + tid] + red[3 * SC_BM + tid]);
                // red[] is rewritten only after the next panel's k loop (at least one barrier later)
                pnl++;
            }
        }
        ptx::cp_async_wait<0>();
        __syncthreads();
        if (tid < SC_BM && j0 + tid < p.L) {
            const int64_t j = j0 + tid;
            bool zero = false;
            for (int z = 0; z < p.n_zero; z++) zero |= (p.zero_rows[z] == j);
            p.out_vara[j] = zero ? 0.0 : vara_run;
        }
    }
}

}  // namespace eg

extern "C" int64_t eg_scan_wp_elems(int64_t n) {
    return eg::round_up(n + 1, eg::SC_BN) * eg::round_up(n, 32);
}

namespace eg {
int launch_scan_i8(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp, int64_t Kpad,
                   const int64_t* d_zero_rows, int n_zero, double* d_vara, cudaStream_t st, bool sliced);
void scan_kernel_mark(int which, cudaStream_t st, double ops);
int scan_mode();  // 0 = FP64 DMMA (scan_f64_kernel), 1 = exact int8 slices (scan_i8_kernel)

__global__ void zero_entries_kernel(double* v, const int64_t* idx, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[idx[i]] = 0.0;
}

// sliced: a later piece of a streamed scan with the same d_Wp (the int8 path keeps the slices of U from the first piece)
int launch_scan(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp,
                const int64_t* d_zero_rows, int n_zero, double* d_a, double* d_vara, cudaStream_t st, bool sliced) {
    ScanParams p;
    p.Mt = d_Mt; p.L = L; p.n = n; p.pitch = pitch; p.Wp = d_Wp;
    p.Kpad = round_up(n, 32);
    p.NP = (int32_t)(round_up(n, SC_BN) / SC_BN);
    p.KT = (int32_t)(p.Kpad / SC_BK);
    p.total_steps = 0;
    for (int q = 0; q < p.NP; q++) {
        const int kt = (q + 1) * (SC_BN / SC_BK);
        p.total_steps += kt < p.KT ? kt : p.KT;
    }
    p.zero_rows = d_zero_rows; p.n_zero = n_zero;
    p.out_vara = d_vara;
    p.num_blocks = (L + SC_BM - 1) / SC_BM;
    // a = Mt * v (v = column n of Wp): bandwidth-bound pass, fixed per-row reduction order
    EG_TRY(eg_dev_gemv_i8(d_Mt, L, n, pitch, d_Wp + n * p.Kpad, 1.0, d_a, st));
    if (n_zero > 0) {
        zero_entries_kernel<<<(n_zero + 127) / 128, 128, 0, st>>>(d_a, d_zero_rows, n_zero);
        EG_TRY(check_launch("zero_entries_kernel"));
    }
    if (scan_mode() == 1) return launch_scan_i8(d_Mt, L, n, pitch, d_Wp, p.Kpad, d_zero_rows, n_zero, d_vara, st, sliced);
    EG_CUDA(cudaFuncSetAttribute(scan_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SC_SMEM_BYTES));
    const int64_t cap = (int64_t)num_sms() * SC_CTAS_PER_SM;
    const int64_t grid = p.num_blocks < cap ? p.num_blocks : cap;
    scan_kernel_mark(0, st, 2.0 * SC_BM * SC_BN * SC_BK * (double)p.total_steps * (double)p.num_blocks);  // executed flops
    scan_f64_kernel<<<(unsigned)grid, SC_THREADS, SC_SMEM_BYTES, st>>>(p);
    scan_kernel_mark(1, st, 0.0);
    return check_launch("scan_f64_kernel");
}
}  // namespace eg

extern "C" int eg_dev_scan(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp,
                           const int64_t* h_zero_rows, int64_t n_zero, double* d_a, double* d_vara, void* stream) {
    using namespace eg;
    if (!d_Mt || !d_Wp || !d_a || !d_vara || L <= 0 || n <= 0 || (pitch & 15) || pitch < round_up(n + 1, SC_BN) ||
        ((uintptr_t)d_Mt & 15) || n_zero < 0 || (n_zero > 0 && !h_zero_rows))
        return set_error(EG_ERR_ARG, "eg_dev_scan: bad argument (Mt pitch must be >= round_up(n+1,128))");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t* d_zero = nullptr;
    if (n_zero > 0) {
        EG_CUDA(cudaMalloc(&d_zero, n_zero * sizeof(int64_t)));
        int rc = check_cuda(cudaMemcpyAsync(d_zero, h_zero_rows, n_zero * sizeof(int64_t), cudaMemcpyHostToDevice, st),
                            "zero rows H2D");
        if (rc) { cudaFree(d_zero); return rc; }
    }
    int rc = launch_scan(d_Mt, L, n, pitch, d_Wp, d_zero, (int)n_zero, d_a, d_vara, st, false);
    if (d_zero) {
        cudaStreamSynchronize(st);
        cudaFree(d_zero);
    }
    return rc;
}
