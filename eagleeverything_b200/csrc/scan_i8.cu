// K3' -- the variance scan evaluated EXACTLY on the int8 tensor cores (tcgen05.mma.kind::i8).
//
// Same quantity as scan_f64.cu (reference src/calculate_a_and_vara_rcpp.cpp:97-112):
//     vara_j = sum_k ( sum_{i<=k} m_ij U_ik ) m_kj ,   U = diag(W) + strict_upper(W + W^T)
// The genotypes m are already int8 in {-1,0,1}.  Each column k of the FP64 matrix U is written as
//     U_ik = 2^(e_k-55) * X_ik + r ,   X_ik = rint(U_ik 2^(55-e_k)) ,  |X| <= 127 * 2^48 ,  |r| <= 2^(e_k-56)
// (below one ulp of the column's largest entry: the full FP64 significand of U is kept), and the
// integer X in BALANCED base-256 digits,   X = sum_{s=0..6} q_s 256^(6-s) ,  q_s in [-128,127] (int8):
// seven full bytes carry the 56 bits that eight 7-bit slices used to.  Then
//     P_s(j,k) = sum_i m_ij q_s(i,k)          is an EXACT int32 (|P| <= 128 n), one int8 GEMM per slice,
//     T'_jk   = 2^(e_k-55) * sum_s P_s 256^(6-s)   is recombined exactly except for ONE rounding,
// which is tighter than the n roundings of an FP64 GEMM accumulation.  7 int8 GEMMs at >3 PFLOP/s
// replace one FP64 GEMM at ~30 TFLOP/s.
//
// Layouts.  A operand: the Mt store (L x n int8, K-major).  B operand: Q, (n/32 groups) x 224 rows x Kp
// bytes, K-major; row (kk>>2)*28 + s*4 + (kk&3) of group g holds slice s of column k = 32 g + kk, so
// that one TMEM load of 28 consecutive columns brings all 7 slices of 4 columns to a thread.  Rows
// i > k and the pad are zero, so the contraction for group g stops at k-block ceil((32g+32)/128).
//
// Kernel: same warp-specialised tcgen05 pipeline as syrk_i8.cu (TMA producer, one-thread UMMA issuer
// M128 N224 K32, double-buffered TMEM, 4 epilogue warps).  Work unit = (128-marker block, group); an
// epilogue thread owns one marker row (one TMEM lane): it recombines the slices, multiplies by the
// marker's own genotype bytes and writes ONE double per (marker, group); a second tiny kernel sums
// the groups in index order.  Fixed order everywhere: identical marker rows give bit-identical
// results whatever their position, tile or GPU.  Units are ordered in (37 marker blocks x 4 groups)
// super-tiles and kept in K lock-step by the same phase counters as the SYRK, so a wave shares its
// operand rows through L2.
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "ptx.cuh"

namespace eg {

constexpr int SI_BM = 128;
constexpr int SI_GCOLS = 32;                  // columns of U per group
constexpr int SI_ACC_COLS = 256;              // TMEM columns between the two accumulators
constexpr int SI_BK = 128;
constexpr int SI_STAGES = 5;
constexpr int SI_A_BYTES = SI_BM * SI_BK;
constexpr int SI_THREADS = 320;        // TMA warp, UMMA warp, 8 epilogue warps (two per TMEM lane quarter)
constexpr int SI_TMEM_COLS = 512;
constexpr int SI_MSUP_DEFAULT = 37;  // super-tile: marker blocks (their Mt rows stay L2-resident over the group sweep)
constexpr int SI_GSUP_DEFAULT = 4;   //             x groups  (~ one wave of 148 CTAs)
constexpr int SI_PHASE = 16;
constexpr int SI_LAG = 4;
constexpr int SP_STAGES = 7;
constexpr int SP_MSUP_DEFAULT = 18;  // super-tile in units of 256-marker blocks x groups (see SI_MSUP_DEFAULT)
constexpr int SP_GSUP_DEFAULT = 4;
constexpr int SP_A_BYTES = SI_BM * SI_BK;               // 128 marker rows
// Everything that depends on the number of digits S per column of U.  S = 7 (default): the full significand of the
// column's largest entry (55 bits + sign), one rounding per entry of Mt U.  S = 6 (opt-in): 47 bits + sign, the
// recombination is exact (48 bits fit a double), the truncation of U is bounded by 2^(e_k - 48) per entry -- inside an FP64
// GEMM's worst-case accumulation bound at these n and five orders of magnitude inside the 1e-9 tolerance -- and every
// k-block costs 6/7 of the tensor work.  Measured at config 3: 260 -> 248 ms (the fill of the A tile does not shrink), and
// 16 x the error of an FP64 evaluation on the adversarial test: not worth being the default.
template <int S>
struct SiT {
    static_assert(S == 6 || S == 7, "digits per column");
    static constexpr int SLICES = S;
    static constexpr int BITS = 8 * S - 1;                   // scale_k = 2^(e_k - BITS)
    static constexpr int BN = SI_GCOLS * S;                  // rows of Q per group = one UMMA N (224 / 192)
    static constexpr int CHUNK = 4 * S;                      // TMEM columns of one 4-column chunk
    static constexpr int B_BYTES = BN * SI_BK;
    static constexpr int STAGE_BYTES = SI_A_BYTES + B_BYTES;
    static constexpr int SMEM_BYTES = SI_STAGES * STAGE_BYTES + 1024 + 256;
    static constexpr int SP_B_BYTES = (BN / 2) * SI_BK;      // CTA pair: half of the slice rows per CTA
    static constexpr int SP_STAGE_BYTES = SP_A_BYTES + SP_B_BYTES;
    static constexpr int SP_SMEM_BYTES = SP_STAGES * SP_STAGE_BYTES + 1024 + 256;
};

struct ScanI8Params {
    int64_t L, n;
    int32_t G, MB, KB;          // groups, marker blocks, k-blocks covering n
    const int8_t* Mt;
    int64_t pitch;
    const double* scale;        // [G*32]  2^(e_k - 55), 0 for pad columns
    double* partial;            // [2 G][L]: (group, column half) x marker
    const int2* units;          // (mb, g)
    int64_t nunits;
    uint32_t* phase_ctr;
    int32_t phases_per_unit;
    // projection mode (launch_project_i8): the right-hand matrix is FULL (no triangular cut of the K loop) and the
    // recombined products are stored, Bout[j * ldb + k] = (Mt U)_jk, instead of being folded into the row-dot
    int32_t full;
    double* Bout;
    int64_t ldb;
};

__device__ __forceinline__ void si_red_add(uint32_t* p, uint32_t v) {
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t si_ld(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int si_kb_end(int g, int KB, int full) {
    const int kb = (g * SI_GCOLS + SI_GCOLS + SI_BK - 1) / SI_BK;  // rows i <= k of U only
    return (full || kb >= KB) ? KB : kb;
}
__device__ __forceinline__ double si_s8_to_f64(uint32_t w, int b) {
    const uint32_t g = (uint32_t)((int32_t)(w << (24 - 8 * b)) >> 24);
    const uint32_t hi = (g & 0x80000000u) | ((g & 1u) * 0x3FF00000u);
    return __hiloint2double((int)hi, 0);
}

// int32 -> double without I2F.F64 (the conversion unit retires only a few results per clock per SM): 2^52 + 2^31 + x
// is exactly representable with x in the low mantissa word.
__device__ __forceinline__ double si_i2d(int x) {
    return __hiloint2double(0x43300000, x ^ (int)0x80000000) - 4503601774854144.0;
}

// One marker row (TMEM lane) of a finished accumulator, 16 of the group's 32 columns (the warp's half): recombine
// the 7 slices of each column, scale, and take the row-dot with the marker's own genotypes at those columns.
// Four independent running sums (one per column position in a chunk) combined at the end: fixed order.
// Measured (EG_SI_PROFILE): ~6,000 clk per unit whatever the arithmetic (9 FP64 operations per column or 2 plus
// integer normalisation): the 114 KB of TMEM reads per unit, competing with the MMAs for the TMEM port, set the
// pace.  Units with fewer than ~14 k-blocks are therefore epilogue-bound (3 % of the time at n = 10k).
template <int S>
__device__ __forceinline__ double si_recombine_rowdot(uint32_t taddr, const uint32_t (&mw)[4], const double* __restrict__ sc,
                                                      bool wide /* P0*256+P1 leaves int32 beyond n = 65280 */) {
    double sum[4] = {0.0, 0.0, 0.0, 0.0};
    uint32_t v4[4][32];
#pragma unroll
    for (int c = 0; c < 4; c++) {  // all 4 S columns of the four chunks in flight before the first use
        if (S == 7) ptx::tmem_ld_32x28(taddr + (uint32_t)(c * SiT<S>::CHUNK), v4[c]);
        else ptx::tmem_ld_32x24(taddr + (uint32_t)(c * SiT<S>::CHUNK), v4[c]);
    }
    ptx::tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < 4; c++) {  // 4 S TMEM columns = S slices x 4 columns (kk = 4c .. 4c+3)
        uint32_t(&v)[32] = v4[c];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            double y01, y23, y45;
            if (!wide) {
                y01 = si_i2d((int)v[0 * 4 + e] * 256 + (int)v[1 * 4 + e]);
                y23 = si_i2d((int)v[2 * 4 + e] * 256 + (int)v[3 * 4 + e]);
                y45 = si_i2d((int)v[4 * 4 + e] * 256 + (int)v[5 * 4 + e]);
            } else {
                y01 = fma(si_i2d((int)v[0 * 4 + e]), 256.0, si_i2d((int)v[1 * 4 + e]));
                y23 = fma(si_i2d((int)v[2 * 4 + e]), 256.0, si_i2d((int)v[3 * 4 + e]));
                y45 = fma(si_i2d((int)v[4 * 4 + e]), 256.0, si_i2d((int)v[5 * 4 + e]));
            }
            const double hi = fma(y01, 65536.0, y23);                      // exact (< 2^48)
            double x;
            if (S == 7) {
                const double lo = fma(y45, 256.0, si_i2d((int)v[6 * 4 + e]));  // exact
                x = fma(hi, 16777216.0, lo);                                   // the one rounding
            } else {
                x = fma(hi, 65536.0, y45);                                     // exact: 48 bits
            }
            const double t = x * __ldg(sc + c * 4 + e);                    // power-of-two scale: exact
            sum[e] = fma(t, si_s8_to_f64(mw[c], e), sum[e]);               // row-dot with m_kj in {-1,0,1}
        }
    }
    return (sum[0] + sum[1]) + (sum[2] + sum[3]);
}

// The same recombination, the 16 values of the row stored instead of summed (projection mode, S = 7 only in practice)
template <int S>
__device__ __forceinline__ void si_recombine_store(uint32_t taddr, const double* __restrict__ sc, bool wide, double* __restrict__ out,
                                                   int ncols) {
    uint32_t v4[4][32];
#pragma unroll
    for (int c = 0; c < 4; c++) {
        if (S == 7) ptx::tmem_ld_32x28(taddr + (uint32_t)(c * SiT<S>::CHUNK), v4[c]);
        else ptx::tmem_ld_32x24(taddr + (uint32_t)(c * SiT<S>::CHUNK), v4[c]);
    }
    ptx::tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < 4; c++) {
        uint32_t(&v)[32] = v4[c];
        double t[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            double y01, y23, y45;
            if (!wide) {
                y01 = si_i2d((int)v[0 * 4 + e] * 256 + (int)v[1 * 4 + e]);
                y23 = si_i2d((int)v[2 * 4 + e] * 256 + (int)v[3 * 4 + e]);
                y45 = si_i2d((int)v[4 * 4 + e] * 256 + (int)v[5 * 4 + e]);
            } else {
                y01 = fma(si_i2d((int)v[0 * 4 + e]), 256.0, si_i2d((int)v[1 * 4 + e]));
                y23 = fma(si_i2d((int)v[2 * 4 + e]), 256.0, si_i2d((int)v[3 * 4 + e]));
                y45 = fma(si_i2d((int)v[4 * 4 + e]), 256.0, si_i2d((int)v[5 * 4 + e]));
            }
            const double hi = fma(y01, 65536.0, y23);
            double x;
            if (S == 7) x = fma(hi, 16777216.0, fma(y45, 256.0, si_i2d((int)v[6 * 4 + e])));   // the one rounding
            else x = fma(hi, 65536.0, y45);
            t[e] = x * __ldg(sc + c * 4 + e);
        }
        if (c * 4 + 3 < ncols) {
            *reinterpret_cast<double2*>(out + c * 4) = make_double2(t[0], t[1]);
            *reinterpret_cast<double2*>(out + c * 4 + 2) = make_double2(t[2], t[3]);
        } else {
#pragma unroll
            for (int e = 0; e < 4; e++)
                if (c * 4 + e < ncols) out[c * 4 + e] = t[e];
        }
    }
}

template <int S>
__global__ void __launch_bounds__(SI_THREADS, 1)
scan_i8_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapB,
               const ScanI8Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SI_STAGES * SiT<S>::STAGE_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + SI_STAGES;
    uint64_t* tmem_full = bars + 2 * SI_STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmapA);
        ptx::prefetch_tmap(&tmapB);
        for (int s = 0; s < SI_STAGES; s++) {
            ptx::mbar_init(&full[s], 1);
            ptx::mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; a++) {
            ptx::mbar_init(&tmem_full[a], 1);
            ptx::mbar_init(&tmem_empty[a], 8);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 1) ptx::tmem_alloc<SI_TMEM_COLS>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer (+ K-phase flow control)
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int round = 0, known = -1;
            auto need_of = [&](int gp) -> uint32_t {
                const int64_t left = p.nunits - (int64_t)(gp / p.phases_per_unit) * gridDim.x;
                return (uint32_t)(left < (int64_t)gridDim.x ? left : (int64_t)gridDim.x);
            };
            for (int64_t u = blockIdx.x; u < p.nunits; u += gridDim.x, round++) {
                const int2 un = p.units[u];
                const int kb1 = si_kb_end(un.y, p.KB, p.full);
                for (int kb = 0; kb < kb1; kb++) {
                    if (p.phase_ctr && (kb % SI_PHASE) == 0) {
                        const int gp = round * p.phases_per_unit + kb / SI_PHASE;
                        if (gp - SI_LAG > known) {
                            uint32_t v[SI_LAG];
#pragma unroll
                            for (int q = 0; q < SI_LAG; q++) v[q] = si_ld(p.phase_ctr + max(gp - 1 - q, 0));
#pragma unroll
                            for (int q = SI_LAG - 1; q >= 0; q--)
                                if (gp - 1 - q >= 0 && gp - 1 - q > known && v[q] >= need_of(gp - 1 - q)) known = gp - 1 - q;
                            uint32_t spins = 0;
                            while (gp - SI_LAG > known) {
                                if (si_ld(p.phase_ctr + gp - SI_LAG) >= need_of(gp - SI_LAG)) known = gp - SI_LAG;
                                else if (++spins > (1u << 24)) {
                                    printf("eagle: scan_i8 flow control timed out (block %d phase %d)\n", (int)blockIdx.x, gp);
                                    __trap();
                                }
                            }
                        }
                    }
                    ptx::mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* sA = smem + stage * SiT<S>::STAGE_BYTES;
                    uint8_t* sB = sA + SI_A_BYTES;
                    ptx::mbar_expect_tx(&full[stage], SiT<S>::STAGE_BYTES);
                    ptx::tma_load_2d(sA, &tmapA, kb * SI_BK, un.x * SI_BM, &full[stage]);
                    ptx::tma_load_2d(sB, &tmapB, kb * SI_BK, un.y * SiT<S>::BN, &full[stage]);
                    ptx::tma_load_2d(sB + SiT<S>::B_BYTES / 2, &tmapB, kb * SI_BK, un.y * SiT<S>::BN + SiT<S>::BN / 2, &full[stage]);
                    if (++stage == SI_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ UMMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = ptx::make_idesc_i8(SI_BM, SiT<S>::BN);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            int round = 0;
#ifdef EG_SI_PROFILE
            long long t_acc = 0, t_full = 0, t_all = clock64(), nkb = 0;
#endif
            for (int64_t u = blockIdx.x; u < p.nunits; u += gridDim.x, round++) {
                const int2 un = p.units[u];
                const int kb1 = si_kb_end(un.y, p.KB, p.full);
#ifdef EG_SI_PROFILE
                long long t0 = clock64();
#endif
                ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
#ifdef EG_SI_PROFILE
                t_acc += clock64() - t0;
                nkb += kb1;
#endif
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * SI_ACC_COLS);
                for (int kb = 0; kb < kb1; kb++) {
#ifdef EG_SI_PROFILE
                    t0 = clock64();
#endif
                    ptx::mbar_wait(&full[stage], phase);
#ifdef EG_SI_PROFILE
                    t_full += clock64() - t0;
#endif
                    if (p.phase_ctr && ((kb % SI_PHASE) == SI_PHASE - 1 || kb == kb1 - 1)) {
                        const int ph = kb / SI_PHASE;
                        uint32_t* c = p.phase_ctr + (int64_t)round * p.phases_per_unit;
                        si_red_add(c + ph, 1u);
                        if (kb == kb1 - 1)
                            for (int q = ph + 1; q < p.phases_per_unit; q++) si_red_add(c + q, 1u);
                    }
                    ptx::tc_fence_after();
                    const uint32_t a_addr = ptx::smem_u32(smem + stage * SiT<S>::STAGE_BYTES);
                    const uint64_t a_desc = ptx::make_desc_k_sw128(a_addr);
                    const uint64_t b_desc = ptx::make_desc_k_sw128(a_addr + SI_A_BYTES);
#pragma unroll
                    for (int k = 0; k < SI_BK / 32; k++)
                        ptx::umma_i8(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc,
                                     (kb > 0 || k > 0) ? 1u : 0u);
                    ptx::umma_commit(&empty[stage]);
                    if (++stage == SI_STAGES) { stage = 0; phase ^= 1; }
                }
                ptx::umma_commit(&tmem_full[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
#ifdef EG_SI_PROFILE
            if (blockIdx.x == 7)
                printf("si profile (MMA thread, block 7): total %lld clk, units %d, k-blocks %lld (x448 = %lld clk of MMA), waiting "
                       "for a free accumulator %lld, for operands %lld\n",
                       clock64() - t_all, round, nkb, nkb * 448, t_acc, t_full);
#endif
        }
    } else {
        // ------------------------------------------------------------ epilogue: one thread = one marker row
        const int q4 = warp & 3;          // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2; // which 16 of the group's 32 columns
        int acc = 0;
        uint32_t acc_phase = 0;
#ifdef EG_SI_PROFILE
        long long e_wait = 0, e_work = 0;
#endif
        // this marker's genotypes at the 32 columns of the group (pad columns are zero in the store); the unit
        // table entry and these bytes are fetched one unit ahead, off the critical path of a short unit
        auto fetch = [&](int64_t u, int2& un, uint4& m0) {
            un = p.units[u];
            const int64_t j = (int64_t)un.x * SI_BM + q4 * 32 + lane;
            m0 = *reinterpret_cast<const uint4*>(p.Mt + (j < p.L ? j : p.L - 1) * p.pitch + (int64_t)un.y * SI_GCOLS + half * 16);
        };
        int2 un_n = make_int2(0, 0);
        uint4 m0_n = make_uint4(0, 0, 0, 0);
        if ((int64_t)blockIdx.x < p.nunits) fetch(blockIdx.x, un_n, m0_n);
        for (int64_t u = blockIdx.x; u < p.nunits; u += gridDim.x) {
            const int2 un = un_n;
            const uint4 m0 = m0_n;
            if (u + gridDim.x < p.nunits) fetch(u + gridDim.x, un_n, m0_n);
            const int64_t j = (int64_t)un.x * SI_BM + q4 * 32 + lane;
            const uint32_t mw[4] = {m0.x, m0.y, m0.z, m0.w};
            const double* sc = p.scale + (int64_t)un.y * SI_GCOLS + half * 16;
#ifdef EG_SI_PROFILE
            long long t0 = clock64();
#endif
            ptx::mbar_wait(&tmem_full[acc], acc_phase);
#ifdef EG_SI_PROFILE
            e_wait += clock64() - t0;
            t0 = clock64();
#endif
            ptx::tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(acc * SI_ACC_COLS + half * 4 * SiT<S>::CHUNK);
            double sum = 0.0;
            if (p.Bout) {   // projection mode: 16 products of this marker row go to B (lanes beyond L still read TMEM)
                const int64_t col0 = (int64_t)un.y * SI_GCOLS + half * 16;
                const int64_t left = p.n - col0;
                double* out = p.Bout + (j < p.L ? j : 0) * p.ldb + col0;
                si_recombine_store<S>(taddr, sc, p.n > 65000, out, j < p.L ? (left > 16 ? 16 : (int)(left < 0 ? 0 : left)) : 0);
            } else {
                sum = si_recombine_rowdot<S>(taddr, mw, sc, p.n > 65000);
            }
            ptx::tc_fence_before();
            __syncwarp();
#ifdef EG_SI_PROFILE
            e_work += clock64() - t0;
#endif
            if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
            if (j < p.L && !p.Bout) p.partial[((int64_t)un.y * 2 + half) * p.L + j] = sum;
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
#ifdef EG_SI_PROFILE
        if (blockIdx.x == 7 && warp == 2 && lane == 0)
            printf("si profile (epilogue warp 2, block 7): waiting for a full accumulator %lld clk, recombining %lld clk\n", e_wait,
                   e_work);
#endif
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<SI_TMEM_COLS>(tmem_base);
    }
}

// ------------------------------------------------------------------ CTA-pair version (EAGLE_SI_PAIR=1)
// Two CTAs of one TPC share a 256-marker x 224 tile: tcgen05.mma.cta_group::2, M = 256.  Each CTA stages its own
// 128 marker rows (A) and only HALF of the slice rows (B, 112 of 224), so a k-block costs 30 KB of shared-memory
// fill per SM instead of 44 KB.  Measured at n=10k (profiles/r1f_scan_sustained.txt): same throughput as the
// single-CTA kernel (70.6 vs 70.2 ms per 250k markers, both at the 1 kW power cap, where a cuBLASLt int8 GEMM
// sustains LESS than either), so the simpler kernel stays the default and this one is kept selectable.
// Barrier protocol: full[s] lives in the leader (rank 0) and collects the bytes of both CTAs' TMA loads; the
// leader's UMMA thread frees a stage / publishes an accumulator in BOTH CTAs with a multicast commit; the epilogue
// warps of both CTAs release an accumulator by arriving on the leader's tmem_empty (count 8).
template <int S>
__global__ void __launch_bounds__(SI_THREADS, 1)
scan_i8_pair_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapB,
                    const ScanI8Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SP_STAGES * SiT<S>::SP_STAGE_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + SP_STAGES;
    uint64_t* tmem_full = bars + 2 * SP_STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const int64_t cid = ptx::cluster_id_x();
    const int64_t ncl = gridDim.x / 2;
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmapA);
        ptx::prefetch_tmap(&tmapB);
        for (int s = 0; s < SP_STAGES; s++) {
            ptx::mbar_init(&full[s], 1);
            ptx::mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; a++) {
            ptx::mbar_init(&tmem_full[a], 1);
            ptx::mbar_init(&tmem_empty[a], 16);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 1) ptx::tmem_alloc_pair<SI_TMEM_COLS>(tmem_slot);
    ptx::tc_fence_before();
    ptx::cluster_sync();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer (flow control in the leader)
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int round = 0, known = -1;
            auto need_of = [&](int gp) -> uint32_t {
                const int64_t left = p.nunits - (int64_t)(gp / p.phases_per_unit) * ncl;
                return (uint32_t)(left < ncl ? left : ncl);
            };
            for (int64_t u = cid; u < p.nunits; u += ncl, round++) {
                const int2 un = p.units[u];
                const int kb1 = si_kb_end(un.y, p.KB, p.full);
                for (int kb = 0; kb < kb1; kb++) {
                    if (rank == 0 && p.phase_ctr && (kb % SI_PHASE) == 0) {
                        const int gp = round * p.phases_per_unit + kb / SI_PHASE;
                        if (gp - SI_LAG > known) {
                            uint32_t v[SI_LAG];
#pragma unroll
                            for (int q = 0; q < SI_LAG; q++) v[q] = si_ld(p.phase_ctr + max(gp - 1 - q, 0));
#pragma unroll
                            for (int q = SI_LAG - 1; q >= 0; q--)
                                if (gp - 1 - q >= 0 && gp - 1 - q > known && v[q] >= need_of(gp - 1 - q)) known = gp - 1 - q;
                            uint32_t spins = 0;
                            while (gp - SI_LAG > known) {
                                if (si_ld(p.phase_ctr + gp - SI_LAG) >= need_of(gp - SI_LAG)) known = gp - SI_LAG;
                                else if (++spins > (1u << 24)) {
                                    printf("eagle: scan_i8 (pair) flow control timed out (cluster %d phase %d)\n", (int)cid, gp);
                                    __trap();
                                }
                            }
                        }
                    }
                    ptx::mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* sA = smem + stage * SiT<S>::SP_STAGE_BYTES;
                    uint8_t* sB = sA + SP_A_BYTES;
                    const uint32_t lead_full = ptx::mapa(ptx::smem_u32(&full[stage]), 0);
                    if (rank == 0) ptx::mbar_expect_tx(&full[stage], 2 * SiT<S>::SP_STAGE_BYTES);
                    ptx::tma_load_2d_pair(sA, &tmapA, kb * SI_BK, un.x * (2 * SI_BM) + (int)rank * SI_BM, lead_full);
                    ptx::tma_load_2d_pair(sB, &tmapB, kb * SI_BK, un.y * SiT<S>::BN + (int)rank * (SiT<S>::BN / 2), lead_full);
                    if (++stage == SP_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ UMMA issuer (leader CTA only)
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc = ptx::make_idesc_i8(2 * SI_BM, SiT<S>::BN);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            int round = 0;
            for (int64_t u = cid; u < p.nunits; u += ncl, round++) {
                const int2 un = p.units[u];
                const int kb1 = si_kb_end(un.y, p.KB, p.full);
                ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * SI_ACC_COLS);
                for (int kb = 0; kb < kb1; kb++) {
                    ptx::mbar_wait(&full[stage], phase);
                    if (p.phase_ctr && ((kb % SI_PHASE) == SI_PHASE - 1 || kb == kb1 - 1)) {
                        const int ph = kb / SI_PHASE;
                        uint32_t* c = p.phase_ctr + (int64_t)round * p.phases_per_unit;
                        si_red_add(c + ph, 1u);
                        if (kb == kb1 - 1)
                            for (int q = ph + 1; q < p.phases_per_unit; q++) si_red_add(c + q, 1u);
                    }
                    ptx::tc_fence_after();
                    const uint32_t a_addr = ptx::smem_u32(smem + stage * SiT<S>::SP_STAGE_BYTES);
                    const uint64_t a_desc = ptx::make_desc_k_sw128(a_addr);
                    const uint64_t b_desc = ptx::make_desc_k_sw128(a_addr + SP_A_BYTES);
#pragma unroll
                    for (int k = 0; k < SI_BK / 32; k++)
                        ptx::umma_i8_pair(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc,
                                          (kb > 0 || k > 0) ? 1u : 0u);
                    ptx::umma_commit_pair(&empty[stage], 3);
                    if (++stage == SP_STAGES) { stage = 0; phase ^= 1; }
                }
                ptx::umma_commit_pair(&tmem_full[acc], 3);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue: one thread = one marker row
        const int q4 = warp & 3;          // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2; // which 16 of the group's 32 columns
        int acc = 0;
        uint32_t acc_phase = 0;
        auto fetch = [&](int64_t u, int2& un, uint4& m0) {
            un = p.units[u];
            const int64_t j = (int64_t)un.x * (2 * SI_BM) + (int64_t)rank * SI_BM + q4 * 32 + lane;
            m0 = *reinterpret_cast<const uint4*>(p.Mt + (j < p.L ? j : p.L - 1) * p.pitch + (int64_t)un.y * SI_GCOLS + half * 16);
        };
        int2 un_n = make_int2(0, 0);
        uint4 m0_n = make_uint4(0, 0, 0, 0);
        if (cid < p.nunits) fetch(cid, un_n, m0_n);
        for (int64_t u = cid; u < p.nunits; u += ncl) {
            const int2 un = un_n;
            const uint4 m0 = m0_n;
            if (u + ncl < p.nunits) fetch(u + ncl, un_n, m0_n);
            const int64_t j = (int64_t)un.x * (2 * SI_BM) + (int64_t)rank * SI_BM + q4 * 32 + lane;
            const uint32_t mw[4] = {m0.x, m0.y, m0.z, m0.w};
            const double* sc = p.scale + (int64_t)un.y * SI_GCOLS + half * 16;
            ptx::mbar_wait(&tmem_full[acc], acc_phase);
            ptx::tc_fence_after();
            const double sum = si_recombine_rowdot<S>(
                tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(acc * SI_ACC_COLS + half * 4 * SiT<S>::CHUNK), mw, sc, p.n > 65000);
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tmem_empty[acc]), 0));
            if (j < p.L) p.partial[((int64_t)un.y * 2 + half) * p.L + j] = sum;
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    ptx::tc_fence_before();
    ptx::cluster_sync();  // no CTA leaves while its peer can still signal it or read its shared memory
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc_pair<SI_TMEM_COLS>(tmem_base);
    }
}

// ------------------------------------------------------------------ slicing of U
// per column: e_k with max_i |U_ik| * 2^(-e_k) in [0.5, 127/128) (so that the top digit, carry included,
// stays <= 127); scale_k = 2^(e_k - 55).  A column whose largest magnitude is below 2^-1020 (e_k < -1019) gets
// scale_k = ldexp(1, e_k - 55) = 0 and its products are flushed to 0: eigenvector columns (unit norm, or scaled by
// sqrt(count) >= 1) and the scan's folded W never come near it (tests/test_gpu_bcache_exact.py pins the behaviour)
__global__ void __launch_bounds__(256) si_colscale_kernel(const double* __restrict__ Wp, int64_t n, int64_t ld,
                                                          int32_t* __restrict__ expo, double* __restrict__ scale,
                                                          int64_t ncols_pad, int bits, int full) {
    // |x| bit patterns order like unsigned integers and NaN > Inf > finite: an integer max finds the column's largest
    // magnitude AND lets a NaN / Inf through (fmax would drop a NaN and turn a poisoned column into zeros)
    const int64_t k = blockIdx.x;
    unsigned long long m = 0;
    if (k < n)
        for (int64_t i = threadIdx.x; i <= (full ? n - 1 : k); i += 256) {
            const unsigned long long b = (unsigned long long)__double_as_longlong(Wp[i + k * ld]) & 0x7FFFFFFFFFFFFFFFull;
            m = b > m ? b : m;
        }
    __shared__ unsigned long long sh[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
        m = t > m ? t : m;
    }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0 && k < ncols_pad) {
        for (int w = 1; w < 8; w++) m = sh[w] > m ? sh[w] : m;
        int e = 0;
        double s = 0.0;
        if (k < n && m >= 0x7FF0000000000000ull) {
            s = __longlong_as_double(0x7FF8000000000000LL);  // NaN / Inf in U poisons the column, as in the reference's product
        } else if (k < n && m) {
            if (frexp(__longlong_as_double((long long)m), &e) >= 0.9921875) e++;
            s = ldexp(1.0, e - bits);
        }
        expo[k] = e;
        scale[k] = s;
    }
}
// Q rows for column k = 32 g + kk: g*224 + (kk>>2)*28 + s*4 + (kk&3); thread -> 4 consecutive i.  Columns are strided
// over gridDim.y, which cannot exceed 65,535: n beyond that (the projection of a larger U) takes a second pass.
template <int S>
__global__ void __launch_bounds__(256) si_slice_kernel(const double* __restrict__ Wp, int64_t n, int64_t ld,
                                                       const int32_t* __restrict__ expo, int8_t* __restrict__ Q,
                                                       int64_t Kp, int full, int64_t ncols_pad) {
    const int64_t i0 = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;
    if (i0 >= Kp) return;
    for (int64_t k = blockIdx.y; k < ncols_pad; k += gridDim.y) {
        const int64_t g = k / SI_GCOLS;
        const int kk = (int)(k - g * SI_GCOLS);
        int8_t* base = Q + (g * SiT<S>::BN + (kk >> 2) * SiT<S>::CHUNK + (kk & 3)) * Kp + i0;
        uint32_t out[S];
#pragma unroll
        for (int s = 0; s < S; s++) out[s] = 0;
        if (k < n) {
            const int e = expo[k];
#pragma unroll
            for (int d = 0; d < 4; d++) {
                const int64_t i = i0 + d;
                if ((full || i <= k) && i < n) {
                    const double xs = ldexp(Wp[i + k * ld], SiT<S>::BITS - e);  // |xs| <= 127 * 2^(8 S - 8) (exact scaling)
                    long long X = fabs(xs) < 3.6e16 ? __double2ll_rn(xs) : 0;  // rint: |residual| <= 1/2 unit = 2^(e - 8 S)  // NaN / Inf: the column's scale is NaN
#pragma unroll
                    for (int s = S - 1; s > 0; s--) {          // balanced digits, least significant first
                        const int q = (int)(int8_t)(X & 0xFF);
                        out[s] |= ((uint32_t)q & 0xFFu) << (8 * d);
                        X = (X - q) >> 8;                              // exact: X - q is a multiple of 256
                    }
                    out[0] |= ((uint32_t)(int)X & 0xFFu) << (8 * d);  // top digit in [-127, 127]
                }
            }
        }
#pragma unroll
        for (int s = 0; s < S; s++) *reinterpret_cast<uint32_t*>(base + (int64_t)s * 4 * Kp) = out[s];
    }
}

// (mb, g) -> position in the super-tile order
__global__ void si_units_kernel(int2* units, int MB, int G, int MSUP, int GSUP) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)MB * G) return;
    const int mb = (int)(t % MB), g = (int)(t / MB);
    const int ms = mb / MSUP, gs = g / GSUP;
    const int msz = min(MSUP, MB - ms * MSUP);
    const int64_t u = (int64_t)ms * MSUP * G + (int64_t)gs * GSUP * msz + (int64_t)(g - gs * GSUP) * msz +
                      (mb - ms * MSUP);
    units[u] = make_int2(mb, g);
}

// vara_j = sum over (group, column half) in index order; zeroed rows give 0
__global__ void __launch_bounds__(256) si_reduce_kernel(const double* __restrict__ partial, int64_t L, int G,
                                                        const int64_t* __restrict__ zero_rows, int n_zero,
                                                        double* __restrict__ vara) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= L) return;
    double s = 0.0;
    for (int g = 0; g < G; g++) s += partial[(int64_t)g * L + j];
    for (int z = 0; z < n_zero; z++)
        if (zero_rows[z] == j) s = 0.0;
    vara[j] = s;
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled si_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(f);
    }
    return fn;
}
static int si_make_map(CUtensorMap* m, const void* base, int64_t inner, int64_t rows, int64_t pitch, int box_rows) {
    PFN_encodeTiled enc = si_encode_fn();
    if (!enc) return set_error(EG_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
    const cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)pitch};
    const cuuint32_t box[2] = {128, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(EG_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return EG_OK;
}

struct ScanI8Workspace {
    int device = -1;
    int8_t* Q = nullptr;        size_t q_cap = 0;
    double* scale = nullptr;    size_t sc_cap = 0;
    int32_t* expo = nullptr;    size_t expo_cap = 0;
    double* partial = nullptr;  size_t part_cap = 0;
    int2* units = nullptr;      size_t unit_cap = 0;  int units_MB = -1, units_G = -1, units_shape = -1;
    uint32_t* phase = nullptr;  size_t phase_cap = 0;
    int64_t sliced_n = -1;      // n and digits of the U whose slices Q / expo / scale hold (launch_scan_i8_t's `sliced`)
    int sliced_digits = 0;
};
static thread_local ScanI8Workspace g_si;

void scan_kernel_mark(int which, cudaStream_t st, double ops);

void scan_i8_release() {
    cudaFree(g_si.Q); cudaFree(g_si.scale); cudaFree(g_si.expo); cudaFree(g_si.partial); cudaFree(g_si.units);
    cudaFree(g_si.phase);
    g_si = ScanI8Workspace();
}
template <class T>
static int si_grow(T** p, size_t* cap, size_t need, const char* what) {
    if (need <= *cap && *p) return EG_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    if (malloc_retry((void**)p, need * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        return set_error(EG_ERR_ALLOC, "out of device memory for %s (%zu bytes)", what, need * sizeof(T));
    }
    *cap = need;
    return EG_OK;
}

// digits per column of U: 7 (default: the full significand of every column's largest entry) or 6 (EAGLE_SCAN_DIGITS=6)
static int g_si_digits = 0;
int scan_i8_digits() {
    if (!g_si_digits) {
        const char* e = getenv("EAGLE_SCAN_DIGITS");
        g_si_digits = (e && e[0] == '6') ? 6 : 7;
    }
    return g_si_digits;
}
void scan_i8_set_digits(int d) { g_si_digits = d == 6 ? 6 : 7; }

// vara for all rows of an Mt store from the folded matrix U (columns 0..n-1 of Wp).  sliced: U is the matrix the previous
// call on this thread sliced (the pieces of a streamed scan after the first): the digits, exponents and column scales in
// the workspace are used as they are, and only the contraction and the reduction run.
template <int S>
static int launch_scan_i8_t(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp, int64_t Kpad,
                            const int64_t* d_zero_rows, int n_zero, double* d_vara, cudaStream_t st, double* d_Bout = nullptr,
                            int64_t ldb = 0, bool sliced = false) {
    const int full = d_Bout ? 1 : 0;
    int dev = 0;
    EG_CUDA(cudaGetDevice(&dev));
    if (g_si.device != dev) {
        if (sliced) return set_error(EG_ERR_ARG, "scan_i8: no sliced U on this device");
        if (g_si.device >= 0) scan_i8_release();
        g_si.device = dev;
    }
    const int G = (int)((n + SI_GCOLS - 1) / SI_GCOLS);
    const char* env_pair = getenv("EAGLE_SI_PAIR");
    const bool pair = env_pair && env_pair[0] == '1' && !full;   // CTA pairs (cta_group::2): opt-in, see the kernel's header
    const int rows_per_unit = pair ? 2 * SI_BM : SI_BM;
    const int MB = (int)((L + rows_per_unit - 1) / rows_per_unit);
    const int64_t Kp = round_up(n, 128);
    const int KB = (int)(Kp / SI_BK);
    if (pitch < Kp || pitch < (int64_t)G * SI_GCOLS)
        return set_error(EG_ERR_ARG, "scan_i8: Mt pitch %lld too small for n=%lld", (long long)pitch, (long long)n);
    EG_TRY(si_grow(&g_si.Q, &g_si.q_cap, (size_t)G * SiT<S>::BN * Kp, "sliced U"));
    EG_TRY(si_grow(&g_si.scale, &g_si.sc_cap, (size_t)G * SI_GCOLS, "column scales"));
    EG_TRY(si_grow(&g_si.expo, &g_si.expo_cap, (size_t)G * SI_GCOLS, "column exponents"));
    if (!full) EG_TRY(si_grow(&g_si.partial, &g_si.part_cap, (size_t)2 * G * L, "per-group partial sums"));
    const int64_t nunits = (int64_t)MB * G;
    int msup = pair ? SP_MSUP_DEFAULT : SI_MSUP_DEFAULT, gsup = pair ? SP_GSUP_DEFAULT : SI_GSUP_DEFAULT;
    if (const char* e = getenv("EAGLE_SI_MSUP")) msup = atoi(e) > 0 ? atoi(e) : msup;
    if (const char* e = getenv("EAGLE_SI_GSUP")) gsup = atoi(e) > 0 ? atoi(e) : gsup;
    const int shape_key = (pair ? 1000000 : 0) + msup * 1000 + gsup;
    if (g_si.units_MB != MB || g_si.units_G != G || g_si.units_shape != shape_key || !g_si.units) {
        EG_TRY(si_grow(&g_si.units, &g_si.unit_cap, (size_t)nunits, "unit table"));
        si_units_kernel<<<(unsigned)((nunits + 255) / 256), 256, 0, st>>>(g_si.units, MB, G, msup, gsup);
        EG_TRY(check_launch("si_units_kernel"));
        g_si.units_MB = MB;
        g_si.units_G = G;
        g_si.units_shape = shape_key;
    }
    if (sliced && (g_si.sliced_n != n || g_si.sliced_digits != S || !g_si.Q))
        return set_error(EG_ERR_ARG, "scan_i8: no sliced U of this shape in the workspace");
    // 1. slice U
    if (!sliced) {
        si_colscale_kernel<<<(unsigned)(G * SI_GCOLS), 256, 0, st>>>(d_Wp, n, Kpad, g_si.expo, g_si.scale, (int64_t)G * SI_GCOLS,
                                                                     SiT<S>::BITS, full);
        EG_TRY(check_launch("si_colscale_kernel"));
        const int64_t ncols_pad = (int64_t)G * SI_GCOLS;
        si_slice_kernel<S><<<dim3((unsigned)((Kp / 4 + 255) / 256), (unsigned)(ncols_pad < 65535 ? ncols_pad : 65535)), 256, 0, st>>>(
            d_Wp, n, Kpad, g_si.expo, g_si.Q, Kp, full, ncols_pad);
        EG_TRY(check_launch("si_slice_kernel"));
        g_si.sliced_n = full ? -1 : n;   // a projection slices another matrix: the scan's U is gone
        g_si.sliced_digits = S;
    }
    // 2. the int8 contraction with fused recombination + row-dot
    CUtensorMap tA, tB;
    EG_TRY(si_make_map(&tA, d_Mt, Kp, L, pitch, SI_BM));
    EG_TRY(si_make_map(&tB, g_si.Q, Kp, (int64_t)G * SiT<S>::BN, Kp, SiT<S>::BN / 2));
    ScanI8Params p;
    p.L = L; p.n = n; p.G = G; p.MB = MB; p.KB = KB;
    p.Mt = d_Mt; p.pitch = pitch; p.scale = g_si.scale; p.partial = g_si.partial;
    p.units = g_si.units; p.nunits = nunits;
    p.full = full; p.Bout = d_Bout; p.ldb = ldb;
    const int sms = num_sms();
    const int workers_max = pair ? sms / 2 : sms;          // CTAs, or CTA pairs
    const int workers = nunits < workers_max ? (int)nunits : workers_max;
    p.phases_per_unit = (KB + SI_PHASE - 1) / SI_PHASE;
    const int64_t rounds = (nunits + workers - 1) / workers;
    const size_t nctr = (size_t)rounds * p.phases_per_unit;
    const char* env_fc = getenv("EAGLE_SCAN_FLOWCTL");
    const bool flow = !(env_fc && env_fc[0] == '0') && workers > 1 && nctr < ((size_t)1 << 28);
    p.phase_ctr = nullptr;
    if (flow) {
        EG_TRY(si_grow(&g_si.phase, &g_si.phase_cap, nctr, "flow-control counters"));
        EG_CUDA(cudaMemsetAsync(g_si.phase, 0, nctr * sizeof(uint32_t), st));
        p.phase_ctr = g_si.phase;
    }
    const int smem_bytes = pair ? SiT<S>::SP_SMEM_BYTES : SiT<S>::SMEM_BYTES;
    if (pair) EG_CUDA(cudaFuncSetAttribute(scan_i8_pair_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    else EG_CUDA(cudaFuncSetAttribute(scan_i8_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(pair ? 2 * workers : workers));
    cfg.blockDim = dim3(SI_THREADS);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeCooperative;           // co-residency: the flow control spins on other CTAs
    attr[0].val.cooperative = flow ? 1 : 0;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pair ? 2 : 1;
    double kblocks = 0.0;  // executed int8 ops: 2 * rows * 224 * 128 per (marker block, k-block of a group)
    for (int g = 0; g < G; g++) {
        const int kb = (g * SI_GCOLS + SI_GCOLS + SI_BK - 1) / SI_BK;
        kblocks += (full || kb >= KB) ? KB : kb;
    }
    scan_kernel_mark(0, st, kblocks * MB * 2.0 * rows_per_unit * SiT<S>::BN * SI_BK);
    if (pair) EG_CUDA(cudaLaunchKernelEx(&cfg, scan_i8_pair_kernel<S>, tA, tB, p));
    else EG_CUDA(cudaLaunchKernelEx(&cfg, scan_i8_kernel<S>, tA, tB, p));
    EG_TRY(check_launch("scan_i8_kernel"));
    scan_kernel_mark(1, st, 0.0);
    if (full) return EG_OK;
    // 3. groups summed in index order
    si_reduce_kernel<<<(unsigned)((L + 255) / 256), 256, 0, st>>>(g_si.partial, L, 2 * G, d_zero_rows, n_zero, d_vara);
    return check_launch("si_reduce_kernel");
}

int launch_scan_i8(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp, int64_t Kpad,
                   const int64_t* d_zero_rows, int n_zero, double* d_vara, cudaStream_t st, bool sliced) {
    return scan_i8_digits() == 7 ? launch_scan_i8_t<7>(d_Mt, L, n, pitch, d_Wp, Kpad, d_zero_rows, n_zero, d_vara, st, nullptr, 0, sliced)
                                 : launch_scan_i8_t<6>(d_Mt, L, n, pitch, d_Wp, Kpad, d_zero_rows, n_zero, d_vara, st, nullptr, 0, sliced);
}

// B = Mt * U for a full n x n FP64 matrix U (column-major, ld): every entry exact up to one rounding (7 digits per
// column of U).  d_B: L rows, row pitch ldb >= n doubles.  What am.AM_resident computes once per search (B = M^T U, U the
// eigenvectors of K) so that every later scan is one pass over B instead of an n^2 L contraction.
int launch_project_i8(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_U, int64_t ld, double* d_B,
                      int64_t ldb, cudaStream_t st) {
    return launch_scan_i8_t<7>(d_Mt, L, n, pitch, d_U, ld, nullptr, 0, nullptr, st, d_B, ldb);
}

}  // namespace eg
