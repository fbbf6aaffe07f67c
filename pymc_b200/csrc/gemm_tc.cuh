// D[c][j] = alpha * sum_k A[c][k] * B[j][k]  on the 5th-generation tensor cores (tcgen05.mma, TMEM, TMA): the
// PERFORMANCE mode of the dense Gaussian config (BASELINE #5: grad = -P q, w = Sigma g, p0 = L^-T z, v0 = L z at
// n = 10^4).  Same arithmetic as csrc/logistic_tc.cuh: every fp64 operand is hi + lo in fp16 (22 significant bits), a
// product is hi*hi + hi*lo + lo*hi in three kind::f16 MMAs with fp32 accumulation, and the fp32 accumulator in TMEM
// only ever covers kGtDrain k-blocks (64 terms each) before it is drained into compensated fp32 register sums (kahan_add).
// The fp64 DMMA kernel of dense.cuh stays the parity mode.
//
// B (the model's n x n matrices) is split once at b200_model_set_precision; A (the chains' vectors) is split by
// gemm_tc_split_kernel before every GEMM.  Both are K-major fp16 [rows][Kpad] in HBM, TMA-loaded in 64-wide k-blocks with
// SWIZZLE_128B.  CTA tile = 128 chains x 144 outputs: 70 x 2 = 140 tiles for n = 10^4 and 256 chains -- one wave of 148 SMs.
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2..9 epilogue (two warps per TMEM subpartition, 72 columns
// each, 72 compensated fp32 sums per thread).  The accumulator is double-buffered in TMEM so a drain overlaps the next MMAs.
#pragma once
#include "logistic_tc.cuh"

namespace b200 {

constexpr int kGtM = 128;        // chains per tile (TMEM lanes)
constexpr int kGtN = 144;        // outputs per tile
constexpr int kGtKB = 64;        // k per block (128 B of fp16: one swizzle row)
constexpr int kGtStages = 3;
constexpr int kGtDrain = 1;      // k-blocks per fp32 accumulation chunk: the tensor cores' accumulate rounds toward zero
                                 // (logistic_tc.cuh), so a chunk is 12 MMAs with only the last 4 (hi*hi) at full magnitude
constexpr int kGtThreads = 320;  // 10 warps
constexpr uint32_t kGtABytes = kGtM * kGtKB * 2;                    // 16 KB per piece
constexpr uint32_t kGtBBytes = kGtN * kGtKB * 2;                    // 18 KB per piece
constexpr uint32_t kGtStageBytes = 2 * kGtABytes + 2 * kGtBBytes;   // 68 KB
constexpr size_t kGtSmemBytes = 1024 + (size_t)kGtStages * kGtStageBytes + 256;
constexpr uint32_t kGtIdesc = (1u << 4) | ((uint32_t)(kGtN >> 3) << 17) | ((uint32_t)(kGtM >> 4) << 24);

__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}

// (tc_ld16: logistic_tc.cuh)

// Compensated (Kahan) fp32 accumulation of one drained value: s + (-c) carries the running sum to ~2^-24 of its magnitude
// independently of the number of terms, with four FADDs (128 lanes/clk/SM).  The first version of this epilogue converted
// every drained value to fp64 (F2F.F64.F32 + DADD): ncu (profiles/r2_tc_gemm_tc_*) showed the tensor pipe 27 % busy and the
// kernel waiting on exactly those two opcodes (22 % of the instructions each, 47 % of the stall samples) with a quarter of the
// accumulators spilled -- the conversion unit, not the MMAs or L2 (40 % of the LTS cap), set the pace.
__device__ __forceinline__ void kahan_add(float& s, float& c, float x) {
    const float y = x - c;
    const float t = s + y;
    c = (t - s) - y;
    s = t;
}

struct GemmTcArgs {
    int C, Nout, n_kblocks;   // chains, outputs, k-blocks of 64 (operands are zero padded to that)
    double alpha;
    double* D;                // [C][ldd]
    long long ldd;
    int n_tiles_n, n_tiles;   // output tiles per chain tile, total tiles
};

__global__ void __launch_bounds__(kGtThreads, 1)
    gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo, const GemmTcArgs G) {
    extern __shared__ char gt_smem_raw[];
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(gt_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(base + kGtStages * kGtStageBytes);
    uint64_t* full = bars;                 // [stages] TMA -> MMA
    uint64_t* empty = bars + kGtStages;    // [stages] MMA -> TMA
    uint64_t* acc_full = bars + 8;         // [2] MMA (chunk done) -> epilogue
    uint64_t* acc_empty = bars + 10;       // [2] epilogue (drained) -> MMA
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int i = 0; i < kGtStages; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 256);
        }
    }
    if (warp == 1) {
        const uint32_t ncols = 512;
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const uint32_t tAcc[2] = {tmem, tmem + 256};
    const int KB = G.n_kblocks;
    const int n_chunks = (KB + kGtDrain - 1) / kGtDrain;

    if (warp == 0) {
        if (lane == 0) {
            long long it = 0;  // k-blocks loaded so far (over all tiles of this CTA)
            for (int tile = blockIdx.x; tile < G.n_tiles; tile += gridDim.x) {
                const int c0 = (tile / G.n_tiles_n) * kGtM, j0 = (tile % G.n_tiles_n) * kGtN;
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    const int st = (int)(it % kGtStages);
                    if (it >= kGtStages) tc_mbar_wait(&empty[st], (uint32_t)(((it / kGtStages) - 1) & 1));
                    char* dst = base + st * kGtStageBytes;
                    mbar_expect_tx(&full[st], kGtStageBytes);
                    tc_tma_load_2d(dst, &map_a_hi, kb * kGtKB, c0, &full[st]);
                    tc_tma_load_2d(dst + kGtABytes, &map_a_lo, kb * kGtKB, c0, &full[st]);
                    tc_tma_load_2d(dst + 2 * kGtABytes, &map_b_hi, kb * kGtKB, j0, &full[st]);
                    tc_tma_load_2d(dst + 2 * kGtABytes + kGtBBytes, &map_b_lo, kb * kGtKB, j0, &full[st]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            long long it = 0, chunk = 0;  // k-blocks / accumulation chunks issued so far
            for (int tile = blockIdx.x; tile < G.n_tiles; tile += gridDim.x) {
                for (int ch = 0; ch < n_chunks; ++ch, ++chunk) {
                    const int b = (int)(chunk & 1);
                    if (chunk >= 2) tc_mbar_wait(&acc_empty[b], (uint32_t)(((chunk >> 1) - 1) & 1));
                    tc_fence_after();
                    const int kb_end = min(KB, (ch + 1) * kGtDrain);
                    uint32_t acc = 0;
                    for (int kb = ch * kGtDrain; kb < kb_end; ++kb, ++it) {
                        const int st = (int)(it % kGtStages);
                        tc_mbar_wait(&full[st], (uint32_t)((it / kGtStages) & 1));
                        tc_fence_after();
                        const uint32_t a_hi = smem_u32(base + st * kGtStageBytes), a_lo = a_hi + kGtABytes;
                        const uint32_t b_hi = a_hi + 2 * kGtABytes, b_lo = b_hi + kGtBBytes;
#pragma unroll
                        for (int prod = 0; prod < 3; ++prod) {  // hi*lo, lo*hi, then hi*hi (small products first)
                            const uint32_t a0 = prod == 1 ? a_lo : a_hi, b0 = prod == 0 ? b_lo : b_hi;
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                tc_mma_ss(tAcc[b], tc_desc(a0 + ks * 32, 16, 1024), tc_desc(b0 + ks * 32, 16, 1024), kGtIdesc, acc);
                                acc = 1;
                            }
                        }
                        tc_commit(&empty[st]);
                    }
                    tc_commit(&acc_full[b]);
                }
            }
        }
    } else {
        // epilogue: warps 2..9; subpartition = warp % 4, column half = (warp - 2) / 4
        const int sub = warp & 3, half = (warp - 2) >> 2;
        const uint32_t lane_addr = (uint32_t)(sub * 32) << 16;
        const int row = sub * 32 + lane;
        // this thread's 72 accumulator columns: [64 half, 64 half + 64) and [128 + 8 half, 128 + 8 half + 8)
        const int colA = half * 64, colB = 128 + half * 8;
        long long chunk = 0;
        for (int tile = blockIdx.x; tile < G.n_tiles; tile += gridDim.x) {
            const int c = (tile / G.n_tiles_n) * kGtM + row, j0 = (tile % G.n_tiles_n) * kGtN;
            float sum[kGtN / 2], comp[kGtN / 2];
#pragma unroll
            for (int k = 0; k < kGtN / 2; ++k) { sum[k] = 0.0f; comp[k] = 0.0f; }
            for (int ch = 0; ch < n_chunks; ++ch, ++chunk) {
                const int b = (int)(chunk & 1);
                tc_mbar_wait(&acc_full[b], (uint32_t)((chunk >> 1) & 1));
                tc_fence_after();
#pragma unroll
                for (int piece = 0; piece < 4; ++piece) {  // 16 TMEM columns at a time: 144 accumulator + 16 staging registers
                    uint32_t v[16];
                    tc_ld16(tAcc[b] + lane_addr + colA + 16 * piece, v);
                    tc_wait_ld();
#pragma unroll
                    for (int k = 0; k < 16; ++k) kahan_add(sum[16 * piece + k], comp[16 * piece + k], __uint_as_float(v[k]));
                }
                {
                    uint32_t v[8];
                    tc_ld8(tAcc[b] + lane_addr + colB, v);
                    tc_wait_ld();
#pragma unroll
                    for (int k = 0; k < 8; ++k) kahan_add(sum[64 + k], comp[64 + k], __uint_as_float(v[k]));
                }
                tc_fence_before();
                tc_mbar_arrive(&acc_empty[b]);
            }
            if (c < G.C) {
                double* d = G.D + (long long)c * G.ldd + j0;
#pragma unroll
                for (int k = 0; k < 64; ++k)
                    if (j0 + colA + k < G.Nout) d[colA + k] = G.alpha * ((double)sum[k] - (double)comp[k]);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (j0 + colB + k < G.Nout) d[colB + k] = G.alpha * ((double)sum[64 + k] - (double)comp[64 + k]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        const uint32_t ncols = 512;
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(ncols) : "memory");
    }
}

// fp64 [rows][ld] (first `cols` columns) -> fp16 pieces [rows_pad][kpad], zero padded
__global__ void __launch_bounds__(256) gemm_tc_split_kernel(const double* __restrict__ X, long long rows, long long cols, long long ld,
                                                            __half* __restrict__ Xh, __half* __restrict__ Xl, long long rows_pad,
                                                            long long kpad) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows_pad * kpad) return;
    const long long r = e / kpad, k = e % kpad;
    const double v = (r < rows && k < cols) ? X[r * ld + k] : 0.0;
    const __half hi = __double2half(v);
    Xh[e] = hi;
    Xl[e] = __double2half(v - (double)__half2float(hi));
}

}  // namespace b200
