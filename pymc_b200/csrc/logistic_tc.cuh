// Logistic GLM, tensor-core PERFORMANCE mode (BASELINE config 3; VERDICT r1 item N2): the two contractions of one batched
// leapfrog,  eta = X beta  and  G = X^T (y - sigmoid(eta)),  on the 5th-generation tensor cores (tcgen05.mma, accumulators
// in TMEM, operands staged by TMA) instead of the fp64 DMMA path of dense.cuh.
//
// tcgen05 has no fp64 kind, so every fp64 operand is split into two fp16 pieces, v = hi + lo with hi = fp16(v) and
// lo = fp16(v - hi) (22 significant bits; absolute floor 2^-25 where lo is subnormal), and a product is evaluated as
// hi*hi + hi*lo + lo*hi in three kind::f16 MMAs with fp32 accumulation (the lo*lo term is below 2^-22 relative).
// fp32 accumulators only ever cover a few slabs: X beta sums K = 128 terms, and the gradient accumulator in TMEM is drained
// into fp64 every kTcDrain 128-row slabs, so neither fp32 rounding nor the tensor cores' one-sided accumulate rounding builds up.
// Accuracy against the fp64 path is measured by tests/test_gpu_tc.py and reported in profiles/ (parity report).  The fp64
// DMMA kernel stays the parity mode.
//
// One CTA = 128 chains x a strided set of 128-row slabs of X.  Per slab (FlashAttention-shaped, P kept in TMEM):
//   TMA   : X_hi, X_lo slab [128 rows][128 features] fp16 -> smem (SWIZZLE_128B, two 64-column boxes each) and the slab's
//           128 labels (fp32), 2 stages
//   GEMM 1: D1[c][i] = sum_k beta[c][k] X[i][k]     A = beta pieces (smem, K-major), B = X pieces (smem, K-major)
//   epilog: thread c (TMEM lane c) reads its eta values (tcgen05.ld), computes r = y - sigmoid(eta) and the
//           log-likelihood terms in fp32, splits r into fp16 pieces and writes them back to TMEM (tcgen05.st)
//   GEMM 2: D2[c][k] += sum_i r[c][i] X[i][k]        A = r pieces (TMEM), B = the SAME X bytes read MN-major
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2..17 = epilogue (four per TMEM
// subpartition, 32 rows of the slab each).  D1 is double-buffered so GEMM 1 of slab s+1 runs under the epilogue of slab s.
// TMEM columns (512): D1[0] 0..127, D1[1] 128..255, D2 256..383, r_hi 384..447, r_lo 448..511.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace b200 {

constexpr int kTcRows = 128;      // rows of X per slab (N of GEMM 1, K of GEMM 2)
constexpr int kTcChains = 128;    // chains per CTA (M of both GEMMs = TMEM lanes)
constexpr int kTcK = 128;         // features (padded)
constexpr int kTcStages = 2;      // X slab stages in shared memory
constexpr int kTcDrain = 2;       // slabs per fp32 gradient accumulation chunk (16 full-magnitude accumulate steps)
constexpr uint32_t kTcBlockBytes = kTcRows * 64 * 2;          // one [128 rows][64 cols] fp16 box = 16 KB
constexpr uint32_t kTcPieceBytes = 2 * kTcBlockBytes;         // one piece of a [128][128] tile = 32 KB
constexpr uint32_t kTcStageBytes = 2 * kTcPieceBytes;         // X_hi + X_lo = 64 KB

// ---- raw PTX wrappers ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni TC_DONE;\n"
        "bra.uni TC_WAIT;\n"
        "TC_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tc_tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {  // arrives on `bar` when every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]
__device__ __forceinline__ void tc_mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void tc_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp): start address, leading / stride byte
// offsets (all >> 4), version 1 (Blackwell) at bit 46, layout type SWIZZLE_128B = 2 at bits 61..63
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (bits 4..5 = 1), A = B = F16 (formats 0), N >> 3 at bit 17,
// M >> 4 at bit 24; bit 16 = B is MN-major
constexpr uint32_t kTcIdesc = (1u << 4) | ((uint32_t)(kTcRows >> 3) << 17) | ((uint32_t)(kTcChains >> 4) << 24);
constexpr uint32_t kTcIdescBmn = kTcIdesc | (1u << 16);

// byte offset of element (row r, column k) of a [128][128] fp16 tile stored as two [128][64] blocks, rows 128 B apart,
// 16-byte chunks XOR-swizzled with the row (SWIZZLE_128B: what TMA writes and what the descriptors above describe)
__device__ __forceinline__ uint32_t tc_tile_off(int r, int k) {
    const int blk = k >> 6, kk = k & 63;
    return (uint32_t)(blk * kTcBlockBytes + r * 128 + ((((kk >> 3) ^ (r & 7)) << 4) | ((kk & 7) << 1)));
}

// logistic_tc2_kernel.  The elementwise sigmoid / softplus work of the epilogue bounds this kernel, not the tensor pipe (a
// design with 8 epilogue warps that drained into global memory kept the tensor pipe 14 % busy, at 63 warp-instructions per
// (row, chain) element and 42 % of the stall samples on long-scoreboard waits: profiles/r2_tc_logistic_tc_ncu_summary.csv),
// so everything around the two GEMMs is shaped to keep the epilogue short:
//   * 16 epilogue warps (four per TMEM subpartition, 32 rows of the slab each): 4 warps per scheduler hide the TMEM-load and
//     MUFU latencies that 2 could not;
//   * the gradient partials stay in REGISTERS as fp64 (32 per thread) across the drains and are written once at the end
//     (adding every drain into global memory is 2 x 64 read-modify-writes per thread every 2 slabs = 2 GB of L2 traffic per
//     launch, the long-scoreboard stalls);
//   * y travels with the slab: the TMA producer copies the slab's 128 labels (fp32, 512 B) into the stage next to the X
//     pieces, so the element loop neither reads global memory nor converts bytes to floats;
//   * elementwise math on the MUFU units directly (ex2 / rcp / lg2 .approx.ftz): 12 instructions per element for
//     sigmoid + softplus + log-likelihood + residual; fp16 pieces of the residual are packed in place;
//   * rows past N need no masking: their X rows are zero, so eta = 0 exactly, the residual multiplies zero rows in GEMM 2, and
//     the log-likelihood they add (-softplus(0) each) is added back per slab.
// Accumulation order and drain period are dictated by the tensor cores' fp32 accumulate, which rounds toward zero: every
// tcgen05.mma into an accumulator of magnitude |D| loses ~2^-25 |D| one-sidedly (measured, round 2 call 3: 24 accumulate
// steps per slab -> 8e-7, 384 steps -> 7.9e-6 relative).  So (i) the small correction products hi*lo and lo*hi are issued
// FIRST, while the accumulator is still tiny, and hi*hi last: 8 full-magnitude steps per GEMM instead of 24; (ii) the
// gradient accumulator is drained into fp64 every kTcDrain = 2 slabs.
constexpr int kTc2EpiWarps = 16;
constexpr int kTc2EpiThreads = 32 * kTc2EpiWarps;
constexpr int kTc2Threads = 64 + kTc2EpiThreads;  // TMA producer, MMA issuer, 16 epilogue warps
constexpr uint32_t kTc2YBytes = kTcRows * sizeof(float);
constexpr size_t kTc2SmemBytes = 1024 /*align*/ + 2 * kTcPieceBytes /*beta hi, lo*/ + kTcStages * kTcStageBytes + 256 /*barriers*/ +
                                 kTcStages * kTc2YBytes /*labels*/;

__device__ __forceinline__ float tc_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float tc_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float tc_lg2(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
// 8 registers -> 8 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tc_st8(uint32_t taddr, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t a4, uint32_t a5,
                                       uint32_t a6, uint32_t a7) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(a0), "r"(a1),
                 "r"(a2), "r"(a3), "r"(a4), "r"(a5), "r"(a6), "r"(a7)
                 : "memory");
}

struct LogisticTc2Args {
    const float* y32;        // [n_slabs * 128] labels as fp32, zero padded
    long long N;             // true rows
    long long n_slabs;
    const double* Q;         // [C][ldq] beta per chain
    long long ldq;
    int C, K;
    double* Gpart;           // [gridDim.x][128 features][Cpad]  (feature-major)
    double* lpart;           // [gridDim.x][Cpad]
    int Cpad;
};

// 18 warps on 4 schedulers: one scheduler hosts 5 of them, and the register file is per scheduler (16 K entries), so the
// kernel gets 96 registers per thread, not 65536 / 576 = 113 (a 112-register build fails to launch: measured, call 11)
__global__ void __launch_bounds__(kTc2Threads, 1)
    logistic_tc2_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, const LogisticTc2Args A) {
    extern __shared__ char tc_smem_raw[];
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
    char* beta_s = base;                                   // [hi | lo] pieces, 32 KB each
    char* x_s = base + 2 * kTcPieceBytes;                  // stages x [X_hi | X_lo]
    uint64_t* bars = reinterpret_cast<uint64_t*>(x_s + kTcStages * kTcStageBytes);
    float* y_s = reinterpret_cast<float*>(reinterpret_cast<char*>(bars) + 256);  // stages x [128] labels
    uint64_t* x_full = bars;          // [2] TMA -> MMA (and the epilogue: y)
    uint64_t* x_empty = bars + 2;     // [2] MMA (GEMM 2 done) -> TMA
    uint64_t* eta_full = bars + 4;    // [2] MMA (GEMM 1 done) -> epilogue
    uint64_t* eta_empty = bars + 6;   // [2] epilogue (D1 read) -> MMA
    uint64_t* r_full = bars + 8;      // epilogue (r written) -> MMA
    uint64_t* r_empty = bars + 9;     // MMA (GEMM 2 done: r and the X stage are free) -> epilogue
    uint64_t* g_full = bars + 10;     // MMA (drain point reached: D2 holds kTcDrain slabs) -> epilogue
    uint64_t* g_empty = bars + 11;    // epilogue (D2 drained) -> MMA
    __shared__ uint32_t tmem_base_s;
    __shared__ double lp_q_s[3][kTcChains];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c_base = blockIdx.y * kTcChains;
    const long long my_slabs = (A.n_slabs > blockIdx.x) ? (A.n_slabs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&x_full[i], 1);
            mbar_init(&x_empty[i], 1);
            mbar_init(&eta_full[i], 1);
            mbar_init(&eta_empty[i], kTc2EpiThreads);
        }
        mbar_init(r_full, kTc2EpiThreads);
        mbar_init(r_empty, 1);
        mbar_init(g_full, 1);
        mbar_init(g_empty, kTc2EpiThreads);
    }
    if (warp == 1) {
        const uint32_t ncols = 512;
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int e = tid; e < kTcChains * kTcK; e += kTc2Threads) {
        const int c = e >> 7, k = e & 127;
        const double v = (c_base + c < A.C && k < A.K) ? A.Q[(long long)(c_base + c) * A.ldq + k] : 0.0;
        const __half hi = __double2half(v);
        const __half lo = __double2half(v - (double)__half2float(hi));
        const uint32_t off = tc_tile_off(c, k);
        *reinterpret_cast<__half*>(beta_s + off) = hi;
        *reinterpret_cast<__half*>(beta_s + kTcPieceBytes + off) = lo;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const uint32_t tD1[2] = {tmem + 0, tmem + 128}, tD2 = tmem + 256, tRh = tmem + 384, tRl = tmem + 448;

    if (warp == 0) {
        // ===== TMA producer: X_hi, X_lo (two 64-column boxes each) and the slab's labels =====
        if (lane == 0) {
            for (long long s = 0; s < my_slabs; ++s) {
                const int st = (int)(s % kTcStages);
                if (s >= kTcStages) tc_mbar_wait(&x_empty[st], (uint32_t)(((s / kTcStages) - 1) & 1));
                const long long slab = blockIdx.x + s * gridDim.x;
                const int row0 = (int)(slab * kTcRows);
                char* dst = x_s + st * kTcStageBytes;
                mbar_expect_tx(&x_full[st], kTcStageBytes + kTc2YBytes);
                tc_tma_load_2d(dst, &map_hi, 0, row0, &x_full[st]);
                tc_tma_load_2d(dst + kTcBlockBytes, &map_hi, 64, row0, &x_full[st]);
                tc_tma_load_2d(dst + kTcPieceBytes, &map_lo, 0, row0, &x_full[st]);
                tc_tma_load_2d(dst + kTcPieceBytes + kTcBlockBytes, &map_lo, 64, row0, &x_full[st]);
                tma_bulk_g2s(y_s + st * kTcRows, A.y32 + (long long)row0, kTc2YBytes, &x_full[st]);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one lane) =====
        if (lane == 0) {
            const uint32_t beta_a = smem_u32(beta_s);
            auto gemm1 = [&](long long s) {
                const int st = (int)(s % kTcStages), b = (int)(s & 1);
                tc_mbar_wait(&x_full[st], (uint32_t)((s / kTcStages) & 1));
                if (s >= 2) tc_mbar_wait(&eta_empty[b], (uint32_t)(((s >> 1) - 1) & 1));
                tc_fence_after();
                const uint32_t xa = smem_u32(x_s + st * kTcStageBytes);
                uint32_t acc = 0;
#pragma unroll
                for (int prod = 0; prod < 3; ++prod) {  // hi*lo, lo*hi, hi*hi
                    const uint32_t a0 = beta_a + (prod == 1 ? kTcPieceBytes : 0);
                    const uint32_t b0 = xa + (prod == 0 ? kTcPieceBytes : 0);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint32_t o = (uint32_t)((ks >> 2) * kTcBlockBytes + (ks & 3) * 32);
                        tc_mma_ss(tD1[b], tc_desc(a0 + o, 16, 1024), tc_desc(b0 + o, 16, 1024), kTcIdesc, acc);
                        acc = 1;
                    }
                }
                tc_commit(&eta_full[b]);
            };
            if (my_slabs > 0) gemm1(0);
            for (long long s = 0; s < my_slabs; ++s) {
                if (s + 1 < my_slabs) gemm1(s + 1);
                tc_mbar_wait(r_full, (uint32_t)(s & 1));
                const bool first = (s % kTcDrain) == 0;
                if (first && s > 0) tc_mbar_wait(g_empty, (uint32_t)(((s / kTcDrain) - 1) & 1));
                tc_fence_after();
                const int st = (int)(s % kTcStages);
                const uint32_t xa = smem_u32(x_s + st * kTcStageBytes);
                uint32_t acc = first ? 0u : 1u;
#pragma unroll
                for (int prod = 0; prod < 3; ++prod) {  // r_hi X_lo, r_lo X_hi, r_hi X_hi
                    const uint32_t ta = (prod == 1) ? tRl : tRh;
                    const uint32_t b0 = xa + (prod == 0 ? kTcPieceBytes : 0);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        tc_mma_ts(tD2, ta + ks * 8, tc_desc(b0 + ks * 2048, kTcBlockBytes, 1024), kTcIdescBmn, acc);
                        acc = 1;
                    }
                }
                tc_commit(&x_empty[st]);
                tc_commit(r_empty);
                if ((s + 1) % kTcDrain == 0 || s + 1 == my_slabs) tc_commit(g_full);
            }
        }
    } else {
        // ===== epilogue: 16 warps; TMEM lane = chain (subpartition = warp % 4); the four warps of a subpartition take a
        //       quarter of the slab's rows (32) and a quarter of the gradient's columns (32 features) each =====
        const int sub = warp & 3, quarter = (warp - 2) >> 2;
        const int c = sub * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(sub * 32) << 16;
        double lp = 0.0;
        double gacc[32];  // this thread's gradient partials: features quarter*32 .. +31 of chain c, over all slabs of the CTA
#pragma unroll
        for (int k = 0; k < 32; ++k) gacc[k] = 0.0;
        long long n_drains = 0;
        auto drain = [&]() {  // fp32 gradient accumulator (kTcDrain slabs) -> the fp64 registers
            tc_mbar_wait(g_full, (uint32_t)(n_drains & 1));
            tc_fence_after();
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                uint32_t v[16];
                tc_ld16(tD2 + lane_addr + quarter * 32 + j * 16, v);
                tc_wait_ld();
#pragma unroll
                for (int k = 0; k < 16; ++k) gacc[j * 16 + k] += (double)__uint_as_float(v[k]);
            }
            ++n_drains;
            tc_fence_before();
            tc_mbar_arrive(g_empty);
        };
        // softplus(0) as the element formula computes it: what every padded row (eta = 0 exactly) subtracts from lp
        const float sp0 = tc_lg2(2.0f) * 0.69314718055994530942f;
        for (long long s = 0; s < my_slabs; ++s) {
            const int b = (int)(s & 1), st = (int)(s % kTcStages);
            const long long row0 = (blockIdx.x + s * gridDim.x) * kTcRows + quarter * 32;
            tc_mbar_wait(&eta_full[b], (uint32_t)((s >> 1) & 1));
            // the labels arrived with the X pieces of this stage (same mbarrier; completed before GEMM 1 was issued)
            tc_mbar_wait(&x_full[st], (uint32_t)((s / kTcStages) & 1));
            tc_fence_after();
            const float4* yq = reinterpret_cast<const float4*>(y_s + st * kTcRows + quarter * 32);
            float lp_s = 0.f;
#pragma unroll
            for (int j = 0; j < 2; ++j) {  // 16 rows of the slab at a time
                uint32_t v[16];
                tc_ld16(tD1[b] + lane_addr + quarter * 32 + j * 16, v);
                tc_wait_ld();
                if (j == 1) {  // this thread's share of D1[b] has been read: GEMM 1 of slab s + 2 may overwrite it
                    tc_fence_before();
                    tc_mbar_arrive(&eta_empty[b]);
                }
#pragma unroll
                for (int i4 = 0; i4 < 4; ++i4) {
                    const float4 y4 = yq[j * 4 + i4];  // same address in every lane: one broadcast LDS.128 per 4 rows
                    const float yv[4] = {y4.x, y4.y, y4.z, y4.w};
                    float rr[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float x = __uint_as_float(v[4 * i4 + u]);
                        const float t = tc_ex2(-1.4426950408889634f * fabsf(x));   // e^-|x|
                        const float w = 1.f + t;
                        const float inv = tc_rcp(w);
                        const float sg = x >= 0.f ? inv : t * inv;                  // sigmoid(x)
                        const float sp = fmaf(tc_lg2(w), 0.69314718055994530942f, fmaxf(x, 0.f));  // softplus(x)
                        lp_s += fmaf(yv[u], x, -sp);
                        rr[u] = yv[u] - sg;
                    }
#pragma unroll
                    for (int u = 0; u < 4; u += 2) {  // fp16 pieces of two residuals, packed in place of their eta values
                        const __half2 h = __floats2half2_rn(rr[u], rr[u + 1]);
                        const float2 hf = __half22float2(h);
                        const __half2 l = __floats2half2_rn(rr[u] - hf.x, rr[u + 1] - hf.y);
                        v[4 * i4 + u] = *reinterpret_cast<const uint32_t*>(&h);
                        v[4 * i4 + u + 1] = *reinterpret_cast<const uint32_t*>(&l);
                    }
                }
                // GEMM 2 of the previous slab (it ran under the arithmetic above) frees r; every kTcDrain slabs its accumulator
                // goes to the fp64 registers first
                const bool drain_now = (j == 0 && s > 0 && s % kTcDrain == 0);
                if (j == 0 && s > 0) {
                    if (drain_now) tc_mbar_wait(g_full, (uint32_t)(n_drains & 1));  // GEMM 2 of slab s-1 done: r free, D2 complete
                    else tc_mbar_wait(r_empty, (uint32_t)((s - 1) & 1));
                    tc_fence_after();
                }
                // 16 rows -> 8 packed columns of r_hi and of r_lo
                tc_st8(tRh + lane_addr + quarter * 16 + j * 8, v[0], v[2], v[4], v[6], v[8], v[10], v[12], v[14]);
                tc_st8(tRl + lane_addr + quarter * 16 + j * 8, v[1], v[3], v[5], v[7], v[9], v[11], v[13], v[15]);
                if (drain_now) {
                    // the drain: both TMEM loads first, D2 handed back to the MMA issuer as soon as they have landed; the fp64
                    // conversions and sums run afterwards, off the GEMM 2 -> GEMM 2 critical path
                    uint32_t d0[16], d1[16];
                    tc_ld16(tD2 + lane_addr + quarter * 32, d0);
                    tc_ld16(tD2 + lane_addr + quarter * 32 + 16, d1);
                    tc_wait_ld();
                    ++n_drains;
                    tc_fence_before();
                    tc_mbar_arrive(g_empty);
#pragma unroll
                    for (int k = 0; k < 16; ++k) gacc[k] += (double)__uint_as_float(d0[k]);
#pragma unroll
                    for (int k = 0; k < 16; ++k) gacc[16 + k] += (double)__uint_as_float(d1[k]);
                }
            }
            tc_wait_st();
            tc_fence_before();
            tc_mbar_arrive(r_full);
            const long long over = row0 + 32 - A.N;  // padded rows of this quarter (the last slab only)
            if (over > 0) lp_s += (float)(over < 32 ? over : 32) * sp0;
            lp += (double)lp_s;
        }
        if (my_slabs > 0) drain();
        // the CTA's fp64 partial gradient, FEATURE-major [128 k][Cpad chains]: for a fixed k the 32 lanes of a warp write 32
        // consecutive chains (coalesced), once
        double* gp = A.Gpart + ((long long)blockIdx.x * kTcK + quarter * 32) * A.Cpad + c_base + c;
#pragma unroll
        for (int k = 0; k < 32; ++k) gp[(long long)k * A.Cpad] = gacc[k];
        if (quarter > 0) lp_q_s[quarter - 1][c] = lp;
        __syncwarp();
        asm volatile("bar.sync 1, %0;" ::"r"(kTc2EpiThreads) : "memory");  // the 16 epilogue warps only
        if (quarter == 0) A.lpart[(long long)blockIdx.x * A.Cpad + c_base + c] = ((lp + lp_q_s[0][c]) + lp_q_s[1][c]) + lp_q_s[2][c];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        const uint32_t ncols = 512;
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(ncols) : "memory");
    }
}

// labels as fp32, zero padded to whole slabs (logistic_tc2_kernel copies them into shared memory with the slab)
__global__ void __launch_bounds__(256) logistic_tc_y_kernel(const uint8_t* __restrict__ y, long long N, float* __restrict__ y32,
                                                            long long rows_pad) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < rows_pad) y32[e] = (e < N) ? (float)y[e] : 0.f;
}

// fp64 design matrix [N][K] (row stride ldx) -> fp16 pieces [n_slabs * 128][128], zero padded
__global__ void __launch_bounds__(256) logistic_tc_split_kernel(const double* __restrict__ X, long long N, int K, long long ldx,
                                                                __half* __restrict__ Xh, __half* __restrict__ Xl, long long rows_pad) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows_pad * kTcK) return;
    const long long r = e >> 7;
    const int k = (int)(e & 127);
    const double v = (r < N && k < K) ? X[r * ldx + k] : 0.0;
    const __half hi = __double2half(v);
    Xh[e] = hi;
    Xl[e] = __double2half(v - (double)__half2float(hi));
}

}  // namespace b200
