// Dense fp64 contractions of the GEMM-shaped models, hand-written on the fp64 tensor-core path
// (mma.sync.aligned.m8n8k4.f64, SASS DMMA.8x8x4; tcgen05 has no fp64 kind).  Measured on B200 (scripts/mb):
// DMMA sustains 37.0 TFLOP/s = the DFMA peak (the fp64 pipe is the roof either way), but needs 1/8 of the issue
// slots and no register-operand bandwidth, which leaves room for the shared-memory fragment loads.
//
//   gemm_nt_dmma_kernel     D[C][Nout] = alpha * Q[C][K] . M[Nout][K]^T        (config 5: grad = -P q, w = Sigma g,
//                                                                              p0 = L^-T z, v0 = L z; chains are rows)
//   logistic_fused_kernel   eta = X beta, r = y - sigmoid(eta), G = X^T r, logp = sum(y eta - softplus(eta))
//                           in ONE pass over the design matrix (config 3); eta/r never leave registers
//
// Fragment layout of m8n8k4 (g = lane/4, t = lane%4):  A[m=g][k=t]  B[k=t][n=g]  C[m=g][n=2t,2t+1].
// Both kernels contract "row-major against row-major" (D[c][j] = sum_k Q[c][k] M[j][k]), so A and B fragments are
// the same access pattern: element [row0+g][k0+t] of a shared-memory tile whose row stride is = 4 (mod 16) doubles,
// which makes every 64-bit fragment load bank-conflict free (a half-warp touches 16 distinct 8-byte bank pairs).
#pragma once
#include "common.cuh"

namespace b200 {

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src, bool valid) {
    const int sz = valid ? 16 : 0;  // src-size 0: the 16 bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ------------------------------------------------------------------------------------------------------------------
// D[c][j] = alpha * sum_k Q[c][k] * M[j][k]     c < C, j < Nout, k < K (K = padded inner size, multiple of 4;
// rows of Q and M are ldq / ldm doubles apart, multiples of 2 so 16-byte cp.async chunks stay aligned).
// CTA = WM warps; warp w owns chains [16 w, 16 w + 16) of the CTA's 16*WM-chain block and ALL 8*NB outputs of the
// CTA's output tile: 2*NB accumulator tiles, (2 + NB) fragment loads per 2*NB DMMAs.  K is streamed in chunks of
// 32 through an NST-stage cp.async pipeline.  grid = (ceil(Nout / 8NB), ceil(C / 16WM)).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kGemmKC = 32;             // k-chunk per pipeline stage
constexpr int kGemmLd = kGemmKC + 4;    // padded shared-memory row stride (doubles), = 4 mod 16

template <int WM, int NB>
__host__ __device__ constexpr size_t gemm_stage_doubles() { return (size_t)(16 * WM + 8 * NB) * kGemmLd; }

template <int WM, int NB, int NST>
__global__ void __launch_bounds__(32 * WM, 1)
    gemm_nt_dmma_kernel(const double* __restrict__ Q, long long ldq, int C, const double* __restrict__ M, long long ldm,
                        int Nout, int K, double alpha, double* __restrict__ D, long long ldd) {
    extern __shared__ __align__(16) char smem_raw[];
    double* sm = reinterpret_cast<double*>(smem_raw);
    constexpr int TM = 16 * WM, TN = 8 * NB, NT = 32 * WM;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int c_base = blockIdx.y * TM, j_base = blockIdx.x * TN;
    const int n_chunks = (K + kGemmKC - 1) / kGemmKC;

    auto load_stage = [&](int chunk, int stage) {
        double* qs = sm + (size_t)stage * gemm_stage_doubles<WM, NB>();
        double* ms = qs + TM * kGemmLd;
        const int k0 = chunk * kGemmKC;
        // 16 chunks of 16 bytes per row
        for (int e = tid; e < TM * 16; e += NT) {
            const int r = e >> 4, kk = (e & 15) * 2;
            const bool ok = (c_base + r < C) && (k0 + kk < K);
            cp_async16(qs + r * kGemmLd + kk, ok ? Q + (long long)(c_base + r) * ldq + k0 + kk : Q, ok);
        }
        for (int e = tid; e < TN * 16; e += NT) {
            const int r = e >> 4, kk = (e & 15) * 2;
            const bool ok = (j_base + r < Nout) && (k0 + kk < K);
            cp_async16(ms + r * kGemmLd + kk, ok ? M + (long long)(j_base + r) * ldm + k0 + kk : M, ok);
        }
    };

    double acc[2][NB][2];
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;

#pragma unroll
    for (int s = 0; s < NST - 1; ++s) {
        if (s < n_chunks) load_stage(s, s);
        cp_async_commit();
    }
    for (int ch = 0; ch < n_chunks; ++ch) {
        cp_async_wait<NST - 2>();
        __syncthreads();  // chunk `ch` has landed for every thread; everyone is done with the stage refilled below
        if (ch + NST - 1 < n_chunks) load_stage(ch + NST - 1, (ch + NST - 1) % NST);
        cp_async_commit();
        const double* qs = sm + (size_t)(ch % NST) * gemm_stage_doubles<WM, NB>() + (warp * 16 + g) * kGemmLd + t;
        const double* ms = sm + (size_t)(ch % NST) * gemm_stage_doubles<WM, NB>() + TM * kGemmLd + g * kGemmLd + t;
#pragma unroll
        for (int ks = 0; ks < kGemmKC; ks += 4) {
            const double a0 = qs[ks], a1 = qs[8 * kGemmLd + ks];
            double b[NB];
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) b[nb] = ms[nb * 8 * kGemmLd + ks];
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
                dmma884(acc[0][nb][0], acc[0][nb][1], a0, b[nb]);
                dmma884(acc[1][nb][0], acc[1][nb][1], a1, b[nb]);
            }
        }
    }
    cp_async_wait<0>();
#pragma unroll
    for (int mb = 0; mb < 2; ++mb) {
        const int c = c_base + warp * 16 + mb * 8 + g;
        if (c < C) {
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
                const int j = j_base + nb * 8 + 2 * t;
                double* d = D + (long long)c * ldd + j;
                if (j + 1 < Nout) *reinterpret_cast<double2*>(d) = make_double2(alpha * acc[mb][nb][0], alpha * acc[mb][nb][1]);
                else if (j < Nout) d[0] = alpha * acc[mb][nb][0];
            }
        }
    }
}

// logp[c] = logp_const + 0.5 * q_c . g_c   (MvNormal: g = -P q, so -0.5 q^T P q = 0.5 q.g); one warp per chain
__global__ void __launch_bounds__(128) half_dot_logp_kernel(const double* __restrict__ Q, const double* __restrict__ G,
                                                            long long ld, int n, int C, double logp_const,
                                                            double* __restrict__ logp) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= C) return;
    double s = 0.0;
    for (int i = lane; i < n; i += 32) s = fma(Q[(long long)c * ld + i], G[(long long)c * ld + i], s);
    s = warp_sum(s);
    if (lane == 0) logp[c] = logp_const + 0.5 * s;
}

// ------------------------------------------------------------------------------------------------------------------
// Logistic GLM (BASELINE config 3): beta ~ Normal(0,1)^K, y_i ~ Bernoulli(logit_p = x_i . beta)
//   logp = sum_i [y_i eta_i - softplus(eta_i)] + sum_k Normal(beta_k | 0, 1)          (discrete.py:351-367 with the
//   grad = X^T (y - sigmoid(eta)) - beta                                              stabilised softplus forms)
// One pass over X per batch of chains.  CTA = 8 warps = 128 chains (warp w: chains 16w..16w+15), looping over slabs of
// 32 rows of X (bulk-TMA, one 8*KP-byte row per copy into padded shared rows, double buffered):
//   GEMM 1   etaT[c][i]  = sum_k Q[c][k] X[i][k]      2 x 4 accumulator tiles per warp (16 chains x 32 rows)
//   epilogue r = y - sigmoid(eta), logp += y eta - softplus(eta)     in the accumulator registers
//   GEMM 2   G[c][k]    += sum_i r[c][i] X[i][k]      2 x KB accumulator tiles per warp, persistent over the slabs
// The accumulator layout of GEMM 1 (lane holds columns 2t, 2t+1) IS an A-fragment of GEMM 2 once the contraction
// index is enumerated as i = 2t + s for k-step s, so r never goes through shared memory.  Rows inside an 8-row group
// are permuted by pi(n) = n ^ ((n >> 2) & 1) so that both GEMMs read X fragments without bank conflicts.
// Partial results per row-CTA are reduced in a fixed order by logistic_finish_kernel (deterministic, no atomics).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kLogiRows = 32;    // rows of X per slab
constexpr int kLogiChains = 128; // chains per CTA

template <int KB>
__host__ __device__ constexpr size_t logistic_smem_bytes() {
    return ((size_t)kLogiChains * (8 * KB + 4) + 2 * (size_t)kLogiRows * (8 * KB + 4)) * sizeof(double) + 64;
}

// 8-chain accumulator blocks per warp: 1 -> 16 warps x 8 chains per CTA (126 regs, 4 warps per scheduler: 10.8 ms per
// 512-chain batch) is faster than 2 -> 8 warps x 16 chains (212 regs, 12.4 ms)
constexpr int kLogiMB = 1;
template <int KB, int MB = kLogiMB>
__global__ void __launch_bounds__(32 * (kLogiChains / (8 * MB)), 1)
    logistic_fused_kernel(const double* __restrict__ X /*[Npad][8KB]*/, const uint8_t* __restrict__ y, long long N,
                          const double* __restrict__ Q, long long ldq, int C, int K,
                          double* __restrict__ Gpart /*[gridDim.x][Cpad][8KB]*/, double* __restrict__ lpart /*[gridDim.x][Cpad]*/,
                          int Cpad) {
    constexpr int KP = 8 * KB, LD = KP + 4, NT = 32 * (kLogiChains / (8 * MB));
    extern __shared__ __align__(16) char smem_raw[];
    double* Qs = reinterpret_cast<double*>(smem_raw);
    double* Xs = Qs + kLogiChains * LD;                       // 2 slabs
    uint64_t* bars = reinterpret_cast<uint64_t*>(Xs + 2 * kLogiRows * LD);  // full[2]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int c_base = blockIdx.y * kLogiChains;
    const long long n_slabs = (N + kLogiRows - 1) / kLogiRows;

    // Q tile (zero rows for chains >= C, zero columns for k >= K)
    for (int e = tid; e < kLogiChains * KP; e += NT) {
        const int r = e / KP, k = e % KP;
        Qs[r * LD + k] = (c_base + r < C && k < K) ? Q[(long long)(c_base + r) * ldq + k] : 0.0;
    }
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
    }
    __syncthreads();
    auto issue = [&](long long slab, int buf) {  // thread 0: one bulk copy per row (rows past the padded end do not exist:
        const long long r0 = slab * kLogiRows;   // X is allocated with Npad = n_slabs * 32 rows, zero filled)
        mbar_expect_tx(&bars[buf], kLogiRows * KP * 8);
        for (int r = 0; r < kLogiRows; ++r) tma_bulk_g2s(Xs + (buf * kLogiRows + r) * LD, X + (r0 + r) * KP, KP * 8, &bars[buf]);
    };
    long long slab = blockIdx.x;
    if (tid == 0 && slab < n_slabs) issue(slab, 0);

    double G[MB][KB][2];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb)
#pragma unroll
        for (int nb = 0; nb < KB; ++nb) G[mb][nb][0] = G[mb][nb][1] = 0.0;
    double lp[MB];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb) lp[mb] = 0.0;
    const double* qa = Qs + (warp * 8 * MB + g) * LD + t;
    const int pg = g ^ ((g >> 2) & 1);  // pi(g)

    uint32_t phase[2] = {0, 0};
    for (int it = 0; slab < n_slabs; slab += gridDim.x, ++it) {
        const int buf = it & 1;
        if (tid == 0 && slab + gridDim.x < n_slabs) issue(slab + gridDim.x, buf ^ 1);  // buffer buf^1 was released by the barrier below
        mbar_wait(&bars[buf], phase[buf]);
        phase[buf] ^= 1;
        const double* xs = Xs + buf * kLogiRows * LD;
        // ---- GEMM 1: etaT[16 chains][32 rows]; B fragment = X[8 nb + pi(g)][k0 + t]
        double E[MB][4][2];
#pragma unroll
        for (int mb = 0; mb < MB; ++mb)
#pragma unroll
            for (int nb = 0; nb < 4; ++nb) E[mb][nb][0] = E[mb][nb][1] = 0.0;
        const double* xb = xs + pg * LD + t;
#pragma unroll 4
        for (int ks = 0; ks < KP; ks += 4) {
            double a[MB];
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) a[mb] = qa[mb * 8 * LD + ks];
#pragma unroll
            for (int nb = 0; nb < 4; ++nb) {
                const double b = xb[nb * 8 * LD + ks];
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) dmma884(E[mb][nb][0], E[mb][nb][1], a[mb], b);
            }
        }
        // ---- epilogue: accumulator column n = 2t + s is row  8 nb + pi(2t + s)  of the slab
        const long long r0 = slab * kLogiRows;
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int nn = 2 * t + s;
                const long long row = r0 + nb * 8 + (nn ^ ((nn >> 2) & 1));
                const bool live = row < N;
                const double yi = live ? (double)y[row] : 0.0;
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) {
                    const double x = E[mb][nb][s];
                    const double ex = exp(-fabs(x));
                    const double rr = 1.0 / (1.0 + ex);
                    const double sg = x >= 0 ? rr : ex * rr;                 // sigmoid(x)
                    const double sp = fmax(x, 0.0) + log1p(ex);             // softplus(x); log(1 + e) instead: no gain measured (r2)
                    lp[mb] += live ? fma(yi, x, -sp) : 0.0;
                    E[mb][nb][s] = live ? yi - sg : 0.0;
                }
            }
        }
        // ---- GEMM 2: G[16 chains][KP] += r[c][i] X[i][k]; k-step (nb, s) contracts rows 8 nb + pi(2t + s), t = 0..3
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int nn = 2 * t + s;
                const double* xr = xs + (nb * 8 + (nn ^ ((nn >> 2) & 1))) * LD + g;
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    const double b = xr[kb * 8];
#pragma unroll
                    for (int mb = 0; mb < MB; ++mb) dmma884(G[mb][kb][0], G[mb][kb][1], E[mb][nb][s], b);
                }
            }
        }
        __syncthreads();  // all warps are done with slab buffer `buf`: it may be refilled at the top of the next turn
    }
    // ---- partial results of this row-CTA
#pragma unroll
    for (int mb = 0; mb < MB; ++mb) {
        const int c = c_base + warp * 8 * MB + mb * 8 + g;
        double l = lp[mb];
        l += __shfl_xor_sync(B200_FULL_MASK, l, 1);
        l += __shfl_xor_sync(B200_FULL_MASK, l, 2);
        if (c < Cpad) {
            double* gp = Gpart + ((long long)blockIdx.x * Cpad + c) * KP;
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
                *reinterpret_cast<double2*>(gp + kb * 8 + 2 * t) = make_double2(G[mb][kb][0], G[mb][kb][1]);
            if (t == 0) lpart[(long long)blockIdx.x * Cpad + c] = l;
        }
    }
}

// G[c][k] = sum_parts Gpart[p][c][k] - beta ; logp[c] = sum_parts lpart[p][c] - 0.5 |beta|^2 - K/2 log 2pi   (fixed order)
__global__ void __launch_bounds__(128) logistic_finish_kernel(const double* __restrict__ Q, long long ldq, double* __restrict__ G,
                                                              long long ldg, int K, int KP, int C, int Cpad,
                                                              const double* __restrict__ Gpart, const double* __restrict__ lpart,
                                                              int nparts, double* __restrict__ logp, int feature_major = 0) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= C) return;
    double s = 0.0;
    for (int k = lane; k < K; k += 32) {
        double a = 0.0;
        for (int p = 0; p < nparts; ++p)
            a += feature_major ? Gpart[((long long)p * KP + k) * Cpad + c] : Gpart[((long long)p * Cpad + c) * KP + k];
        const double b = Q[(long long)c * ldq + k];
        G[(long long)c * ldg + k] = a - b;
        s = fma(b, b, s);
    }
    s = warp_sum(s);
    if (lane == 0) {
        double l = 0.0;
        for (int p = 0; p < nparts; ++p) l += lpart[(long long)p * Cpad + c];
        logp[c] = l - 0.5 * s - K * B200_HALF_LOG_2PI;
    }
}

// The same reduction for FEATURE-major partials Gpart[p][k][c] (the tensor-core kernels' layout: chains contiguous).  The
// kernel above walks them with lane = feature, i.e. with a stride of Cpad doubles (measured: 74 us per 512-chain batch, 16 % of
// the tensor-core lock-step loop, profiles/r2l_launches_logistic_tc_summary.csv).  Here a CTA owns a 32-chain x 16-feature tile:
// lane = chain while summing (coalesced, 4 independent partial loads in flight per thread, the same fixed order over p as
// above, so the same bits), a shared-memory transpose for the row-major gradient, and the blockIdx.y == 0 CTAs also produce
// logp with the arithmetic of the kernel above.
__global__ void __launch_bounds__(256) logistic_finish_fm_kernel(const double* __restrict__ Q, long long ldq, double* __restrict__ G,
                                                                 long long ldg, int K, int KP, int C, int Cpad,
                                                                 const double* __restrict__ Gpart, const double* __restrict__ lpart,
                                                                 int nparts, double* __restrict__ logp) {
    __shared__ double tile[16][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;  // 8 warps: features 2 w, 2 w + 1 of the tile
    const int c0 = blockIdx.x * 32, k0 = blockIdx.y * 16;
    const int c = c0 + lane;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int k = k0 + 2 * w + u;
        double a = 0.0;
        if (k < KP && c < Cpad) {
            const double* src = Gpart + (long long)k * Cpad + c;
            const long long step = (long long)KP * Cpad;
            int p = 0;
            for (; p + 4 <= nparts; p += 4) {
                const double x0 = src[(long long)p * step], x1 = src[(long long)(p + 1) * step];
                const double x2 = src[(long long)(p + 2) * step], x3 = src[(long long)(p + 3) * step];
                a += x0; a += x1; a += x2; a += x3;
            }
            for (; p < nparts; ++p) a += src[(long long)p * step];
        }
        tile[2 * w + u][lane] = a;
    }
    __syncthreads();
    // row-major gradient: thread (cc, kk) of the tile, 16 consecutive features of one chain per half-warp
    for (int e = threadIdx.x; e < 32 * 16; e += 256) {
        const int cc = e >> 4, kk = e & 15;
        const int ch = c0 + cc, k = k0 + kk;
        if (ch < C && k < K) G[(long long)ch * ldg + k] = tile[kk][cc] - Q[(long long)ch * ldq + k];
    }
    if (blockIdx.y == 0) {  // logp of the tile's 32 chains: warp w takes chains w, w + 8, ...
        for (int cc = w; cc < 32; cc += 8) {
            const int ch = c0 + cc;
            if (ch >= C) continue;
            double s = 0.0;
            for (int k = lane; k < K; k += 32) {
                const double b = Q[(long long)ch * ldq + k];
                s = fma(b, b, s);
            }
            s = warp_sum(s);
            if (lane == 0) {
                double l = 0.0;
                for (int p = 0; p < nparts; ++p) l += lpart[(long long)p * Cpad + ch];
                logp[ch] = l - 0.5 * s - K * B200_HALF_LOG_2PI;
            }
        }
    }
}

}  // namespace b200
