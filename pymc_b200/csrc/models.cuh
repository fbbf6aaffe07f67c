// Hand-written fused log-density + reverse-mode gradient device functions, one per model kind.
//
// Each `*Model::eval` replaces ONE call of the compiled PyTensor function
//     ValueGradFunction._pytensor_function(q) -> (logp, dlogp)
// (built at pymc/model/core.py:232-267, called at hmc/integration.py:52,70,129) for a chain owned by a
// WARP: q lives in the warp's shared-memory slice `q_s` (padded to NP = 32*NPL, pad = 0), the gradient
// is written to `g_s`, and logp is returned warp-uniform (xor-butterfly reductions).
// The math restates the reference densities (cited per model) with the gradients of SURVEY.md
// Appendix C; bad parameters cannot occur because scale parameters are exp() of unconstrained values.
#pragma once
#include "common.cuh"

namespace b200 {

// ------------------------------------------------------------------------------------------------
// x ~ Normal(0,1)^n  (test model; Normal.logp distributions/continuous.py:526-527)
// ------------------------------------------------------------------------------------------------
struct StdNormalModel {
    struct Params {
        int n;
    };
    __host__ __device__ static size_t shared_bytes(const Params&) { return 0; }
    __device__ static void stage(const Params&, char*, uint64_t*) {}
    template <int NPL, int W, bool SMALL = false>
    __device__ static double eval(const Params& P, const char*, const double* q_s, double* g_s, int tid, double* red) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = tid + 32 * W * k;
            const double x = q_s[i];
            s = fma(x, x, s);
            g_s[i] = -x;
        }
        s = team_sum<W>(s, tid, red);
        return -0.5 * s - P.n * B200_HALF_LOG_2PI;
    }
};

// ------------------------------------------------------------------------------------------------
// Eight Schools, non-centred (BASELINE config 1).  q = [mu, log tau, theta_t[J]]
//   mu~Normal(0,5); tau~HalfCauchy(5) (log transform); theta_t~Normal(0,1); y_j~Normal(mu+tau*theta_t_j, sigma_j)
// Densities: Normal continuous.py:526-527; HalfCauchy :2383-2385 (+Cauchy :2287-2288); log transform
// + Jacobian logprob/transforms.py:880-891.  Gradient: SURVEY Appendix C-1.
// ------------------------------------------------------------------------------------------------
struct EightSchoolsModel {
    struct Params {
        const double* y;       // [J]
        const double* inv_s2;  // [J] 1/sigma^2
        const double* log_s;   // [J] log sigma
        int J;
    };
    __host__ __device__ static size_t shared_bytes(const Params&) { return 0; }
    __device__ static void stage(const Params&, char*, uint64_t*) {}
    template <int NPL, int W, bool SMALL = false>
    __device__ static double eval(const Params& P, const char*, const double* q_s, double* g_s, int lane, double*) {
        static_assert(W == 1, "EightSchoolsModel is a chain-per-warp model");
        const double mu = q_s[0], ltau = q_s[1];
        const double tau = exp(ltau);
        double acc[4] = {0.0, 0.0, 0.0, 0.0};  // sum r, sum r*tt, sum tt^2, sum loglik (w/o const)
        for (int j = lane; j < P.J; j += 32) {
            const double tt = q_s[2 + j];
            const double th = fma(tau, tt, mu);
            const double d = P.y[j] - th;
            const double r = d * P.inv_s2[j];
            acc[0] += r;
            acc[1] = fma(r, tt, acc[1]);
            acc[2] = fma(tt, tt, acc[2]);
            acc[3] += -0.5 * d * r - P.log_s[j];
            g_s[2 + j] = fma(tau, r, -tt);
        }
        warp_sum_n(acc);
        double hc, dhc;
        halfcauchy_log(ltau, tau, 5.0, 1.6094379124341002818 /* log 5 */, hc, dhc);
        if (lane == 0) {
            g_s[0] = -mu * (1.0 / 25.0) + acc[0];
            g_s[1] = fma(tau, acc[1], dhc);
        }
        const double z = mu * 0.2;
        const double lp_mu = -0.5 * z * z - B200_HALF_LOG_2PI - 1.6094379124341002818;
        return lp_mu + hc + (-0.5 * acc[2] - P.J * B200_HALF_LOG_2PI) + (acc[3] - P.J * B200_HALF_LOG_2PI);
    }
};

// ------------------------------------------------------------------------------------------------
// Radon hierarchical regression (BASELINE config 2; model benchmarks/benchmarks/benchmarks.py:34-45)
//   q = [mu_a, log sigma_a, mu_b, log sigma_b, a[J], b[J], log eps]
//   alpha_c = mu_a + sigma_a a_c ; beta_c = mu_b + sigma_b b_c ; y_i ~ Normal(alpha_c(i) + beta_c(i) x_i, eps)
//   mu_* ~ Normal(0, 100**2) ; sigma_*, eps ~ HalfCauchy(5) ; a, b ~ Normal(0,1)
// Gradient: SURVEY Appendix C-2.  The per-county segmented sums G_alpha, G_beta are the per-chain
// reduction.  At model-create time counties are sorted by size and dealt to the 32 lanes row by row
// (row j = the j-th county of every lane; sorting makes the sizes within a row nearly equal), and each
// row is padded to its longest county, so all lanes reach the end of their county at the SAME inner
// iteration: the loop body is branch-free (padding is masked by a select) and the "county finished"
// epilogue is warp-uniform.  A lane keeps its county's (alpha, beta, G_alpha, G_beta) in registers and
// completes that county's two gradient entries itself.  The (x, y) pairs are an ELL array [K][32] of
// double2 staged once per CTA into shared memory by bulk TMA and shared by all the CTA's chains.
// ------------------------------------------------------------------------------------------------
struct RadonModel {
    struct Params {
        const double2* xy;   // [K][32]  (floor_i, y_i); row j occupies 4 * nblk_j consecutive k, rows back to back,
                             //          followed by 4 all-zero k (the block prefetched past the last row)
        const int32_t* seg;  // [M][32]  (count << 16) | county, county = 0xffff: lane idle in this row
                             // followed by rows[M]: (off_j << 16) | nblk_j   (padded to a multiple of 4 ints)
        const int32_t* empty;  // [E] counties without observations (prior terms only)
        int K, M, J, n_obs, E;
    };
    __host__ __device__ static size_t xy_bytes(const Params& P) { return (size_t)P.K * 32 * sizeof(double2); }
    __host__ __device__ static size_t seg_bytes(const Params& P) {
        return ((size_t)P.M * 32 + ((P.M + 3) & ~3)) * sizeof(int32_t);
    }
    __host__ __device__ static size_t shared_bytes(const Params& P) { return xy_bytes(P) + seg_bytes(P); }

    // CTA-wide: thread 0 issues two bulk-TMA copies (xy, then seg+rows which are contiguous in HBM).
    __device__ static void stage(const Params& P, char* smem, uint64_t* bar) {
        if (threadIdx.x == 0) {
            const uint32_t b0 = (uint32_t)xy_bytes(P), b1 = (uint32_t)seg_bytes(P);
            mbar_expect_tx(bar, b0 + b1);
            tma_bulk_g2s(smem, P.xy, b0, bar);
            tma_bulk_g2s(smem + b0, P.seg, b1, bar);
        }
    }

    template <int NPL, int W, bool SMALL = false>
    __device__ static double eval(const Params& P, const char* smem, const double* q_s, double* g_s, int lane,
                                                   double*) {
        static_assert(W == 1, "RadonModel is a chain-per-warp model");
        const double2* xy = reinterpret_cast<const double2*>(smem) + lane;
        const int32_t* seg = reinterpret_cast<const int32_t*>(smem + xy_bytes(P));
        const int32_t* rows = seg + P.M * 32;
        const int J = P.J;
        const double mu_a = q_s[0], mu_b = q_s[2];
        // one exp() for the warp: lanes 0,1,2 take log sigma_a, log sigma_b, log eps; lane 3 takes -2 log eps
        const int zi = ((lane & 3) == 0) ? 1 : ((lane & 3) == 1 ? 3 : 4 + 2 * J);
        const double zl = q_s[zi];
        const double ex = exp((lane & 3) == 3 ? -2.0 * zl : zl);
        // HalfCauchy(5)+Jacobian of the same three, one log1p() for the warp
        double hc_l, dhc_l;
        halfcauchy_log(zl, ex, 5.0, 1.6094379124341002818, hc_l, dhc_l);
        const double sa = __shfl_sync(B200_FULL_MASK, ex, 0), sb = __shfl_sync(B200_FULL_MASK, ex, 1),
                     eps = __shfl_sync(B200_FULL_MASK, ex, 2);
        const double hca = __shfl_sync(B200_FULL_MASK, hc_l, 0), hcb = __shfl_sync(B200_FULL_MASK, hc_l, 1),
                     hce = __shfl_sync(B200_FULL_MASK, hc_l, 2);
        const double dhca = __shfl_sync(B200_FULL_MASK, dhc_l, 0), dhcb = __shfl_sync(B200_FULL_MASK, dhc_l, 1),
                     dhce = __shfl_sync(B200_FULL_MASK, dhc_l, 2);
        const double leps = q_s[4 + 2 * J];
        const double inv_e2 = __shfl_sync(B200_FULL_MASK, ex, 3);  // 1 / eps^2 = exp(-2 log eps)
        const double sa_ie2 = sa * inv_e2, sb_ie2 = sb * inv_e2;

        // acc: S2, sum Ga, sum a*Ga, sum Gb, sum b*Gb, sum a^2, sum b^2   (Ga/Gb raw: sums of residuals)
        double acc[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        // Rows are padded to multiples of 4 observations and stored back to back, so the whole data set is ONE stream of
        // 4-observation blocks: the next block (of this row or of the next one; 4 zero blocks follow the last row) is
        // loaded while the current one is consumed, and even/odd observations feed two independent accumulator sets.
        const double2* ptr = xy;
        double2 c0 = ptr[0], c1 = ptr[32], c2 = ptr[64], c3 = ptr[96];
        for (int j = 0; j < P.M; ++j) {
            const int nblk = rows[j] & 0xffff;
            const int sg = seg[j * 32 + lane];
            const int cnt = sg >> 16, c = sg & 0xffff;
            const bool live = c != 0xffff;
            const int ci = live ? c : 0;
            const double a_c = q_s[4 + ci], b_c = q_s[4 + J + ci];
            const double al = fma(sa, a_c, mu_a), be = fma(sb, b_c, mu_b);
            double Ga0 = 0.0, Gb0 = 0.0, S20 = 0.0, Ga1 = 0.0, Gb1 = 0.0, S21 = 0.0;
            // SMALL: no unrolling inside the persistent NUTS kernel, whose hot code must stay inside the instruction cache
            // (measured: 511 vs 562 ms per bench step; ping-ponging the prefetch registers with an unroll of 2: 526 vs 506);
            // the stand-alone leapfrog/logp kernels unroll (540 vs 393 M evals/s).
            // Padding slots hold (x, y) = (0, 0): their residual is -alpha exactly, so instead of masking every slot
            // (2 selects + a compare per observation: a fifth of the loop's issue slots) the lane removes its padding's
            // contribution after the row:  Ga += npad alpha,  S2 -= npad alpha^2,  Gb untouched (x = 0).
#pragma unroll(SMALL ? 1 : 4)
            for (int b = 0; b < nblk; ++b) {
                ptr += 128;
                const double2 n0 = ptr[0], n1 = ptr[32], n2 = ptr[64], n3 = ptr[96];
                const double r0 = c0.y - fma(be, c0.x, al), r1 = c1.y - fma(be, c1.x, al);
                const double r2 = c2.y - fma(be, c2.x, al), r3 = c3.y - fma(be, c3.x, al);
                S20 = fma(r0, r0, S20); Ga0 += r0; Gb0 = fma(r0, c0.x, Gb0);
                S21 = fma(r1, r1, S21); Ga1 += r1; Gb1 = fma(r1, c1.x, Gb1);
                S20 = fma(r2, r2, S20); Ga0 += r2; Gb0 = fma(r2, c2.x, Gb0);
                S21 = fma(r3, r3, S21); Ga1 += r3; Gb1 = fma(r3, c3.x, Gb1);
                c0 = n0; c1 = n1; c2 = n2; c3 = n3;
            }
            const double npad = (double)(4 * nblk - cnt);
            const double Ga = fma(npad, al, Ga0 + Ga1), Gb = Gb0 + Gb1;
            const double S2r = fma(-npad * al, al, S20 + S21);
            acc[0] += live ? S2r : 0.0;  // an idle lane (no county in this row) saw only padding
            if (live) {  // county finished: its two gradient entries are complete
                g_s[4 + c] = fma(sa_ie2, Ga, -a_c);
                g_s[4 + J + c] = fma(sb_ie2, Gb, -b_c);
                acc[1] += Ga;
                acc[2] = fma(a_c, Ga, acc[2]);
                acc[3] += Gb;
                acc[4] = fma(b_c, Gb, acc[4]);
                acc[5] = fma(a_c, a_c, acc[5]);
                acc[6] = fma(b_c, b_c, acc[6]);
            }
        }
        for (int e = lane; e < P.E; e += 32) {  // counties with no observations: prior terms only
            const int ce = P.empty[e];
            const double ae = q_s[4 + ce], bb = q_s[4 + J + ce];
            g_s[4 + ce] = -ae;
            g_s[4 + J + ce] = -bb;
            acc[5] = fma(ae, ae, acc[5]);
            acc[6] = fma(bb, bb, acc[6]);
        }
        warp_sum_bcast_n(acc, lane);
        const double S = 1.0e4;  // sigma = 100**2
        if (lane == 0) {
            g_s[0] = fma(inv_e2, acc[1], -mu_a * (1.0 / (S * S)));
            g_s[1] = fma(sa_ie2, acc[2], dhca);
            g_s[2] = fma(inv_e2, acc[3], -mu_b * (1.0 / (S * S)));
            g_s[3] = fma(sb_ie2, acc[4], dhcb);
            g_s[4 + 2 * J] = dhce + fma(acc[0], inv_e2, -(double)P.n_obs);
        }
        const double za = mu_a * 1.0e-4, zb = mu_b * 1.0e-4;
        const double log_S = 9.2103403719761827361;  // log 1e4
        double lp = (-0.5 * za * za - B200_HALF_LOG_2PI - log_S) + (-0.5 * zb * zb - B200_HALF_LOG_2PI - log_S);
        lp += hca + hcb + hce;
        lp += -0.5 * acc[5] - J * B200_HALF_LOG_2PI;
        lp += -0.5 * acc[6] - J * B200_HALF_LOG_2PI;
        lp += -0.5 * acc[0] * inv_e2 - P.n_obs * (B200_HALF_LOG_2PI + leps);
        return lp;
    }
};

// ------------------------------------------------------------------------------------------------
// Stochastic volatility (BASELINE config 4).  q = [mu, z_phi, log sigma, h_0 .. h_{T-1}], chain = CTA.
//   mu~Normal(0,5); phi~Uniform(-1,1) (interval transform); sigma~Exponential(10) (log transform);
//   h~AR(rho=[phi], sigma, init_dist=Normal(0,1)); y_t~Normal(0, exp((mu+h_t)/2))
// Densities: AR logp timeseries.py:646-676; Uniform + IntervalTransform continuous.py:309,
// logprob/transforms.py:1026-1073; Exponential continuous.py:1478-1480; Normal :526-527.
// Gradient: SURVEY Appendix C-4.  Thread t handles times t, t+TS, ...; neighbours h_{t-1}, h_{t+1} come
// from the chain's shared-memory copy of q; y_t^2 is read through L1 (24 KB, shared by all CTAs of the SM).
// ------------------------------------------------------------------------------------------------
struct StochVolModel {
    struct Params {
        const double* y2;  // [T] y_t^2
        int T;
    };
    __host__ __device__ static size_t shared_bytes(const Params&) { return 0; }
    __device__ static void stage(const Params&, char*, uint64_t*) {}
    template <int NPL, int W, bool SMALL = false>
    __device__ static double eval(const Params& P, const char*, const double* q_s, double* g_s, int tid, double* red) {
        constexpr int TS = 32 * W;
        const int T = P.T;
        const double mu = q_s[0], zphi = q_s[1], lsig = q_s[2];
        const double* h = q_s + 3;
        double* gh = g_s + 3;
        const double s = sigmoid(zphi);
        const double phi = 2.0 * s - 1.0;
        const double sig = exp(lsig);
        const double inv_s2 = exp(-2.0 * lsig);
        // acc: sum w_t, sum e_t h_{t-1}, sum e_t^2, sum h_t
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 2
        for (int k = 0; k < NPL; ++k) {
            const int t = tid + TS * k;
            if (t < T) {
                const double ht = h[t];
                const double w = P.y2[t] * exp(-(mu + ht));
                double g = 0.5 * w - 0.5;
                acc[0] += w;
                acc[3] += ht;
                if (t >= 1) {
                    const double hm = h[t - 1];
                    const double e = ht - phi * hm;
                    g -= e * inv_s2;
                    acc[1] = fma(e, hm, acc[1]);
                    acc[2] = fma(e, e, acc[2]);
                } else {
                    g -= ht;  // init_dist Normal(0,1) on h_0
                }
                if (t + 1 < T) {
                    const double en = h[t + 1] - phi * ht;
                    g = fma(phi * inv_s2, en, g);
                }
                gh[t] = g;
            }
        }
        team_sum_n<W>(acc, tid, red);
        const double h0 = h[0];
        if (tid == 0) {
            g_s[0] = -mu * (1.0 / 25.0) + (0.5 * acc[0] - 0.5 * T);
            g_s[1] = (1.0 - 2.0 * s) + 2.0 * s * (1.0 - s) * acc[1] * inv_s2;
            g_s[2] = 1.0 - 10.0 * sig + acc[2] * inv_s2 - (double)(T - 1);
        }
        const double z = mu * 0.2;
        double lp = -0.5 * z * z - B200_HALF_LOG_2PI - 1.6094379124341002818;           // Normal(mu | 0, 5)
        lp += -2.0 * softplus(-zphi) - zphi;                                              // Uniform(-1,1) + interval Jacobian
        lp += 2.3025850929940456840 - 10.0 * sig + lsig;                                  // Exponential(10) + log Jacobian
        lp += -0.5 * h0 * h0 - B200_HALF_LOG_2PI;                                         // h_0 ~ Normal(0,1)
        lp += -0.5 * acc[2] * inv_s2 - (T - 1) * (B200_HALF_LOG_2PI + lsig);              // innovations
        lp += -0.5 * acc[0] - T * B200_HALF_LOG_2PI - 0.5 * (T * mu + acc[3]);            // observations
        return lp;
    }
};

}  // namespace b200
