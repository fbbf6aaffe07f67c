// The persistent NUTS kernel, chain = warp.
//
// One warp runs ONE chain for the whole run (tune + draws iterations) with no host round-trip:
// momentum draw, start state, tree doubling with the generalised U-turn checks, multinomial picks,
// dual-averaging step-size adaptation and the diagonal mass-matrix Welford windows all happen here.
// It restates, operation by operation (see SURVEY.md Appendix A/B):
//     BaseHMC.astep                hmc/base_hmc.py:196-288
//     NUTS._hamiltonian_step       hmc/nuts.py:204-225
//     _Tree.extend                 hmc/nuts.py:334-392
//     _Tree._build_subtree         hmc/nuts.py:442-476   (recursion unrolled into a binary-counter stack)
//     _Tree._single_step           hmc/nuts.py:394-440
//     CpuLeapfrogIntegrator._step  hmc/integration.py:109-145
//     QuadPotentialDiag(Adapt)     hmc/quadpotential.py:211-355, :582-630
//     DualAverageAdaptation        step_sizes.py:41-84
// and consumes the chain's NumPy PCG64 `step` stream in the reference order (SURVEY 8a row a15).
//
// Data placement (n <= 32*NPL, NP = 32*NPL, lane l owns elements l + 32k):
//   registers : p (momentum of the integrator state), var (diag inverse mass), and the subtree under
//               construction: left.p, p_sum, proposal q   -> 5*NPL doubles per lane
//   shared    : q and grad of the integrator state (the model function needs all of q), the HOT lowest
//               levels of the pending-subtree stack (level h is touched every 2^h leapfrogs), per-level
//               scalars, and the model's observed data (staged once per CTA by bulk TMA)
//   global/L2 : the colder stack levels, the main tree (both edge states, p_sum, proposal q) and the
//               Welford accumulators -- touched once per doubling / per draw
#pragma once
#include "../../include/b200nuts.h"
#include "common.cuh"
#include "rng.cuh"

namespace b200 {

constexpr int kMaxLevels = 12;  // pending-subtree levels (max_treedepth <= 12)

// A subtree's multinomial weight is carried as the pair (m, s), log-weight = m + log(s), instead of one log-weight.  A
// leaf is (-dE, 1); merging (m1, s1) and (m2, s2) gives m = max(m1, m2), s = s1 e^(m1-m) + s2 e^(m2-m): one exp and no log
// per merge, and no overflow for any energy change because m carries the scale and 1 <= s <= number of leaves.  The pick
// probabilities are the numbers logaddexp gives (nuts.py:465-467, :370-376) up to rounding; measured on the bench
// workload (round 2, profiles/r2_variants.md): 481.6 vs 506.3 ms per step, every golden tree decision unchanged.

struct NutsDev {
    int C, n, tune, draws, max_td, early_td, adapt_step, mass_kind, momentum_source, store_warmup;
    int window, discard, hot_levels, chain_offset;
    int it0, n_iter;                           // this call runs the iterations [it0, it0 + n_iter) of the chain's schedule
    b200_chain_state resume, save;             // optional per-chain state in / out (null pointers: not used)
    int sampler, max_steps, stop_adaptation;   // B200_SAMPLER_*; HMC: max leapfrogs; DIAG_ADAPT_GRAD: stop after this many
    double path_length, mass_alpha;            // HMC trajectory length; DIAG_ADAPT_GRAD decay rate
    double eps0, target, gamma, kappa, t0, Emax, init_weight;
    unsigned long long philox_seed;
    const double* q0;     // [C][n]
    const double* var0;   // [C][n] or null
    const double* mean0;  // [C][n] or null
    const double* eps0c;  // [C] or null: per-chain initial step size
    const double* z;      // [C][Ttot][n] or null
    b200_pcg64* rng;      // [C]
    double* draws_out;    // [C][T][n]
    const signed char* tr_kind;  // [n] or null: record CONSTRAINED values (0 identity, 1 exp, 2 lo + (hi - lo) sigmoid)
    const double* tr_lo;         // [n]
    const double* tr_hi;         // [n]
    b200_stats st;
    b200_chain_summary sm;
    double* scratch;            // per-chain global scratch
    long long scratch_stride;   // doubles per chain
    // dynamic scheduling (see "Scheduling" below)
    struct ChainCtx* ctx;       // [C] per-chain scalar state between segments
    int* done;                  // [C] segments completed per chain
    unsigned int* ticket;       // [1] next work unit
    int seg_iters;              // iterations per work unit
};

// Scheduling.  A work unit is (chain, segment of `seg_iters` consecutive iterations).  Teams (a warp, or a CTA for W > 1)
// of a PERSISTENT grid (every CTA resident) take units from a global ticket counter in segment-major order
// (all chains' segment 0, then segment 1, ...) and keep the chain's state in global memory between segments (position,
// inverse mass, adaptation scalars, stream position: ~3 KB per boundary).  A unit whose predecessor segment is still
// running (only ever a LOWER ticket, held by a resident team: no deadlock) is waited for, so a slow chain runs back to
// back while fast chains yield their slot.  Compared with "a CTA owns its chains for the whole run" this removes (i) the
// idle warps of a CTA whose other chains are still running, (ii) the whole-wave quantisation of C chains over the resident
// slots (2048 chains over 1184 warp slots cost 1.73 rounds instead of 2) and (iii) most of the straggler tail (per-chain
// step sizes make the slowest chain 1.7x the mean).  A chain's arithmetic and stream consumption are unchanged, so
// results stay bit-identical and independent of the schedule.
struct ChainCtx {
    double log_step, log_bar, hbar, fg_n, bg_n;
    long long n_grad;
    int da_count, k_samples, window, fg_m, fg_v, bg_m, bg_v, bad_at;
};

__device__ __forceinline__ int ld_acquire_i32(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_i32(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// global scratch layout per chain, in units of NP doubles
enum { G_LQ = 0, G_LP, G_LG, G_RQ, G_RP, G_RG, G_PS, G_PQ, G_NEARP, G_FGM, G_FGV, G_BGM, G_BGV, G_Q, G_VAR, G_STACK };

__host__ __device__ inline long long nuts_scratch_doubles(int NP, int levels) {
    return (long long)(G_STACK + 4 * levels) * NP;
}
// shared memory per warp (bytes): q, g, hot stack levels (level 0: 2 vectors, others: 4), scalars
// (per chain; + 3 vectors when the subtree under construction is kept in shared memory; + the team's reduction pad)
__host__ __device__ inline size_t nuts_warp_smem_bytes(int NP, int hot, bool subs, int W) {
    const int vecs = 2 + (subs ? 3 : 0) + (hot > 0 ? 2 + 4 * (hot - 1) : 0);
    return (size_t)vecs * NP * sizeof(double) + 5 * kMaxLevels * sizeof(double) +
           (W > 1 ? W * 8 * sizeof(double) : 0);
}

// chains (warps) per CTA of the chain-per-warp kernel: 8 warps, 1 CTA per SM (measured best, round 2)
constexpr int kNutsWarpChains = 8;
// W = warps per chain (team).  SUBS: left.p / p_sum / proposal q of the subtree under construction live in shared memory
// (a team, W > 1) or in registers (a warp, W = 1).
// Register caps below the ~240 the kernel wants were measured and rejected (round 2, profiles/r2_variants.md): 224 registers
// (9 warps/SM) 460 ms, 200 (10 warps/SM, 264 B of spills) 521 ms, 168 (12 warps/SM) 685 ms vs 370 ms at 2 x 4 warps per SM.
template <class Model, int NPL, int W, bool SUBS = (W > 1)>
__global__ void __launch_bounds__(W > 1 ? 32 * W : 32 * kNutsWarpChains, 1)
    nuts_warp_kernel(const NutsDev P, const typename Model::Params M) {
    constexpr int TS = 32 * W;      // threads per chain
    constexpr int NP = TS * NPL;    // padded vector length
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ __align__(8) uint64_t tma_bar;

    // ---- CTA prologue: stage the observed data into shared memory (bulk TMA) -------------------
    const size_t data_bytes = (Model::shared_bytes(M) + 15) & ~(size_t)15;
    if (data_bytes) {
        if (threadIdx.x == 0) mbar_init(&tma_bar, 1);
        __syncthreads();
        Model::stage(M, smem_raw, &tma_bar);
        mbar_wait(&tma_bar, 0);
    }
    const char* data_s = smem_raw;

    // `lane` is the thread's index inside its team (0 .. TS-1)
    const int lane = (W == 1) ? (threadIdx.x & 31) : (int)threadIdx.x;
    const int wib = (W == 1) ? (threadIdx.x >> 5) : 0;
    __shared__ unsigned int ticket_s;  // W > 1: the CTA's current ticket

    const int hot = P.hot_levels;
    double* ws = reinterpret_cast<double*>(smem_raw + data_bytes + wib * nuts_warp_smem_bytes(NP, hot, SUBS, W));
    double* q_s = ws;
    double* g_s = ws + NP;
    double* sub_s = ws + 2 * NP + lane;            // SUBS: left.p, p_sum, proposal q of the subtree under construction
    double* hot_base = ws + (SUBS ? 5 : 2) * NP;
#define VAR(k) var[k]
    double lp_r[SUBS ? 1 : NPL], ps_r[SUBS ? 1 : NPL], pq_r[SUBS ? 1 : NPL];
    auto LPf = [&](int k) -> double& { if constexpr (SUBS) return sub_s[TS * k]; else return lp_r[k]; };
    auto PSf = [&](int k) -> double& { if constexpr (SUBS) return sub_s[NP + TS * k]; else return ps_r[k]; };
    auto PQf = [&](int k) -> double& { if constexpr (SUBS) return sub_s[2 * NP + TS * k]; else return pq_r[k]; };
#define LP(k) LPf(k)
#define PS(k) PSf(k)
#define PQ(k) PQf(k)
    double* sc_logw = hot_base + (hot > 0 ? 2 + 4 * (hot - 1) : 0) * NP;
    double* sc_pe = sc_logw + kMaxLevels;
    double* sc_plogp = sc_pe + kMaxLevels;
    double* sc_pidx = sc_plogp + kMaxLevels;
    double* sc_s = sc_pidx + kMaxLevels;
    double* red = sc_s + kMaxLevels;     // W x 8 doubles, cross-warp reductions (W > 1)
    const int n = P.n;
    const int it_lo = P.it0, it_hi = P.it0 + P.n_iter;  // global iteration indices of this call
    const int rec_lo = P.store_warmup ? it_lo : max(P.tune, it_lo);  // first recorded iteration
    const int T_out = max(0, it_hi - rec_lo);
    const int seg_iters = P.seg_iters > 0 ? P.seg_iters : P.n_iter;
    const unsigned int n_seg = (unsigned int)((P.n_iter + seg_iters - 1) / seg_iters);
    const unsigned int n_units = n_seg * (unsigned int)P.C;

    // ---- work loop: one (chain, segment) unit per turn ---------------------------------------------------
    for (;;) {
    unsigned int unit;
    if constexpr (W == 1) {
        unit = 0;
        if (lane == 0) unit = atomicAdd(P.ticket, 1u);
        unit = __shfl_sync(B200_FULL_MASK, unit, 0);
    } else {
        __syncthreads();  // everyone is done with the previous unit (and with ticket_s)
        if (threadIdx.x == 0) ticket_s = atomicAdd(P.ticket, 1u);
        __syncthreads();
        unit = ticket_s;
    }
    if (unit >= n_units) break;
    const int seg = (int)(unit / (unsigned int)P.C);
    const int chain = (int)(unit - (unsigned int)seg * (unsigned int)P.C);
    const int it_begin = it_lo + seg * seg_iters, it_end = min(it_hi, it_begin + seg_iters);
    if (seg > 0) {  // the chain's previous segment may still be running on another team (every thread acquires)
        while (ld_acquire_i32(P.done + chain) < seg) __nanosleep(64);
        team_sync<W>();
    }
    double* gs = P.scratch + (long long)chain * P.scratch_stride;

    // which: 0 = left.p, 1 = right.p, 2 = p_sum, 3 = proposal q.  Level 0 (a single leaf) keeps only 2, 3.
    auto lvl = [&](int h, int which) -> double* {
        if (h < hot) return hot_base + (h == 0 ? (which - 2) : (2 + 4 * (h - 1) + which)) * NP;
        return gs + (long long)(G_STACK + 4 * h + which) * NP;
    };
    auto gvec = [&](int which) -> double* { return gs + (long long)which * NP; };

    // ---- per-chain state: initialised by the first segment, carried through global memory afterwards ------------
    double var[NPL], p[NPL];
    int fg_m, fg_v, bg_m, bg_v, k_samples, window, da_count, bad_at;
    double fg_n, bg_n, log_step, log_bar, hbar;
    long long n_grad;
    const double eps_init = P.eps0c ? P.eps0c[chain] : P.eps0;
    const double da_mu = log(10.0 * eps_init);  // dual averaging (step_sizes.py:50-57)
    if (seg == 0) {
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            q_s[i] = (i < n) ? P.q0[(long long)chain * n + i] : 0.0;
            g_s[i] = 0.0;
            VAR(k) = (i < n && P.var0) ? P.var0[(long long)chain * n + i] : 1.0;
            // Welford estimators: foreground starts at (mean0, var0 * weight, weight); background empty
            if (P.mass_kind == B200_MASS_DIAG_ADAPT) {
                gvec(G_FGM)[i] = (i < n && P.mean0) ? P.mean0[(long long)chain * n + i] : 0.0;
                gvec(G_FGV)[i] = VAR(k) * P.init_weight;
                gvec(G_BGM)[i] = 0.0;
                gvec(G_BGV)[i] = 0.0;
            }
        }
        fg_m = G_FGM; fg_v = G_FGV; bg_m = G_BGM; bg_v = G_BGV;
        fg_n = P.init_weight; bg_n = 0.0;
        k_samples = 0; window = P.window;
        log_step = log(eps_init); log_bar = log_step; hbar = 0.0;
        da_count = 1;
        n_grad = 0;
        bad_at = -1;
        if (P.resume.log_step) {  // continue a chain from an exported state (BaseHMC / potential / step_adapt sampling_state)
            const b200_chain_state& R = P.resume;
            log_step = R.log_step[chain]; log_bar = R.log_bar[chain]; hbar = R.hbar[chain]; da_count = R.da_count[chain];
            k_samples = R.n_samples[chain]; window = R.window[chain];
            fg_n = R.fg_n[chain]; bg_n = R.bg_n[chain]; n_grad = R.n_grad[chain];
#pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                const long long o = (long long)chain * n + i;
                const bool in = i < n;
                q_s[i] = in ? R.q[o] : 0.0;
                VAR(k) = in ? R.var[o] : 1.0;
                gvec(G_FGM)[i] = in ? R.fg_mean[o] : 0.0;
                gvec(G_FGV)[i] = in ? R.fg_m2[o] : 0.0;
                gvec(G_BGM)[i] = in ? R.bg_mean[o] : 0.0;
                gvec(G_BGV)[i] = in ? R.bg_m2[o] : 0.0;
            }
        }
    } else {
        const ChainCtx cx = P.ctx[chain];
        fg_m = cx.fg_m; fg_v = cx.fg_v; bg_m = cx.bg_m; bg_v = cx.bg_v;
        fg_n = cx.fg_n; bg_n = cx.bg_n; k_samples = cx.k_samples; window = cx.window;
        log_step = cx.log_step; log_bar = cx.log_bar; hbar = cx.hbar; da_count = cx.da_count;
        n_grad = cx.n_grad; bad_at = cx.bad_at;
        const double* sq = gvec(G_Q); const double* sv = gvec(G_VAR);
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            q_s[i] = sq[i];
            g_s[i] = 0.0;
            VAR(k) = sv[i];
        }
    }
    Pcg64 rng;
    {
        const b200_pcg64 r = P.rng[chain];
        rng.load(r.state_hi, r.state_lo, r.inc_hi, r.inc_lo);
    }
    team_sync<W>();

    // QuadPotentialDiagAdaptExp.update with use_grads (quadpotential.py:531-579); sample = q_s, grad = g_s.  The four
    // Welford slots of the scratch hold (mean, var) of the draws and of the gradients.
    auto grad_mass_update = [&](double* em, double* ev, double* gm, double* gv) {
        if (k_samples >= P.stop_adaptation) return;
        const double al = P.mass_alpha, om = 1.0 - P.mass_alpha;
        if (k_samples > P.discard) {
#pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                double d = q_s[i] - em[i];
                em[i] = __dadd_rn(em[i], __dmul_rn(al, d));
                ev[i] = __dmul_rn(om, __dadd_rn(ev[i], __dmul_rn(al, __dmul_rn(d, d))));
                d = g_s[i] - gm[i];
                gm[i] = __dadd_rn(gm[i], __dmul_rn(al, d));
                gv[i] = __dmul_rn(om, __dadd_rn(gv[i], __dmul_rn(al, __dmul_rn(d, d))));
            }
        } else if (k_samples == P.discard) {
#pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                em[i] = q_s[i]; ev[i] = 0.0; gm[i] = g_s[i]; gv[i] = 0.0;
            }
        }
        if (k_samples > 2 * P.discard) {  // _update_from_variances :569-575: var = sqrt(var_draws / var_grads), no clipping
#pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                if (i < n) VAR(k) = sqrt(ev[i] / gv[i]);
            }
        }
        ++k_samples;
    };

    for (int it = it_begin; it < it_end && bad_at < 0; ++it) {
        const bool tuning = it < P.tune;
        const bool adapting = tuning && P.adapt_step;

        // ---- start = integrator.compute_state(q0, p0)  (integration.py:68-75): the evaluation at q0 does not depend on
        //      p0, so it runs first ...
        team_sync<W>();
        const double logp0 = Model::template eval<NPL, W, true>(M, data_s, q_s, g_s, lane, red);
        team_sync<W>();
        ++n_grad;
        // ---- ... which lets QuadPotentialDiagAdaptExp.update(sample, grad) (quadpotential.py:531-567) of the PREVIOUS
        //      iteration run here, where the accepted position's gradient is at hand (the reference calls it at the end of
        //      astep, base_hmc.py:238, before the next potential.random(): same order of effects, no gradient carried
        //      through the tree).  _ExpWeightedVariance.add_sample :465-469 with NumPy's unfused elementwise arithmetic.
        if (P.mass_kind == B200_MASS_DIAG_ADAPT_GRAD && it > 0 && it - 1 < P.tune)
            grad_mass_update(gvec(G_FGM), gvec(G_FGV), gvec(G_BGM), gvec(G_BGV));
        // ---- p0 = potential.random(): inv_std * z  (quadpotential.py:323-326, :617-619) ------------
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            double zz = 0.0;
            if (i < n) {
                zz = (P.momentum_source == B200_MOMENTUM_HOST_BUFFER)
                         ? P.z[((long long)chain * P.n_iter + (it - it_lo)) * n + i]
                         : philox_normal(P.philox_seed, (uint32_t)(chain + P.chain_offset), (uint32_t)it, (uint32_t)i);
            }
            p[k] = (1.0 / sqrt(VAR(k))) * zz;
        }
        double kin = 0.0;
#pragma unroll
        for (int k = 0; k < NPL; ++k) kin = fma(p[k], VAR(k) * p[k], kin);
        const double E0 = 0.5 * team_sum<W>(kin, lane, red) - logp0;
        if (!isfinite(E0)) {  // "Bad initial energy" (base_hmc.py:205-224): freeze the chain
            bad_at = it;
            break;
        }
        const double eps = exp(adapting ? log_step : log_bar);  // step_adapt.current (step_sizes.py:60-64)
        const int maxd = (tuning && it < 200) ? P.early_td : P.max_td;  // nuts.py:205-208

        double m_logw = 0.0, m_pe = E0, m_plogp = logp0;
        double m_s = 1.0;
        int m_pidx = 0;
        double accept_sum = 0.0, max_de = 0.0;  // sum of min(1, exp(-dE)): exp(log_accept_sum) of nuts.py:415 without the log
        int n_prop = 0, depth = 0;
        bool diverged = false, turned = false, hit_max = false;
        double hmc_accept = 0.0;
        double* PQv = gvec(G_PQ);
        int d_iter = 0;
        if (P.sampler == B200_SAMPLER_HMC) {
            // ---- HamiltonianMC._hamiltonian_step (hmc/hmc.py:143-200): a fixed-length trajectory, Metropolis accept ----
            d_iter = -1;  // no tree: `reached_max_treedepth` stays false
#pragma unroll
            for (int k = 0; k < NPL; ++k) PQv[lane + TS * k] = q_s[lane + TS * k];  // end = start unless accepted
            // step_rand = unif (hmc.py:35-36, :141): Generator.uniform(0.85, 1.15) = low + (high - low) * next_double
            const double es = (0.85 + (1.15 - 0.85) * rng.next_double()) * eps, dt = 0.5 * es;
            const double ratio = P.path_length / es;
            int n_steps = (ratio >= (double)P.max_steps) ? P.max_steps : (int)ratio;  // max(1, int(.)), min(max_steps, .)
            if (n_steps < 1) n_steps = 1;
            double logp = logp0, E = E0;
            for (int sidx = 0; sidx < n_steps; ++sidx) {  // integrator.step (integration.py:109-145)
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    const int i = lane + TS * k;
                    p[k] = fma(dt, g_s[i], p[k]);
                    q_s[i] = fma(es, VAR(k) * p[k], q_s[i]);
                }
                team_sync<W>();
                logp = Model::template eval<NPL, W, true>(M, data_s, q_s, g_s, lane, red);
                team_sync<W>();
                ++n_grad;
                double kk = 0.0;
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    p[k] = fma(dt, g_s[lane + TS * k], p[k]);
                    kk = fma(p[k], VAR(k) * p[k], kk);
                }
                E = 0.5 * team_sum<W>(kk, lane, red) - logp;
            }
            n_prop = n_steps;
            bool div = !isfinite(E);           // "Divergence encountered, bad energy."
            double dE = E - E0;
            if (isnan(dE)) dE = INFINITY;
            if (fabs(dE) > P.Emax) div = true;  // two-sided, unlike NUTS (hmc.py:164)
            hmc_accept = fmin(1.0, exp(-dE));
            bool accepted = false;
            if (!div) accepted = !(rng.next_double() >= hmc_accept);  // the uniform is drawn only without a divergence
            if (accepted) {
#pragma unroll
                for (int k = 0; k < NPL; ++k) PQv[lane + TS * k] = q_s[lane + TS * k];
                m_pidx = n_steps;
            }
            diverged = div; m_pe = E; m_plogp = logp; max_de = dE;  // stats report the trajectory's LAST state (hmc.py:180-188)
        } else {
            // ---- _Tree.__init__ (nuts.py:292-332): both edges, proposal and p_sum are the start state ----
            double* Lq = gvec(G_LQ); double* Lp = gvec(G_LP); double* Lg = gvec(G_LG);
            double* Rq = gvec(G_RQ); double* Rp = gvec(G_RP); double* Rg = gvec(G_RG);
            double* PSv = gvec(G_PS); double* NEARP = gvec(G_NEARP);
    #pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                const double qi = q_s[i], gi = g_s[i];
                Lq[i] = qi; Rq[i] = qi; PQv[i] = qi;
                Lg[i] = gi; Rg[i] = gi;
                Lp[i] = p[k]; Rp[i] = p[k]; PSv[i] = p[k];
            }
            int L_idx = 0, R_idx = 0;
            for (; d_iter < maxd; ++d_iter) {
                const int dir = (rng.next_double() < 0.5) ? 1 : -1;  // nuts.py:215
                // ---- load the edge we grow from into the integrator state; remember its p ----------------
                const double* Eq = dir > 0 ? Rq : Lq;
                const double* Ep = dir > 0 ? Rp : Lp;
                const double* Eg = dir > 0 ? Rg : Lg;
                int w_idx = dir > 0 ? R_idx : L_idx;
    #pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    const int i = lane + TS * k;
                    q_s[i] = Eq[i];
                    g_s[i] = Eg[i];
                    p[k] = Ep[i];
                    NEARP[i] = p[k];
                }
                const double es = dir * eps, dt = 0.5 * es;

                // ---- _build_subtree(edge, depth, +-eps): 2^depth leaves, merges driven by a binary counter --
                bool sub_div = false, sub_turn = false;
                double c_logw = 0.0, c_pe = 0.0, c_plogp = 0.0;
                double c_s = 1.0;
                int c_pidx = 0;
                const int n_leaf = 1 << depth;
                for (int leaf = 0; leaf < n_leaf; ++leaf) {
                    // -- one leapfrog (integration.py:109-145)
    #pragma unroll
                    for (int k = 0; k < NPL; ++k) {
                        const int i = lane + TS * k;
                        p[k] = fma(dt, g_s[i], p[k]);
                        q_s[i] = fma(es, VAR(k) * p[k], q_s[i]);
                    }
                    team_sync<W>();
                    const double logp = Model::template eval<NPL, W, true>(M, data_s, q_s, g_s, lane, red);
                    team_sync<W>();
                    ++n_grad;
                    double kk = 0.0;
    #pragma unroll
                    for (int k = 0; k < NPL; ++k) {
                        const int i = lane + TS * k;
                        p[k] = fma(dt, g_s[i], p[k]);
                        kk = fma(p[k], VAR(k) * p[k], kk);
                    }
                    const double E = 0.5 * team_sum<W>(kk, lane, red) - logp;
                    w_idx += dir;
                    // -- _single_step bookkeeping (nuts.py:406-440)
                    ++n_prop;
                    double dE = E - E0;
                    if (isnan(dE)) dE = INFINITY;
                    accept_sum += (dE > 0) ? exp(-dE) : 1.0;
                    if (fabs(dE) > fabs(max_de)) max_de = dE;
                    if (!(dE < P.Emax)) {
                        sub_div = true;
                        break;
                    }
                    // the leaf as a height-0 subtree: left = right = p_sum = p, proposal = itself
    #pragma unroll
                    for (int k = 0; k < NPL; ++k) {
                        LP(k) = p[k];
                        PS(k) = p[k];
                        PQ(k) = q_s[lane + TS * k];
                    }
                    c_logw = -dE; c_pe = E; c_plogp = logp; c_pidx = w_idx;
                    c_s = 1.0;

                    // -- merge with pending left siblings while the counter carries (nuts.py:452-476)
                    int h = 0;
                    for (int m = leaf; m & 1; m >>= 1, ++h) {
                        const double* t_ps = lvl(h, 2);
                        const double* t_lp = h ? lvl(h, 0) : t_ps;
                        const double* t_rp = h ? lvl(h, 1) : t_ps;
                        double dots[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                        if (h == 0) {
    #pragma unroll
                            for (int k = 0; k < NPL; ++k) {
                                const int i = lane + TS * k;
                                const double tp = t_ps[i];
                                const double s = tp + PS(k);
                                dots[0] = fma(s, VAR(k) * tp, dots[0]);
                                dots[1] = fma(s, VAR(k) * p[k], dots[1]);
                                LP(k) = tp;
                                PS(k) = s;
                            }
                            double d2[2] = {dots[0], dots[1]};
                            team_sum_n<W>(d2, lane, red);
                            dots[0] = d2[0]; dots[1] = d2[1];
                            dots[2] = dots[3] = dots[4] = dots[5] = 1.0;
                        } else {
    #pragma unroll
                            for (int k = 0; k < NPL; ++k) {
                                const int i = lane + TS * k;
                                const double tl = t_lp[i], tr = t_rp[i], tp = t_ps[i];
                                const double s = tp + PS(k);
                                const double vl = VAR(k) * tl, vr = VAR(k) * p[k];
                                dots[0] = fma(s, vl, dots[0]);
                                dots[1] = fma(s, vr, dots[1]);
                                const double s1 = tp + LP(k);  // tree1.p_sum + tree2.left.p
                                dots[2] = fma(s1, vl, dots[2]);
                                dots[3] = fma(s1, VAR(k) * LP(k), dots[3]);
                                const double s2 = tr + PS(k);  // tree1.right.p + tree2.p_sum
                                dots[4] = fma(s2, VAR(k) * tr, dots[4]);
                                dots[5] = fma(s2, vr, dots[5]);
                                LP(k) = tl;
                                PS(k) = s;
                            }
                        }
                        if (h) team_sum_n<W>(dots, lane, red);
                        const bool turn = (dots[0] <= 0) || (dots[1] <= 0) || (dots[2] <= 0) || (dots[3] <= 0) ||
                                          (dots[4] <= 0) || (dots[5] <= 0);
                        // weights (m, s): tree1 = (sc_logw[h], sc_s[h]), tree2 = (c_logw, c_s); P(pick tree2) = w2 / (w1 + w2)
                        const double t_m = sc_logw[h], t_s = sc_s[h];
                        const double dm = c_logw - t_m;
                        const double e_w = exp(-fabs(dm));
                        const double w2 = (dm >= 0.0) ? c_s : c_s * e_w, w1 = (dm >= 0.0) ? t_s * e_w : t_s;
                        const double ws = w1 + w2;
                        const double u = rng.next_double();  // drawn whenever both halves succeeded (nuts.py:466)
                        if (!(u * ws < w2)) {  // keep tree1's proposal
                            const double* t_pq = lvl(h, 3);
    #pragma unroll
                            for (int k = 0; k < NPL; ++k) PQ(k) = t_pq[lane + TS * k];
                            c_pe = sc_pe[h]; c_plogp = sc_plogp[h]; c_pidx = (int)sc_pidx[h];
                        }
                        c_logw = fmax(c_logw, t_m);
                        c_s = ws;
                        if (turn) {
                            sub_turn = true;
                            break;
                        }
                    }
                    if (sub_turn) break;
                    // -- not the last leaf: park the subtree (height h) until its right sibling is built
                    if (leaf + 1 < n_leaf) {
                        double* s_ps = lvl(h, 2);
                        double* s_pq = lvl(h, 3);
                        if (h == 0) {
    #pragma unroll
                            for (int k = 0; k < NPL; ++k) {
                                const int i = lane + TS * k;
                                s_ps[i] = PS(k);
                                s_pq[i] = PQ(k);
                            }
                        } else {
                            double* s_lp = lvl(h, 0);
                            double* s_rp = lvl(h, 1);
    #pragma unroll
                            for (int k = 0; k < NPL; ++k) {
                                const int i = lane + TS * k;
                                s_lp[i] = LP(k);
                                s_rp[i] = p[k];
                                s_ps[i] = PS(k);
                                s_pq[i] = PQ(k);
                            }
                        }
                        if (lane == 0) {
                            sc_logw[h] = c_logw; sc_pe[h] = c_pe; sc_plogp[h] = c_plogp; sc_pidx[h] = (double)c_pidx;
                            sc_s[h] = c_s;
                        }
                        team_sync<W>();
                    }
                }
                ++depth;  // nuts.py:365 (counts the aborted doubling too)
                if (sub_div || sub_turn) {
                    diverged = sub_div;
                    turned = sub_turn;
                    break;
                }
                // ---- the new outer edge is the integrator state (self.right/left = tree.right) ------------
                {
                    double* Nq = dir > 0 ? Rq : Lq;
                    double* Np = dir > 0 ? Rp : Lp;
                    double* Ng = dir > 0 ? Rg : Lg;
    #pragma unroll
                    for (int k = 0; k < NPL; ++k) {
                        const int i = lane + TS * k;
                        Nq[i] = q_s[i];
                        Ng[i] = g_s[i];
                        Np[i] = p[k];
                    }
                    if (dir > 0) R_idx = w_idx; else L_idx = w_idx;
                }
                // ---- biased progressive pick (nuts.py:370-374), drawn before the full-tree U-turn checks --
                {
                    // accept the new subtree's proposal iff u < w_new / w_old  (log(u) < log_size_new - log_size_old)
                    const double u = rng.next_double();
                    const double dm = c_logw - m_logw;
                    const double e_w = exp(-fabs(dm));
                    const double wn = (dm >= 0.0) ? c_s : c_s * e_w, wo = (dm >= 0.0) ? m_s * e_w : m_s;
                    if (u * wo < wn) {
    #pragma unroll
                        for (int k = 0; k < NPL; ++k) PQv[lane + TS * k] = PQ(k);
                        m_pe = c_pe; m_plogp = c_plogp; m_pidx = c_pidx;
                    }
                    m_logw = fmax(c_logw, m_logw);
                    m_s = wo + wn;
                }
                // ---- U-turn checks on the whole tree (nuts.py:376-390) ------------------------------------
                {
                    const double* FARP = dir > 0 ? Lp : Rp;
                    double dots[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    #pragma unroll
                    for (int k = 0; k < NPL; ++k) {
                        const int i = lane + TS * k;
                        const double so = PSv[i], fp = FARP[i], np_ = NEARP[i];
                        const double s = so + PS(k);
                        PSv[i] = s;
                        const double vf = VAR(k) * fp, vw = VAR(k) * p[k];
                        dots[0] = fma(s, vf, dots[0]);
                        dots[1] = fma(s, vw, dots[1]);
                        const double a = so + LP(k);   // old p_sum + (new subtree's edge adjacent to the old tree).p
                        dots[2] = fma(a, vf, dots[2]);
                        dots[3] = fma(a, VAR(k) * LP(k), dots[3]);
                        const double b = np_ + PS(k);  // (old tree's edge adjacent to the new subtree).p + new p_sum
                        dots[4] = fma(b, VAR(k) * np_, dots[4]);
                        dots[5] = fma(b, vw, dots[5]);
                    }
                    team_sum_n<W>(dots, lane, red);
                    if ((dots[0] <= 0) || (dots[1] <= 0) || (dots[2] <= 0) || (dots[3] <= 0) || (dots[4] <= 0) ||
                        (dots[5] <= 0)) {
                        turned = true;
                        break;
                    }
                }
            }
        }
        if (d_iter == maxd) hit_max = !tuning;  // for/else of nuts.py:220-221

        // ---- the accepted position becomes the chain state -------------------------------------------
        const double accept = (P.sampler == B200_SAMPLER_HMC) ? hmc_accept : accept_sum / n_prop;  // nuts.py:479
        const bool rec = P.store_warmup || !tuning;
        const int t_out = it - rec_lo;
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            const double qi = PQv[i];
            q_s[i] = qi;
            PQ(k) = qi;
            if (rec && i < n) P.draws_out[((long long)chain * T_out + t_out) * n + i] = constrained(qi, i, P.tr_kind, P.tr_lo, P.tr_hi);
        }
        // ---- step_adapt.update (step_sizes.py:66-78); products/sums kept unfused like the Python scalars
        if (adapting) {
            const double w = 1.0 / (da_count + P.t0);
            hbar = __dadd_rn(__dmul_rn(1.0 - w, hbar), __dmul_rn(w, P.target - accept));
            log_step = da_mu - __dmul_rn(hbar, sqrt((double)da_count)) / P.gamma;
            const double mk = pow((double)da_count, -P.kappa);
            log_bar = __dadd_rn(__dmul_rn(mk, log_step), __dmul_rn(1.0 - mk, log_bar));
            ++da_count;
        }
        // ---- potential.update (quadpotential.py:335-355, _WeightedVariance.add_sample :431-437) --------
        if (tuning && P.mass_kind == B200_MASS_DIAG_ADAPT) {
            if (k_samples > P.discard) {
                fg_n += 1.0;
                bg_n += 1.0;
                double* fm = gvec(fg_m); double* fv = gvec(fg_v);
                double* bm = gvec(bg_m); double* bv = gvec(bg_v);
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    const int i = lane + TS * k;
                    const double x = PQ(k);
                    double mean = fm[i];
                    double d0 = x - mean;
                    mean = __dadd_rn(mean, d0 / fg_n);
                    fm[i] = mean;
                    fv[i] = __dadd_rn(fv[i], __dmul_rn(d0, x - mean));
                    mean = bm[i];
                    d0 = x - mean;
                    mean = __dadd_rn(mean, d0 / bg_n);
                    bm[i] = mean;
                    bv[i] = __dadd_rn(bv[i], __dmul_rn(d0, x - mean));
                }
            }
            if (k_samples > window) {
                const double* fv = gvec(fg_v);
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    const int i = lane + TS * k;
                    if (i < n) VAR(k) = fmin(fmax(fv[i] / fg_n, 1e-12), 1e12);
                }
            }
            if (k_samples > 0 && k_samples % window == 0) {
                const int tm = fg_m, tv = fg_v;
                fg_m = bg_m; fg_v = bg_v; fg_n = bg_n;
                bg_m = tm; bg_v = tv; bg_n = 0.0;
                double* bm = gvec(bg_m); double* bv = gvec(bg_v);
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    bm[lane + TS * k] = 0.0;
                    bv[lane + TS * k] = 0.0;
                }
            }
            ++k_samples;
        }
        // ---- stats (nuts.py:478-489, base_hmc.py:275-286) --------------------------------------------
        if (rec && lane == 0) {
            const long long o = (long long)chain * T_out + t_out;
            if (P.st.depth) P.st.depth[o] = depth;
            if (P.st.tree_size) P.st.tree_size[o] = n_prop;
            if (P.st.index_in_trajectory) P.st.index_in_trajectory[o] = m_pidx;
            if (P.st.diverging) P.st.diverging[o] = diverged ? 1 : 0;
            if (P.st.reached_max_treedepth) P.st.reached_max_treedepth[o] = hit_max ? 1 : 0;
            if (P.st.step_size) P.st.step_size[o] = exp(log_step);
            if (P.st.step_size_bar) P.st.step_size_bar[o] = exp(log_bar);
            if (P.st.mean_tree_accept) P.st.mean_tree_accept[o] = accept;
            if (P.st.energy) P.st.energy[o] = m_pe;
            if (P.st.energy_error) P.st.energy_error[o] = (P.sampler == B200_SAMPLER_HMC) ? max_de : m_pe - E0;
            if (P.st.max_energy_error) P.st.max_energy_error[o] = max_de;
            if (P.st.model_logp) P.st.model_logp[o] = m_plogp;
        }
        (void)turned;
        team_sync<W>();
    }

    // ---- a frozen chain ("Bad initial energy"): the iterations that never ran are NaN in the output --------------
    if (bad_at >= 0) {
        for (int t = max(bad_at, it_begin); t < it_end; ++t) {
            if (!(P.store_warmup || t >= P.tune)) continue;
            const int t_out = t - rec_lo;
#pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                if (i < n) P.draws_out[((long long)chain * T_out + t_out) * n + i] = nan("");
            }
            if (lane == 0) stats_sentinel(P.st, (long long)chain * T_out + t_out);
        }
    }
    // ---- end of the segment: the stream position goes back to the caller's array (it is also where the next segment
    //      picks it up); last segment: adaptation results; otherwise: the chain's state for the next segment ------------
    const bool last_seg = it_end >= it_hi;
    if (lane == 0) {
        b200_pcg64 r;
        r.state_hi = (uint64_t)(rng.state >> 64); r.state_lo = (uint64_t)rng.state;
        r.inc_hi = (uint64_t)(rng.inc >> 64); r.inc_lo = (uint64_t)rng.inc;
        P.rng[chain] = r;
        if (last_seg) {
            if (P.sm.grad_evals) P.sm.grad_evals[chain] = n_grad;
            if (P.sm.bad_energy_at) P.sm.bad_energy_at[chain] = bad_at;
            if (P.sm.final_step_size) P.sm.final_step_size[chain] = exp(log_bar);
        } else {
            ChainCtx cx;
            cx.log_step = log_step; cx.log_bar = log_bar; cx.hbar = hbar; cx.fg_n = fg_n; cx.bg_n = bg_n;
            cx.n_grad = n_grad; cx.da_count = da_count; cx.k_samples = k_samples; cx.window = window;
            cx.fg_m = fg_m; cx.fg_v = fg_v; cx.bg_m = bg_m; cx.bg_v = bg_v; cx.bad_at = bad_at;
            P.ctx[chain] = cx;
        }
    }
    if (last_seg && P.save.log_step) {  // export the chain's state (the pending DIAG_ADAPT_GRAD update stays pending)
        const b200_chain_state& S = P.save;
        if (lane == 0) {
            S.log_step[chain] = log_step; S.log_bar[chain] = log_bar; S.hbar[chain] = hbar; S.da_count[chain] = da_count;
            S.n_samples[chain] = k_samples; S.window[chain] = window;
            S.fg_n[chain] = fg_n; S.bg_n[chain] = bg_n; S.n_grad[chain] = n_grad;
        }
        const double* fm = gvec(fg_m); const double* fv = gvec(fg_v); const double* bm = gvec(bg_m); const double* bv = gvec(bg_v);
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            if (i < n) {
                const long long o = (long long)chain * n + i;
                S.q[o] = q_s[i]; S.var[o] = VAR(k);
                S.fg_mean[o] = fm[i]; S.fg_m2[o] = fv[i]; S.bg_mean[o] = bm[i]; S.bg_m2[o] = bv[i];
            }
        }
    }
    if (last_seg) {
        if (P.mass_kind == B200_MASS_DIAG_ADAPT_GRAD && it_hi >= P.tune + P.draws && P.draws == 0 && bad_at < 0 && P.sm.final_var &&
            !P.save.log_step) {
            // the update that follows the last tuning iteration needs that position's gradient: one more evaluation
            team_sync<W>();
            (void)Model::template eval<NPL, W, true>(M, data_s, q_s, g_s, lane, red);
            team_sync<W>();
            grad_mass_update(gvec(G_FGM), gvec(G_FGV), gvec(G_BGM), gvec(G_BGV));
        }
        if (P.sm.final_var) {
#pragma unroll
            for (int k = 0; k < NPL; ++k) {
                const int i = lane + TS * k;
                if (i < n) P.sm.final_var[(long long)chain * n + i] = VAR(k);
            }
        }
    } else {
        double* sq = gvec(G_Q); double* sv = gvec(G_VAR);
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            sq[i] = q_s[i];
            sv[i] = VAR(k);
        }
        __threadfence();   // every thread's state writes are visible device-wide before the segment is published
        team_sync<W>();
        if (lane == 0) st_release_i32(P.done + chain, seg + 1);
    }
    }  // work loop
}

#undef VAR

// ---------------------------------------------------------------------------------------------------
// Batched logp + gradient: one warp per point.  Replaces ValueGradFunction._pytensor_function
// (model/core.py:232-267) evaluated at C points.
// ---------------------------------------------------------------------------------------------------
template <class Model, int NPL, int W>
__global__ void __launch_bounds__(256) logp_grad_warp_kernel(const typename Model::Params M, int n, int C,
                                                             const double* __restrict__ q,
                                                             double* __restrict__ logp_out,
                                                             double* __restrict__ grad_out, long long ldq, long long ldg) {
    constexpr int TS = 32 * W;
    constexpr int NP = TS * NPL;
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ __align__(8) uint64_t tma_bar;
    const size_t data_bytes = (Model::shared_bytes(M) + 15) & ~(size_t)15;
    if (data_bytes) {
        if (threadIdx.x == 0) mbar_init(&tma_bar, 1);
        __syncthreads();
        Model::stage(M, smem_raw, &tma_bar);
        mbar_wait(&tma_bar, 0);
    }
    const int lane = (W == 1) ? (threadIdx.x & 31) : (int)threadIdx.x;
    const int wib = (W == 1) ? (threadIdx.x >> 5) : 0, wpb = (W == 1) ? (blockDim.x >> 5) : 1;
    double* q_s = reinterpret_cast<double*>(smem_raw + data_bytes) + (size_t)wib * (2 * NP + (W > 1 ? 8 * W : 0));
    double* g_s = q_s + NP;
    double* red = g_s + NP;
    for (int c = blockIdx.x * wpb + wib; c < C; c += gridDim.x * wpb) {
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            q_s[i] = (i < n) ? q[(long long)c * ldq + i] : 0.0;
            g_s[i] = 0.0;
        }
        team_sync<W>();
        const double lp = Model::template eval<NPL, W>(M, smem_raw, q_s, g_s, lane, red);
        team_sync<W>();
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            if (i < n) grad_out[(long long)c * ldg + i] = g_s[i];
        }
        if (lane == 0) logp_out[c] = lp;
        team_sync<W>();
    }
}

// ---------------------------------------------------------------------------------------------------
// Batched leapfrog with a diagonal potential: compute_state (n_steps == 0) or n_steps x _step
// (integration.py:68-75, :109-145).  One warp per chain; State is struct-of-arrays in global memory.
// ---------------------------------------------------------------------------------------------------
template <class Model, int NPL, int W>
__global__ void __launch_bounds__(256)
    leapfrog_warp_kernel(const typename Model::Params M, int n, int C, const double* __restrict__ var_in,
                         const double* __restrict__ eps_in, int n_steps, double* q, double* p_io, double* v_io,
                         double* grad, double* energy, double* logp_io, long long* idx) {
    constexpr int TS = 32 * W;
    constexpr int NP = TS * NPL;
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ __align__(8) uint64_t tma_bar;
    const size_t data_bytes = (Model::shared_bytes(M) + 15) & ~(size_t)15;
    if (data_bytes) {
        if (threadIdx.x == 0) mbar_init(&tma_bar, 1);
        __syncthreads();
        Model::stage(M, smem_raw, &tma_bar);
        mbar_wait(&tma_bar, 0);
    }
    const int lane = (W == 1) ? (threadIdx.x & 31) : (int)threadIdx.x;
    const int wib = (W == 1) ? (threadIdx.x >> 5) : 0, wpb = (W == 1) ? (blockDim.x >> 5) : 1;
    double* q_s = reinterpret_cast<double*>(smem_raw + data_bytes) + (size_t)wib * (2 * NP + (W > 1 ? 8 * W : 0));
    double* g_s = q_s + NP;
    double* red = g_s + NP;
    for (int c = blockIdx.x * wpb + wib; c < C; c += gridDim.x * wpb) {
        double var[NPL], p[NPL];
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            const bool in = i < n;
            q_s[i] = in ? q[(long long)c * n + i] : 0.0;
            g_s[i] = (in && n_steps > 0) ? grad[(long long)c * n + i] : 0.0;
            p[k] = in ? p_io[(long long)c * n + i] : 0.0;
            var[k] = in ? var_in[(long long)c * n + i] : 1.0;
        }
        team_sync<W>();
        double lp = 0.0, E = 0.0;
        if (n_steps == 0) {
            lp = Model::template eval<NPL, W>(M, smem_raw, q_s, g_s, lane, red);
            team_sync<W>();
            double kk = 0.0;
#pragma unroll
            for (int k = 0; k < NPL; ++k) kk = fma(p[k], var[k] * p[k], kk);
            E = 0.5 * team_sum<W>(kk, lane, red) - lp;
        } else {
            const double es = eps_in[c], dt = 0.5 * es;
            for (int s = 0; s < n_steps; ++s) {
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    const int i = lane + TS * k;
                    p[k] = fma(dt, g_s[i], p[k]);
                    q_s[i] = fma(es, var[k] * p[k], q_s[i]);
                }
                team_sync<W>();
                lp = Model::template eval<NPL, W>(M, smem_raw, q_s, g_s, lane, red);
                team_sync<W>();
                double kk = 0.0;
#pragma unroll
                for (int k = 0; k < NPL; ++k) {
                    p[k] = fma(dt, g_s[lane + TS * k], p[k]);
                    kk = fma(p[k], var[k] * p[k], kk);
                }
                E = 0.5 * team_sum<W>(kk, lane, red) - lp;
            }
            if (lane == 0) idx[c] += (es > 0 ? 1 : (es < 0 ? -1 : 0)) * (long long)n_steps;
        }
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int i = lane + TS * k;
            if (i < n) {
                const long long o = (long long)c * n + i;
                q[o] = q_s[i];
                grad[o] = g_s[i];
                p_io[o] = p[k];
                v_io[o] = var[k] * p[k];
            }
        }
        if (lane == 0) {
            energy[c] = E;
            logp_io[c] = lp;
        }
        team_sync<W>();
    }
}

}  // namespace b200
