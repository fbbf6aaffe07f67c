// Lock-step ("batched leapfrog") NUTS engine for models whose log-density is a dense contraction shared by
// all chains (BASELINE config 3: X.beta over a 1e6 x 128 design matrix; config 5: dense precision / dense mass
// matrix, n = 10^4).  Those chains must meet at a GEMM every leapfrog, so instead of one persistent kernel per
// run the host alternates
//        [ ls_advance_kernel ]  ->  [ batched model evaluation (dense.cuh) ]  ->  [ dense mass GEMM ]  -> ...
// and every chain is a resumable state machine: one call of ls_advance consumes the (logp, grad, Sigma.grad)
// of the position the chain asked for, runs the reference's bookkeeping up to the next gradient request
// (leaf statistics, binary-counter merges with the generalised U-turn checks, multinomial picks, top-level
// doubling, end-of-draw adaptation), writes the next position into the dense request matrix and returns.
// The logic and the order of random-number consumption are those of nuts_warp.cuh (same reference citations:
// hmc/nuts.py:204-489, hmc/integration.py:68-145, hmc/base_hmc.py:196-288, step_sizes.py:41-84,
// hmc/quadpotential.py:211-355 diag-adapt, :680-725 QuadPotentialFull).
//
// Dense mass matrix (QuadPotentialFull): v = Sigma p is a GEMM.  By linearity ONE mass GEMM per leapfrog is
// enough: every state carries w = Sigma.grad, then  v(p + dt g) = v + dt w  and  v(p' ) = v_half + dt w'.
// (The reference does two Sigma.p products per leapfrog, integration.py:124,134; results differ by rounding.)
// p0 = solve_triangular(L^T, z) and v0 = Sigma p0 = L z are batched GEMMs with L^-1 and L^T for the chains that
// start a draw, prefetched one draw ahead so no chain idles.
//
// chain = warp; all vectors live in HBM ([C][n] row-major, coalesced lane-strided loops); the O(n) vector work
// per leaf is negligible next to the O(n^2) or O(N K) contraction.
#pragma once
#include "../../include/b200nuts.h"
#include "common.cuh"
#include "rng.cuh"

namespace b200 {

constexpr int kLsLevels = 12;

// the O(n) vector passes of the advance kernel are latency-bound strided loops: unrolling keeps several loads in flight
constexpr int kLsUnroll = 4;

// A pass over a chain's vectors in tiles of U elements per thread: ALL loads of a tile, then the arithmetic and the stores.
// Written as `for (i) { load; store; }` the compiler must keep every load behind the previous iteration's store (the vectors
// are slots of one allocation, so it cannot rule out aliasing), and the pass runs one DRAM latency per element: measured
// 1.3 TB/s for ls_advance_kernel<16> at n = 10^4 (profiles/r2_tc_launches_mvgauss_tc_summary.csv).  Element order per thread is
// unchanged (i = lane, lane + TS, ...), so every per-thread partial sum keeps its bits.
template <int U, int TS, class Load, class Store>
__device__ __forceinline__ void ls_tiled(int lane, int n, Load&& load, Store&& store) {
    for (int i0 = lane; i0 < n; i0 += TS * U) {
#pragma unroll
        for (int u = 0; u < U; ++u) { const int i = i0 + u * TS; if (i < n) load(u, i); }
#pragma unroll
        for (int u = 0; u < U; ++u) { const int i = i0 + u * TS; if (i < n) store(u, i); }
    }
}

struct LsState {  // per-chain scalars, resident in HBM between calls
    int phase;    // 0 = INIT (waiting for the evaluation at q0), 1 = LEAF (waiting for a leapfrog's evaluation), 2 = DONE,
                  // 3 = MASS (dense mass: a draw is over and the next draw's momentum has not been served yet -- DENSE_ADAPT
                  //     always stops here for the potential's update; a fixed dense mass only when its prefetch is still
                  //     queued, see "deferred momentum" in b200nuts.cu run_lockstep)
    int it, d_iter, maxd, depth, leaf, n_leaf, dir, w_idx, L_idx, R_idx, n_prop, m_pidx, c_pidx;
    int da_count, k_samples, window, fg_m, fg_v, bg_m, bg_v, bad_at, diverged, need_mom, mom_it;
    int prev_update, fa_fg, upd_pending, chol_bad;  // DENSE_ADAPT (dense_adapt.cuh): window start, foreground slot, flags
    int mom_have;  // dense mass: the iteration whose momentum (p0, v0) currently sits in the chain's rows of P0n / V0n
    double eps, E0, accept_sum, max_de, m_logw, m_pe, m_plogp, c_logw, c_pe, c_plogp, cur_logp;
    double log_step, log_bar, hbar, da_mu, fg_n, bg_n;
    unsigned long long rs_hi, rs_lo, ri_hi, ri_lo;
    long long n_grad;
    double sc_logw[kLsLevels], sc_pe[kLsLevels], sc_plogp[kLsLevels];
    int sc_pidx[kLsLevels];
};

// per-chain vector slots (each n doubles)
enum {
    LV_Q = 0, LV_P, LV_G, LV_V, LV_W,                                 // integrator state
    LV_LQ, LV_LP, LV_LG, LV_LV, LV_LW, LV_RQ, LV_RP, LV_RG, LV_RV, LV_RW,  // tree edges
    LV_PS, LV_PQ, LV_PQG, LV_PQW, LV_NEARP, LV_NEARV,                  // main tree
    LV_CLP, LV_CLV, LV_CPS, LV_CPQ, LV_CPQG, LV_CPQW,                  // subtree under construction
    LV_VAR, LV_FGM, LV_FGV, LV_BGM, LV_BGV,                            // diagonal mass + Welford
    LV_STACK                                                           // 8 per level: lp, lv, rp, rv, ps, pq, pqg, pqw
};
__host__ __device__ inline long long ls_vec_count(int levels) { return LV_STACK + 8LL * levels; }

struct LsDev {
    int C, n, tune, draws, max_td, early_td, adapt_step, mass_kind, momentum_source, store_warmup;
    int window, discard, chain_offset, dense;
    double eps0, target, gamma, kappa, t0, Emax, init_weight, logp_const;
    unsigned long long philox_seed;
    const double* q0; const double* var0; const double* mean0; const double* eps0c; const double* z;
    b200_pcg64* rng;
    double* draws_out;
    const signed char* tr_kind; const double* tr_lo; const double* tr_hi;  // record constrained values (common.cuh)
    b200_stats st;
    b200_chain_summary sm;
    LsState* state;
    double* vecs; long long vec_stride;     // per-chain vector block
    long long ld;                              // row stride (doubles) of the request / result matrices: n rounded up to 4
    double* Qreq; double* Greq; double* Wreq;  // dense request / result matrices [C][ld], padding columns stay zero
    double* logp_req;                          // [C] (models that return logp from their own kernel)
    double* P0n; double* V0n;                  // prefetched momentum of the next draw [C][ld] (dense mass)
    int* slot;                                 // [C] row of chain c in the request / result matrices (compaction; null: c)
    int* counters;                             // [0] active chains, [1] chains stalled on their momentum (both per advance),
                                               // [2] momentum requests queued since the last service
    int* mom_list;                             // [C] chains that requested momentum
    int logp_from_dot;                         // 1: logp = logp_const + 0.5 q.g  (Gaussian model)
    // DENSE_ADAPT (QuadPotentialFullAdapt): per-chain matrices [C][n][n] (dense_adapt.cuh)
    double* fa_cov; double* fa_chol; double* fa_raw;  // covariance, its lower Cholesky factor, 2 raw scatter matrices per chain
    int upd_window; double win_mult;
};

// W = warps per chain.  W = 1: four chains per 128-thread CTA (small n); W = 8: chain = CTA, so that the O(n) vector
// passes of a long chain state (n = 10^4) are spread over 256 threads.  All reductions return identical bits to every
// thread of the team (common.cuh), so every thread carries an identical private copy of the scalar state.
template <int W>
__global__ void __launch_bounds__(W == 1 ? 128 : 32 * W) ls_advance_kernel(const LsDev P) {
    constexpr int TS = 32 * W, U = kLsUnroll;
    __shared__ double red_s[W == 1 ? 1 : 8 * W];
    double* red = red_s;
    const int lane = (W == 1) ? (threadIdx.x & 31) : (int)threadIdx.x;  // index inside the team
    const int chain = (W == 1) ? blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) : blockIdx.x;
    if (chain >= P.C) return;
    LsState* SP = P.state + chain;
    if (SP->phase == 2) return;
    LsState S = *SP;  // every lane keeps an identical private copy (all updates are warp-uniform)
    const int n = P.n;
    double* vb = P.vecs + (long long)chain * P.vec_stride;
    auto V = [&](int slot) -> double* { return vb + (long long)slot * n; };
    auto LVL = [&](int h, int which) -> double* { return vb + (long long)(LV_STACK + 8 * h + which) * n; };
    const int row = P.slot ? P.slot[chain] : chain;  // finished chains give their rows up (ls_compact_* below)
    double* qreq = P.Qreq + (long long)row * P.ld;
    const double* greq = P.Greq + (long long)row * P.ld;
    const double* wreq = P.dense ? P.Wreq + (long long)row * P.ld : nullptr;
    const int Ttot = P.tune + P.draws, T_out = P.store_warmup ? Ttot : P.draws;
    Pcg64 rng;
    rng.load(S.rs_hi, S.rs_lo, S.ri_hi, S.ri_lo);
    const bool dense = P.dense != 0;
    const bool fa = P.mass_kind == B200_MASS_DENSE_ADAPT;  // per-chain adaptive dense mass (dense_adapt.cuh)

    // logp of the requested point (Gaussian: from the gradient; otherwise produced by the model kernel)
    auto req_logp = [&]() -> double {
        if (P.logp_from_dot) {
            double s = 0.0;
#pragma unroll kLsUnroll
            for (int i = lane; i < n; i += TS) s = fma(qreq[i], greq[i], s);
            return P.logp_const + 0.5 * team_sum<W>(s, lane, red);
        }
        return P.logp_req[row];
    };

    bool begin_draw = false, next_doubling = false, start_leapfrog = false, finish_draw = false, exhausted = false;

    if (S.phase == 3) {
        // ---- DENSE_ADAPT: the potential has been updated and the draw's momentum is in P0n / V0n ------------------
        begin_draw = true;
    } else if (S.phase == 0) {
        // ---- evaluation at q0 has arrived: the start state of the first draw --------------------------------
        S.cur_logp = req_logp();
#pragma unroll kLsUnroll
        for (int i = lane; i < n; i += TS) {
            V(LV_Q)[i] = qreq[i];
            V(LV_G)[i] = greq[i];
            if (dense) V(LV_W)[i] = wreq[i];
        }
        ++S.n_grad;
        begin_draw = true;
    } else {
        // ---- a leapfrog's evaluation has arrived: second half-kick, energy (integration.py:131-145) ---------
        const double es = S.dir * S.eps, dt = 0.5 * es;
        const double logp = req_logp();
        double kk = 0.0;
        {
            double* p = V(LV_P); double* v = V(LV_V); double* q = V(LV_Q); double* g = V(LV_G); double* w = V(LV_W);
            const double* var = V(LV_VAR);
            double g_[U], p_[U], q_[U], w_[U], v_[U];
            ls_tiled<U, TS>(lane, n,
                [&](int u, int i) {
                    g_[u] = greq[i]; p_[u] = p[i]; q_[u] = qreq[i];
                    if (dense) { w_[u] = wreq[i]; v_[u] = v[i]; } else v_[u] = var[i];
                },
                [&](int u, int i) {
                    const double pi = fma(dt, g_[u], p_[u]);
                    double vi;
                    if (dense) { vi = fma(dt, w_[u], v_[u]); w[i] = w_[u]; }
                    else vi = v_[u] * pi;
                    p[i] = pi; v[i] = vi; g[i] = g_[u]; q[i] = q_[u];
                    kk = fma(pi, vi, kk);
                });
        }
        const double E = 0.5 * team_sum<W>(kk, lane, red) - logp;
        ++S.n_grad;
        S.w_idx += S.dir;
        // ---- _single_step bookkeeping (nuts.py:406-440) ---------------------------------------------------
        ++S.n_prop;
        double dE = E - S.E0;
        if (isnan(dE)) dE = INFINITY;
        S.accept_sum += (dE > 0) ? exp(-dE) : 1.0;
        if (fabs(dE) > fabs(S.max_de)) S.max_de = dE;
        bool sub_div = false, sub_turn = false;
        if (!(dE < P.Emax)) {
            sub_div = true;
        } else {
            // the leaf as a height-0 subtree
            {
                double p_[U], v_[U], q_[U], g_[U], w_[U];
                ls_tiled<U, TS>(lane, n,
                    [&](int u, int i) {
                        p_[u] = V(LV_P)[i]; v_[u] = V(LV_V)[i]; q_[u] = V(LV_Q)[i]; g_[u] = V(LV_G)[i];
                        if (dense) w_[u] = V(LV_W)[i];
                    },
                    [&](int u, int i) {
                        V(LV_CLP)[i] = p_[u]; V(LV_CPS)[i] = p_[u]; V(LV_CLV)[i] = v_[u];
                        V(LV_CPQ)[i] = q_[u]; V(LV_CPQG)[i] = g_[u];
                        if (dense) V(LV_CPQW)[i] = w_[u];
                    });
            }
            S.c_logw = -dE; S.c_pe = E; S.c_plogp = logp; S.c_pidx = S.w_idx;
            // ---- merges while the binary counter carries (nuts.py:452-476) -------------------------------
            int h = 0;
            for (int m = S.leaf; m & 1; m >>= 1, ++h) {
                const double* t_lp = LVL(h, 0); const double* t_lv = LVL(h, 1);
                const double* t_rp = LVL(h, 2); const double* t_rv = LVL(h, 3);
                const double* t_ps = LVL(h, 4);
                double* c_lp = V(LV_CLP); double* c_lv = V(LV_CLV); double* c_ps = V(LV_CPS);
                const double* wp = V(LV_P); const double* wv = V(LV_V);
                double dots[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                {
                    double tl_[U], tlv_[U], tr_[U], trv_[U], tp_[U], cl_[U], clv_[U], cp_[U], vr_[U];
                    ls_tiled<U, TS>(lane, n,
                        [&](int u, int i) {
                            tl_[u] = t_lp[i]; tlv_[u] = t_lv[i]; tr_[u] = t_rp[i]; trv_[u] = t_rv[i]; tp_[u] = t_ps[i];
                            cl_[u] = c_lp[i]; clv_[u] = c_lv[i]; cp_[u] = c_ps[i]; vr_[u] = wv[i];
                        },
                        [&](int u, int i) {
                            const double s = tp_[u] + cp_[u];
                            dots[0] = fma(s, tlv_[u], dots[0]);
                            dots[1] = fma(s, vr_[u], dots[1]);
                            const double s1 = tp_[u] + cl_[u];
                            dots[2] = fma(s1, tlv_[u], dots[2]);
                            dots[3] = fma(s1, clv_[u], dots[3]);
                            const double s2 = tr_[u] + cp_[u];
                            dots[4] = fma(s2, trv_[u], dots[4]);
                            dots[5] = fma(s2, vr_[u], dots[5]);
                            c_lp[i] = tl_[u]; c_lv[i] = tlv_[u]; c_ps[i] = s;
                        });
                    (void)wp;
                }
                team_sum_n<W>(dots, lane, red);
                bool turn = (dots[0] <= 0) || (dots[1] <= 0);
                if (h > 0) turn = turn || (dots[2] <= 0) || (dots[3] <= 0) || (dots[4] <= 0) || (dots[5] <= 0);
                const double t_logw = S.sc_logw[h];
                const double dlw = S.c_logw - t_logw;
                const double e_w = exp(-fabs(dlw));
                const double logw = (dlw == 0.0) ? S.c_logw + 0.69314718055994530942
                                                 : (isnan(dlw) ? S.c_logw + t_logw : fmax(S.c_logw, t_logw) + log1p_abs(e_w));
                const double u = rng.next_double();
                if (!(u * (1.0 + e_w) < (dlw >= 0.0 ? 1.0 : e_w))) {  // keep tree1's proposal
                    const double* t_pq = LVL(h, 5); const double* t_pqg = LVL(h, 6); const double* t_pqw = LVL(h, 7);
                    double a_[U], b_[U], c_[U];
                    ls_tiled<U, TS>(lane, n,
                        [&](int u, int i) { a_[u] = t_pq[i]; b_[u] = t_pqg[i]; if (dense) c_[u] = t_pqw[i]; },
                        [&](int u, int i) { V(LV_CPQ)[i] = a_[u]; V(LV_CPQG)[i] = b_[u]; if (dense) V(LV_CPQW)[i] = c_[u]; });
                    S.c_pe = S.sc_pe[h]; S.c_plogp = S.sc_plogp[h]; S.c_pidx = S.sc_pidx[h];
                }
                S.c_logw = logw;
                if (turn) { sub_turn = true; break; }
            }
            if (!sub_turn && S.leaf + 1 < S.n_leaf) {
                // park the finished subtree (height h) until its right sibling is built
                double r_[8][U];
                ls_tiled<U, TS>(lane, n,
                    [&](int u, int i) {
                        r_[0][u] = V(LV_CLP)[i]; r_[1][u] = V(LV_CLV)[i]; r_[2][u] = V(LV_P)[i]; r_[3][u] = V(LV_V)[i];
                        r_[4][u] = V(LV_CPS)[i]; r_[5][u] = V(LV_CPQ)[i]; r_[6][u] = V(LV_CPQG)[i];
                        if (dense) r_[7][u] = V(LV_CPQW)[i];
                    },
                    [&](int u, int i) {
                        LVL(h, 0)[i] = r_[0][u]; LVL(h, 1)[i] = r_[1][u]; LVL(h, 2)[i] = r_[2][u]; LVL(h, 3)[i] = r_[3][u];
                        LVL(h, 4)[i] = r_[4][u]; LVL(h, 5)[i] = r_[5][u]; LVL(h, 6)[i] = r_[6][u];
                        if (dense) LVL(h, 7)[i] = r_[7][u];
                    });
                S.sc_logw[h] = S.c_logw; S.sc_pe[h] = S.c_pe; S.sc_plogp[h] = S.c_plogp; S.sc_pidx[h] = S.c_pidx;
            }
        }
        ++S.leaf;
        if (!sub_div && !sub_turn && S.leaf < S.n_leaf) {
            start_leapfrog = true;  // next leaf of the same subtree
        } else {
            // ---- the doubling is over (completed, diverged or turned) ------------------------------------
            ++S.depth;
            if (sub_div || sub_turn) {
                S.diverged = sub_div ? 1 : 0;
                finish_draw = true;
            } else {
                const int dir = S.dir;
                // new outer edge = integrator state
                {
                    const int b = dir > 0 ? LV_RQ : LV_LQ;
                    double r_[5][U];
                    ls_tiled<U, TS>(lane, n,
                        [&](int u, int i) {
                            r_[0][u] = V(LV_Q)[i]; r_[1][u] = V(LV_P)[i]; r_[2][u] = V(LV_G)[i]; r_[3][u] = V(LV_V)[i];
                            if (dense) r_[4][u] = V(LV_W)[i];
                        },
                        [&](int u, int i) {
                            V(b + 0)[i] = r_[0][u]; V(b + 1)[i] = r_[1][u]; V(b + 2)[i] = r_[2][u]; V(b + 3)[i] = r_[3][u];
                            if (dense) V(b + 4)[i] = r_[4][u];
                        });
                    if (dir > 0) S.R_idx = S.w_idx; else S.L_idx = S.w_idx;
                }
                // biased progressive pick (nuts.py:370-374)
                {
                    const double u = rng.next_double();
                    const double dlw = S.c_logw - S.m_logw;
                    const double e_w = exp(-fabs(dlw));
                    if (dlw >= 0.0 || u < e_w) {
                        double a_[U], b_[U], c_[U];
                        ls_tiled<U, TS>(lane, n,
                            [&](int u, int i) { a_[u] = V(LV_CPQ)[i]; b_[u] = V(LV_CPQG)[i]; if (dense) c_[u] = V(LV_CPQW)[i]; },
                            [&](int u, int i) { V(LV_PQ)[i] = a_[u]; V(LV_PQG)[i] = b_[u]; if (dense) V(LV_PQW)[i] = c_[u]; });
                        S.m_pe = S.c_pe; S.m_plogp = S.c_plogp; S.m_pidx = S.c_pidx;
                    }
                    S.m_logw = (dlw == 0.0) ? S.c_logw + 0.69314718055994530942
                                            : (isnan(dlw) ? S.c_logw + S.m_logw : fmax(S.c_logw, S.m_logw) + log1p_abs(e_w));
                }
                // U-turn checks on the whole tree (nuts.py:376-390)
                {
                    const double* farp = V(dir > 0 ? LV_LP : LV_RP); const double* farv = V(dir > 0 ? LV_LV : LV_RV);
                    const double* nearp = V(LV_NEARP); const double* nearv = V(LV_NEARV);
                    double* PS = V(LV_PS);
                    const double* cps = V(LV_CPS); const double* clp = V(LV_CLP); const double* clv = V(LV_CLV);
                    const double* wv = V(LV_V);
                    double dots[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                    {
                        double so_[U], cp_[U], vf_[U], vw_[U], cl_[U], clv_[U], np_[U], nv_[U];
                        ls_tiled<U, TS>(lane, n,
                            [&](int u, int i) {
                                so_[u] = PS[i]; cp_[u] = cps[i]; vf_[u] = farv[i]; vw_[u] = wv[i];
                                cl_[u] = clp[i]; clv_[u] = clv[i]; np_[u] = nearp[i]; nv_[u] = nearv[i];
                            },
                            [&](int u, int i) {
                                const double s = so_[u] + cp_[u];
                                PS[i] = s;
                                dots[0] = fma(s, vf_[u], dots[0]);
                                dots[1] = fma(s, vw_[u], dots[1]);
                                const double a = so_[u] + cl_[u];
                                dots[2] = fma(a, vf_[u], dots[2]);
                                dots[3] = fma(a, clv_[u], dots[3]);
                                const double b = np_[u] + cp_[u];
                                dots[4] = fma(b, nv_[u], dots[4]);
                                dots[5] = fma(b, vw_[u], dots[5]);
                            });
                        (void)farp;
                    }
                    team_sum_n<W>(dots, lane, red);
                    const bool turn = (dots[0] <= 0) || (dots[1] <= 0) || (dots[2] <= 0) || (dots[3] <= 0) ||
                                      (dots[4] <= 0) || (dots[5] <= 0);
                    if (turn) finish_draw = true;                                   // `break` in nuts.py:218-219
                    else if (++S.d_iter >= S.maxd) { finish_draw = true; exhausted = true; }  // for/else, nuts.py:220-221
                    else next_doubling = true;
                }
            }
        }
    }

    // ------------------------------------------------------------------------------------------------------
    if (finish_draw) {
        const bool tuning = S.it < P.tune;
        const bool adapting = tuning && P.adapt_step;
        const bool hit_max = exhausted ? !tuning : false;
        const double accept = S.accept_sum / S.n_prop;
        const bool rec = P.store_warmup || !tuning;
        const int t_out = P.store_warmup ? S.it : S.it - P.tune;
        // accepted position (+ its gradient, Sigma.gradient and logp) becomes the chain state
        {
            double a_[U], b_[U], c_[U];
            ls_tiled<U, TS>(lane, n,
                [&](int u, int i) { a_[u] = V(LV_PQ)[i]; b_[u] = V(LV_PQG)[i]; if (dense) c_[u] = V(LV_PQW)[i]; },
                [&](int u, int i) {
                    V(LV_Q)[i] = a_[u]; V(LV_G)[i] = b_[u];
                    if (dense) V(LV_W)[i] = c_[u];
                    if (rec) P.draws_out[((long long)chain * T_out + t_out) * n + i] = constrained(a_[u], i, P.tr_kind, P.tr_lo, P.tr_hi);
                });
        }
        S.cur_logp = S.m_plogp;
        if (adapting) {  // step_sizes.py:66-78
            const double w = 1.0 / (S.da_count + P.t0);
            S.hbar = __dadd_rn(__dmul_rn(1.0 - w, S.hbar), __dmul_rn(w, P.target - accept));
            S.log_step = S.da_mu - __dmul_rn(S.hbar, sqrt((double)S.da_count)) / P.gamma;
            const double mk = pow((double)S.da_count, -P.kappa);
            S.log_bar = __dadd_rn(__dmul_rn(mk, S.log_step), __dmul_rn(1.0 - mk, S.log_bar));
            ++S.da_count;
        }
        if (tuning && P.mass_kind == B200_MASS_DIAG_ADAPT) {  // quadpotential.py:335-355
            if (S.k_samples > P.discard) {
                S.fg_n += 1.0; S.bg_n += 1.0;
                double* fm = V(S.fg_m); double* fv = V(S.fg_v); double* bm = V(S.bg_m); double* bv = V(S.bg_v);
                double x_[U], fm_[U], fv_[U], bm_[U], bv_[U];
                ls_tiled<U, TS>(lane, n,
                    [&](int u, int i) { x_[u] = V(LV_Q)[i]; fm_[u] = fm[i]; fv_[u] = fv[i]; bm_[u] = bm[i]; bv_[u] = bv[i]; },
                    [&](int u, int i) {
                        const double x = x_[u];
                        double mean = fm_[u], d0 = x - mean;
                        mean = __dadd_rn(mean, d0 / S.fg_n); fm[i] = mean;
                        fv[i] = __dadd_rn(fv_[u], __dmul_rn(d0, x - mean));
                        mean = bm_[u]; d0 = x - mean;
                        mean = __dadd_rn(mean, d0 / S.bg_n); bm[i] = mean;
                        bv[i] = __dadd_rn(bv_[u], __dmul_rn(d0, x - mean));
                    });
            }
            if (S.k_samples > S.window) {
                const double* fv = V(S.fg_v);
                double f_[U];
                ls_tiled<U, TS>(lane, n, [&](int u, int i) { f_[u] = fv[i]; },
                                [&](int u, int i) { V(LV_VAR)[i] = fmin(fmax(f_[u] / S.fg_n, 1e-12), 1e12); });
            }
            if (S.k_samples > 0 && S.k_samples % S.window == 0) {
                const int tm = S.fg_m, tv = S.fg_v;
                S.fg_m = S.bg_m; S.fg_v = S.bg_v; S.fg_n = S.bg_n;
                S.bg_m = tm; S.bg_v = tv; S.bg_n = 0.0;
#pragma unroll kLsUnroll
                for (int i = lane; i < n; i += TS) { V(S.bg_m)[i] = 0.0; V(S.bg_v)[i] = 0.0; }
            }
            ++S.k_samples;
        }
        if (rec && lane == 0) {
            const long long o = (long long)chain * T_out + t_out;
            if (P.st.depth) P.st.depth[o] = S.depth;
            if (P.st.tree_size) P.st.tree_size[o] = S.n_prop;
            if (P.st.index_in_trajectory) P.st.index_in_trajectory[o] = S.m_pidx;
            if (P.st.diverging) P.st.diverging[o] = S.diverged ? 1 : 0;
            if (P.st.reached_max_treedepth) P.st.reached_max_treedepth[o] = hit_max ? 1 : 0;
            if (P.st.step_size) P.st.step_size[o] = exp(S.log_step);
            if (P.st.step_size_bar) P.st.step_size_bar[o] = exp(S.log_bar);
            if (P.st.mean_tree_accept) P.st.mean_tree_accept[o] = accept;
            if (P.st.energy) P.st.energy[o] = S.m_pe;
            if (P.st.energy_error) P.st.energy_error[o] = S.m_pe - S.E0;
            if (P.st.max_energy_error) P.st.max_energy_error[o] = S.max_de;
            if (P.st.model_logp) P.st.model_logp[o] = S.m_plogp;
        }
        ++S.it;
        if (S.it >= Ttot) S.phase = 2;
        else if (fa) {
            // potential.update(sample, grad, tune) (base_hmc.py:238) then potential.random() of the next draw: both need the
            // chain's n x n matrices, so they run in fa_update_momentum_kernel between two advance calls
            S.phase = 3; S.need_mom = 1; S.mom_it = S.it; S.upd_pending = tuning ? 1 : 0;
        } else begin_draw = true;
    }

    bool stalled = false;
    if (begin_draw && S.phase != 2 && dense && S.mom_have != S.it) {
        // the draw's momentum is still in the request queue (the host serves requests in batches): wait one round
        S.phase = 3;
        begin_draw = false;
        stalled = true;
    }
    if (begin_draw && S.phase != 2) {
        team_sync<W>();
        const bool tuning = S.it < P.tune;
        const bool adapting = tuning && P.adapt_step;
        // ---- p0 = potential.random(); v0 (quadpotential.py:323-326, :619, :710-713) -------------------------
        double kin = 0.0;
        {
            double* p = V(LV_P); double* v = V(LV_V);
            if (dense) {
                const double* p0 = P.P0n + (long long)chain * P.ld; const double* v0 = P.V0n + (long long)chain * P.ld;
                double a_[U], b_[U];
                ls_tiled<U, TS>(lane, n, [&](int u, int i) { a_[u] = p0[i]; b_[u] = v0[i]; },
                                [&](int u, int i) { p[i] = a_[u]; v[i] = b_[u]; kin = fma(a_[u], b_[u], kin); });
            } else {
                const double* var = V(LV_VAR);
#pragma unroll kLsUnroll
                for (int i = lane; i < n; i += TS) {
                    const double zz = (P.momentum_source == B200_MOMENTUM_HOST_BUFFER)
                                          ? P.z[((long long)chain * Ttot + S.it) * n + i]
                                          : philox_normal(P.philox_seed, (uint32_t)(chain + P.chain_offset), (uint32_t)S.it, (uint32_t)i);
                    const double pi = (1.0 / sqrt(var[i])) * zz, vi = var[i] * pi;
                    p[i] = pi; v[i] = vi; kin = fma(pi, vi, kin);
                }
            }
        }
        S.E0 = 0.5 * team_sum<W>(kin, lane, red) - S.cur_logp;
        // a failed Cholesky (quadpotential.py:812-816, raise_ok :845-847 raises before the next draw) freezes the chain too
        if (!isfinite(S.E0) || S.chol_bad) {  // "Bad initial energy" (base_hmc.py:205-224): freeze; the iterations that never ran are NaN
            S.bad_at = S.it;
            S.phase = 2;
            for (int t = S.it; t < Ttot; ++t) {
                if (!(P.store_warmup || t >= P.tune)) continue;
                const int t_o = P.store_warmup ? t : t - P.tune;
#pragma unroll kLsUnroll
                for (int i = lane; i < n; i += TS) P.draws_out[((long long)chain * T_out + t_o) * n + i] = nan("");
                if (lane == 0) stats_sentinel(P.st, (long long)chain * T_out + t_o);
            }
        } else {
            S.eps = exp(adapting ? S.log_step : S.log_bar);
            S.maxd = (tuning && S.it < 200) ? P.early_td : P.max_td;
            {
                double q_[U], p_[U], g_[U], v_[U], w_[U];
                ls_tiled<U, TS>(lane, n,
                    [&](int u, int i) {
                        q_[u] = V(LV_Q)[i]; p_[u] = V(LV_P)[i]; g_[u] = V(LV_G)[i]; v_[u] = V(LV_V)[i];
                        if (dense) w_[u] = V(LV_W)[i];
                    },
                    [&](int u, int i) {
                        const double qi = q_[u], pi = p_[u], gi = g_[u], vi = v_[u];
                        V(LV_LQ)[i] = qi; V(LV_RQ)[i] = qi; V(LV_PQ)[i] = qi;
                        V(LV_LP)[i] = pi; V(LV_RP)[i] = pi; V(LV_PS)[i] = pi;
                        V(LV_LG)[i] = gi; V(LV_RG)[i] = gi; V(LV_PQG)[i] = gi;
                        V(LV_LV)[i] = vi; V(LV_RV)[i] = vi;
                        if (dense) { const double wi = w_[u]; V(LV_LW)[i] = wi; V(LV_RW)[i] = wi; V(LV_PQW)[i] = wi; }
                    });
            }
            S.L_idx = S.R_idx = 0;
            S.m_logw = 0.0; S.m_pe = S.E0; S.m_plogp = S.cur_logp; S.m_pidx = 0;
            S.accept_sum = 0.0; S.max_de = 0.0; S.n_prop = 0; S.depth = 0; S.diverged = 0; S.d_iter = 0;
            if (dense && !fa && S.it + 1 < Ttot) { S.need_mom = 1; S.mom_it = S.it + 1; }  // prefetch the next draw's momentum
            next_doubling = true;
        }
    }

    if (next_doubling) {
        team_sync<W>();
        S.dir = (rng.next_double() < 0.5) ? 1 : -1;  // nuts.py:215
        const int b = S.dir > 0 ? LV_RQ : LV_LQ;
        {
            double r_[5][U];
            ls_tiled<U, TS>(lane, n,
                [&](int u, int i) {
                    r_[0][u] = V(b + 0)[i]; r_[1][u] = V(b + 1)[i]; r_[2][u] = V(b + 2)[i]; r_[3][u] = V(b + 3)[i];
                    if (dense) r_[4][u] = V(b + 4)[i];
                },
                [&](int u, int i) {
                    V(LV_Q)[i] = r_[0][u]; V(LV_P)[i] = r_[1][u]; V(LV_G)[i] = r_[2][u]; V(LV_V)[i] = r_[3][u];
                    if (dense) V(LV_W)[i] = r_[4][u];
                    V(LV_NEARP)[i] = r_[1][u]; V(LV_NEARV)[i] = r_[3][u];
                });
        }
        S.w_idx = S.dir > 0 ? S.R_idx : S.L_idx;
        S.leaf = 0;
        S.n_leaf = 1 << S.depth;
        start_leapfrog = true;
    }

    if (start_leapfrog) {
        team_sync<W>();
        // first half-kick and drift (integration.py:118-127); the gradient at the new position is requested
        const double es = S.dir * S.eps, dt = 0.5 * es;
        double* p = V(LV_P); double* v = V(LV_V);
        const double* q = V(LV_Q); const double* g = V(LV_G); const double* w = V(LV_W); const double* var = V(LV_VAR);
        double g_[U], p_[U], q_[U], w_[U], v_[U];
        ls_tiled<U, TS>(lane, n,
            [&](int u, int i) {
                g_[u] = g[i]; p_[u] = p[i]; q_[u] = q[i];
                if (dense) { w_[u] = w[i]; v_[u] = v[i]; } else v_[u] = var[i];
            },
            [&](int u, int i) {
                const double pi = fma(dt, g_[u], p_[u]);
                const double vi = dense ? fma(dt, w_[u], v_[u]) : v_[u] * pi;
                p[i] = pi; v[i] = vi;
                qreq[i] = fma(es, vi, q_[u]);
            });
        S.phase = 1;
    }

    // ---- persist --------------------------------------------------------------------------------------------
    S.rs_hi = (unsigned long long)(rng.state >> 64); S.rs_lo = (unsigned long long)rng.state;
    if (lane == 0) {
        if (S.phase != 2) atomicAdd(&P.counters[0], 1);
        if (stalled) atomicAdd(&P.counters[1], 1);
        if (S.need_mom) { const int j = atomicAdd(&P.counters[2], 1); P.mom_list[j] = chain; }
        if (S.phase == 2) {
            b200_pcg64 r;
            r.state_hi = S.rs_hi; r.state_lo = S.rs_lo; r.inc_hi = S.ri_hi; r.inc_lo = S.ri_lo;
            P.rng[chain] = r;
            if (P.sm.grad_evals) P.sm.grad_evals[chain] = S.n_grad;
            if (P.sm.bad_energy_at) P.sm.bad_energy_at[chain] = S.bad_at;
            if (P.sm.final_step_size) P.sm.final_step_size[chain] = exp(S.log_bar);
        }
        S.need_mom = 0;  // the host serves the request before the next advance
        *SP = S;
    }
    if (S.phase == 2 && P.sm.final_var)
#pragma unroll kLsUnroll
        for (int i = lane; i < n; i += TS) P.sm.final_var[(long long)chain * n + i] = V(LV_VAR)[i];
    if (S.phase == 2 && fa && P.sm.final_cov) {
        const long long nn = (long long)n * n;
        for (long long i = lane; i < nn; i += TS) P.sm.final_cov[chain * nn + i] = P.fa_cov[chain * nn + i];
    }
}

// one-time initialisation of the per-chain state; requests the evaluation at q0 (and the first momentum)
__global__ void __launch_bounds__(128) ls_init_kernel(const LsDev P) {
    const int lane = threadIdx.x & 31;
    const int chain = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (chain >= P.C) return;
    const int n = P.n;
    double* vb = P.vecs + (long long)chain * P.vec_stride;
    for (int i = lane; i < n; i += 32) {
        P.Qreq[(long long)chain * P.ld + i] = P.q0[(long long)chain * n + i];
        const double var = P.var0 ? P.var0[(long long)chain * n + i] : 1.0;
        vb[(long long)LV_VAR * n + i] = var;
        vb[(long long)LV_FGM * n + i] = P.mean0 ? P.mean0[(long long)chain * n + i] : 0.0;
        vb[(long long)LV_FGV * n + i] = var * P.init_weight;
        vb[(long long)LV_BGM * n + i] = 0.0;
        vb[(long long)LV_BGV * n + i] = 0.0;
    }
    if (lane == 0) {
        LsState S;
        memset(&S, 0, sizeof(S));
        S.phase = 0;
        S.bad_at = -1;
        const double e0 = P.eps0c ? P.eps0c[chain] : P.eps0;
        S.log_step = log(e0); S.log_bar = S.log_step; S.hbar = 0.0; S.da_mu = log(10.0 * e0); S.da_count = 1;
        S.window = P.window; S.fg_m = LV_FGM; S.fg_v = LV_FGV; S.bg_m = LV_BGM; S.bg_v = LV_BGV;
        S.prev_update = 0; S.fa_fg = 0; S.upd_pending = 0; S.chol_bad = 0; S.mom_have = -1;
        S.fg_n = P.init_weight; S.bg_n = 0.0;
        const b200_pcg64 r = P.rng[chain];
        S.rs_hi = r.state_hi; S.rs_lo = r.state_lo; S.ri_hi = r.inc_hi; S.ri_lo = r.inc_lo;
        if (P.dense) { S.need_mom = 0; S.mom_it = 0; P.mom_list[chain] = chain; }
        if (P.slot) P.slot[chain] = chain;
        P.state[chain] = S;
    }
}

// ---- compaction of the request rows -------------------------------------------------------------------------------------
// Chains finish at different times (a few warm-up trees of depth 10 decide a chain's total), and the batched evaluation costs
// the same for a finished chain's row as for a live one.  When enough chains have finished to free a whole tile of rows, the
// live chains are renumbered to consecutive rows (in chain order) and the batch shrinks.  Two kernels: the new row of every
// chain (one CTA, ballot scan), then the move of the pending request rows into the other request matrix.
__global__ void __launch_bounds__(1024) ls_compact_slots_kernel(const LsDev P, int* new_slot) {
    __shared__ int warp_tot[32];
    __shared__ int carry;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < P.C; base += 1024) {
        const int c = base + (int)threadIdx.x;
        const int live = (c < P.C && P.state[c].phase != 2) ? 1 : 0;
        const unsigned b = __ballot_sync(0xffffffffu, live);
        if (lane == 0) warp_tot[w] = __popc(b);
        __syncthreads();
        int off = carry;
        for (int j = 0; j < w; ++j) off += warp_tot[j];
        if (c < P.C) new_slot[c] = live ? off + __popc(b & ((1u << lane) - 1u)) : -1;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int j = 0; j < 32; ++j) t += warp_tot[j];
            carry += t;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) ls_compact_move_kernel(const LsDev P, const int* new_slot, double* Qnew) {
    const int chain = blockIdx.x;
    const int ns = new_slot[chain];
    if (ns < 0) return;
    const double* src = P.Qreq + (long long)P.slot[chain] * P.ld;
    double* dst = Qnew + (long long)ns * P.ld;
    for (long long i = threadIdx.x; i < P.ld; i += blockDim.x) dst[i] = src[i];
    __syncthreads();
    if (threadIdx.x == 0) P.slot[chain] = ns;
}

// z rows of the chains that asked for momentum -> dense batch Zb[m][ld]
__global__ void __launch_bounds__(256) ls_gather_z_kernel(const LsDev P, int m, double* Zb) {
    const int j = blockIdx.x;
    if (j >= m) return;
    const int chain = P.mom_list[j];
    const int it = P.state[chain].mom_it;
    const int n = P.n, Ttot = P.tune + P.draws;
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        Zb[(long long)j * P.ld + i] = (P.momentum_source == B200_MOMENTUM_HOST_BUFFER)
                                       ? P.z[((long long)chain * Ttot + it) * n + i]
                                       : philox_normal(P.philox_seed, (uint32_t)(chain + P.chain_offset), (uint32_t)it, (uint32_t)i);
}
__global__ void __launch_bounds__(256) ls_scatter_mom_kernel(const LsDev P, int m, const double* P0b, const double* V0b) {
    const int j = blockIdx.x;
    if (j >= m) return;
    const int chain = P.mom_list[j];
    const int n = P.n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        P.P0n[(long long)chain * P.ld + i] = P0b[(long long)j * P.ld + i];
        P.V0n[(long long)chain * P.ld + i] = V0b[(long long)j * P.ld + i];
    }
    if (threadIdx.x == 0) P.state[chain].mom_have = P.state[chain].mom_it;
}

}  // namespace b200
