// libb200nuts.so -- C ABI implementation (see include/b200nuts.h for the contract and the reference
// interfaces each entry point replaces).  Host side: model preparation (data re-layout for coalesced,
// lane-balanced access), staging of host buffers, kernel dispatch on (model kind, elements per lane).
#include "../../include/b200nuts.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <numeric>
#include <string>
#include <type_traits>
#include <chrono>
#include <vector>

#include "dense.cuh"
#include "ir_model.cuh"
#include "logistic_tc.cuh"
#include "gemm_tc.cuh"
#include "lockstep.cuh"
#include "dense_adapt.cuh"
#include "models.cuh"
#include "nuts_warp.cuh"

using namespace b200;

// ------------------------------------------------------------------------------------------------
// error plumbing: no exception crosses the ABI
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local double g_last_ms = 0.0;
static thread_local int g_last_launches = 0;

static int fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return -1;
}
#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                           __FILE__, __LINE__);                                   \
    } while (0)

struct DevBuf {  // owning device allocation
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16); }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

struct b200_model {
    int kind = 0, n = 0, device = 0;
    std::vector<void*> owned;  // device allocations
    StdNormalModel::Params std_normal{};
    EightSchoolsModel::Params eight{};
    RadonModel::Params radon{};
    StochVolModel::Params stochvol{};
    const signed char* tr_kind = nullptr;  // per-element backward transforms (b200_model_set_transforms)
    const double* tr_lo = nullptr;
    const double* tr_hi = nullptr;
    IrModel::Params ir{};
    long long ir_max_obs = 0;
    void* ir_scratch = nullptr;   // per-team scratch of the generic IR device function: [slots][n_pad + max N] doubles
    size_t ir_scratch_bytes = 0;
    cudaError_t ensure_ir_scratch(long long slots) {
        const size_t bytes = (size_t)slots * (size_t)ir.stride * sizeof(double);
        if (bytes > ir_scratch_bytes) {
            if (ir_scratch) cudaFree(ir_scratch);
            ir_scratch = nullptr;
            ir_scratch_bytes = 0;
            cudaError_t e = cudaMalloc(&ir_scratch, bytes);
            if (e != cudaSuccess) return e;
            ir_scratch_bytes = bytes;
        }
        ir.scratch = static_cast<double*>(ir_scratch);
        return cudaSuccess;
    }
    // lock-step (GEMM-shaped) models; every matrix is row-major with rows `ld` doubles apart (n rounded up to 4, zero pad)
    long long ld = 0;
    const double* prec = nullptr;   // MVGAUSS: precision P [n][ld]
    // dense mass matrix of ANY model (b200_model_set_dense_mass; MVGAUSS sets it from its own covariance at create)
    const double* cov = nullptr;    // velocity:  v = cov p            (QuadPotentialFull: Sigma; FullInv: A^-1)   [n][ld]
    const double* linvT = nullptr;  // momentum:  p0 = linvT z         (Full: L^-T, L = chol(Sigma); FullInv: chol(A))
    const double* chol = nullptr;   // its velocity: v0 = chol z       (Full: L;    FullInv: chol(A)^-T)
    double logp_const = 0.0;
    const double* X = nullptr;      // LOGISTIC: design matrix [Npad][KP] row-major, zero padded (KP = 8, 32 or 128)
    const uint8_t* y8 = nullptr;    // LOGISTIC: y[N]
    long long n_rows = 0;
    int KP = 0;
    // LOGISTIC, tensor-core performance mode (csrc/logistic_tc.cuh): fp16 hi/lo pieces of X and their TMA tensor maps
    int precision = B200_PRECISION_FP64;
    const __half* Xh = nullptr;
    const __half* Xl = nullptr;
    const float* y32 = nullptr;
    long long tc_slabs = 0;
    CUtensorMap map_hi{}, map_lo{};
    // dense Gaussian, tensor-core performance mode (csrc/gemm_tc.cuh): fp16 pieces of the n x n matrices (B operands) and the
    // per-call pieces of the chains' vectors (A operand)
    struct TcMat { const double* src = nullptr; const __half* hi = nullptr; const __half* lo = nullptr; CUtensorMap map_hi{}, map_lo{}; };
    TcMat tc_mats[4];
    long long tc_kpad = 0, tc_npad = 0;
    __half* tc_a_hi = nullptr; __half* tc_a_lo = nullptr;   // [tc_a_rows][tc_kpad]
    long long tc_a_rows = 0;
    // per-chain tree scratch of the persistent kernel, kept between runs (cudaMalloc/cudaFree of 100+ MB per call costs
    // tens of milliseconds of host time on the end-to-end path)
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    void* ls_arena = nullptr;  // lock-step engine: per-chain state machines, vectors, request matrices (kept between runs)
    size_t ls_arena_bytes = 0;
    cudaError_t ensure_ls_arena(size_t bytes) {
        if (bytes <= ls_arena_bytes) return cudaSuccess;
        if (ls_arena) cudaFree(ls_arena);
        ls_arena = nullptr;
        ls_arena_bytes = 0;
        cudaError_t e = cudaMalloc(&ls_arena, bytes);
        if (e == cudaSuccess) ls_arena_bytes = bytes;
        return e;
    }
    void* stage_arena = nullptr;  // device staging of per-draw sampler statistics bound for host memory (kept between runs)
    size_t stage_bytes = 0;
    cudaError_t ensure_stage(size_t bytes) {
        if (bytes <= stage_bytes) return cudaSuccess;
        if (stage_arena) cudaFree(stage_arena);
        stage_arena = nullptr;
        stage_bytes = 0;
        cudaError_t e = cudaMalloc(&stage_arena, bytes);
        if (e == cudaSuccess) stage_bytes = bytes;
        return e;
    }
    cudaError_t ensure_scratch(size_t bytes) {
        if (bytes <= scratch_bytes) return cudaSuccess;
        if (scratch) cudaFree(scratch);
        scratch = nullptr;
        scratch_bytes = 0;
        cudaError_t e = cudaMalloc(&scratch, bytes);
        if (e == cudaSuccess) scratch_bytes = bytes;
        return e;
    }
    ~b200_model() {
        if (ls_arena) cudaFree(ls_arena);
        if (stage_arena) cudaFree(stage_arena);
        if (tc_a_hi) cudaFree(tc_a_hi);
        if (tc_a_lo) cudaFree(tc_a_lo);
        if (ir_scratch) cudaFree(ir_scratch);
        if (scratch) cudaFree(scratch);
        for (void* p : owned) cudaFree(p);
    }
};

static bool is_lockstep_kind(int kind);
template <class F> static int dispatch(const b200_model* m, F&& f);
static int lockstep_logp(b200_model* m, const double* q_dev, int C, double* logp_dev, double* grad_dev, cudaStream_t st);

template <class T>
static int upload(b200_model* m, const std::vector<T>& h, const T** out) {
    void* d = nullptr;
    CU(cudaMalloc(&d, std::max<size_t>(h.size() * sizeof(T), 16)));
    m->owned.push_back(d);
    if (!h.empty()) CU(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<const T*>(d);
    return 0;
}

extern "C" int b200_version(void) { return B200NUTS_VERSION; }
extern "C" const char* b200_last_error(void) { return g_err.c_str(); }
extern "C" int b200_struct_size(int which) {
    switch (which) {
        case 0: return (int)sizeof(b200_model_desc);
        case 1: return (int)sizeof(b200_nuts_cfg);
        case 2: return (int)sizeof(b200_stats);
        case 3: return (int)sizeof(b200_chain_summary);
        case 4: return (int)sizeof(b200_pcg64);
        case 5: return (int)sizeof(b200_ir);
        case 6: return (int)sizeof(b200_ir_var);
        case 7: return (int)sizeof(b200_ir_prior);
        case 8: return (int)sizeof(b200_ir_term);
        case 9: return (int)sizeof(b200_ir_lik);
        case 10: return (int)sizeof(b200_ir_ar1);
        case 11: return (int)sizeof(b200_ir_param);
        case 12: return (int)sizeof(b200_ir_factor);
        case 13: return (int)sizeof(b200_chain_state);
        default: return -1;
    }
}

extern "C" int b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int b200_set_device(int device) {
    CU(cudaSetDevice(device));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// model creation: "compile" step.  Re-lays the observed data out for the device functions.
// ------------------------------------------------------------------------------------------------
static int prepare_radon(b200_model* m, const b200_model_desc* d) {
    const int J = d->n_groups;
    const long long N = d->n_obs;
    if (J <= 0 || N <= 0 || !d->x || !d->y || !d->idx) return fail("radon: missing data");
    if (d->n != 2 * J + 5) return fail("radon: n=%d but 2*n_groups+5=%d", d->n, 2 * J + 5);
    if (J > 0xffff) return fail("radon: n_groups > 65535 unsupported");
    std::vector<std::vector<int>> members(J);
    for (long long i = 0; i < N; ++i) {
        const int c = d->idx[i];
        if (c < 0 || c >= J) return fail("radon: county_idx[%lld]=%d out of range", i, c);
        members[c].push_back((int)i);
    }
    // counties sorted by size; row j = counties order[32j .. 32j+31], one per lane, padded to the row's longest
    std::vector<int> order;
    std::vector<int> empty;
    for (int c = 0; c < J; ++c) (members[c].empty() ? empty : order).push_back(c);
    std::stable_sort(order.begin(), order.end(),
                     [&](int a, int b) { return members[a].size() > members[b].size(); });
    const int M = std::max<int>(1, ((int)order.size() + 31) / 32);
    std::vector<int32_t> seg((size_t)M * 32 + ((M + 3) & ~3), 0);
    for (size_t i = 0; i < (size_t)M * 32; ++i) seg[i] = 0xffff;  // idle lane
    int K = 0;
    std::vector<int> row_off(M, 0), row_len(M, 0);
    for (int j = 0; j < M; ++j) {
        row_off[j] = K;
        for (int l = 0; l < 32 && (size_t)(j * 32 + l) < order.size(); ++l)
            row_len[j] = std::max<int>(row_len[j], (int)members[order[j * 32 + l]].size());
        row_len[j] = (row_len[j] + 3) & ~3;  // whole blocks of 4 observations
        K += row_len[j];
    }
    K += 4;  // the block the kernel prefetches past the last row
    if (K >= 0xffff) return fail("radon: padded observation rows exceed 65534");
    std::vector<double2> xy((size_t)K * 32, make_double2(0.0, 0.0));
    for (int j = 0; j < M; ++j) {
        for (int l = 0; l < 32 && (size_t)(j * 32 + l) < order.size(); ++l) {
            const int c = order[j * 32 + l];
            int k = row_off[j];
            for (int i : members[c]) xy[(size_t)(k++) * 32 + l] = make_double2(d->x[i], d->y[i]);
            seg[(size_t)j * 32 + l] = ((int32_t)members[c].size() << 16) | c;
        }
        seg[(size_t)M * 32 + j] = (row_off[j] << 16) | (row_len[j] / 4);
    }
    RadonModel::Params& P = m->radon;
    P.K = K; P.M = M; P.J = J; P.n_obs = (int)N; P.E = (int)empty.size();
    if (upload(m, xy, &P.xy)) return -1;
    if (upload(m, seg, &P.seg)) return -1;
    if (upload(m, empty, &P.empty)) return -1;
    return 0;
}

static int prepare_eight(b200_model* m, const b200_model_desc* d) {
    const int J = (int)d->n_obs;
    if (J <= 0 || !d->y || !d->aux) return fail("eight_schools: missing data");
    if (d->n != J + 2) return fail("eight_schools: n=%d but J+2=%d", d->n, J + 2);
    std::vector<double> y(d->y, d->y + J), is2(J), ls(J);
    for (int j = 0; j < J; ++j) {
        if (!(d->aux[j] > 0)) return fail("eight_schools: sigma[%d] must be > 0", j);
        is2[j] = 1.0 / (d->aux[j] * d->aux[j]);
        ls[j] = std::log(d->aux[j]);
    }
    EightSchoolsModel::Params& P = m->eight;
    P.J = J;
    if (upload(m, y, &P.y)) return -1;
    if (upload(m, is2, &P.inv_s2)) return -1;
    if (upload(m, ls, &P.log_s)) return -1;
    return 0;
}

static int prepare_stochvol(b200_model* m, const b200_model_desc* d) {
    const int T = (int)d->n_obs;
    if (T < 2 || !d->y) return fail("stochvol: missing data");
    if (d->n != T + 3) return fail("stochvol: n=%d but T+3=%d", d->n, T + 3);
    std::vector<double> y2(T);
    for (int t = 0; t < T; ++t) y2[t] = d->y[t] * d->y[t];
    m->stochvol.T = T;
    return upload(m, y2, &m->stochvol.y2);
}

template <class T>
static int upload_raw(b200_model* m, const T* h, size_t count, const T** out) {
    void* d = nullptr;
    CU(cudaMalloc(&d, std::max<size_t>(count * sizeof(T), 16)));
    m->owned.push_back(d);
    CU(cudaMemcpy(d, h, count * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<const T*>(d);
    return 0;
}

// host matrix [rows][cols] -> device [rows_pad][ld], zero padded
static int upload_padded(b200_model* m, const double* h, size_t rows, size_t cols, size_t rows_pad, size_t ld, const double** out) {
    void* d = nullptr;
    CU(cudaMalloc(&d, std::max<size_t>(rows_pad * ld * sizeof(double), 16)));
    m->owned.push_back(d);
    if (rows_pad != rows || ld != cols) CU(cudaMemset(d, 0, rows_pad * ld * sizeof(double)));
    CU(cudaMemcpy2D(d, ld * sizeof(double), h, cols * sizeof(double), cols * sizeof(double), rows, cudaMemcpyHostToDevice));
    *out = static_cast<const double*>(d);
    return 0;
}

static int prepare_mvgauss(b200_model* m, const b200_model_desc* d) {
    const size_t n = (size_t)d->n;
    if (!d->x || !d->aux || !d->m1 || !d->m2) return fail("mvgauss: prec, cov, L^-T and L are required");
    m->ld = (long long)((n + 3) & ~(size_t)3);
    const size_t ld = (size_t)m->ld;
    if (upload_padded(m, d->x, n, n, n, ld, &m->prec) || upload_padded(m, d->aux, n, n, n, ld, &m->cov) ||
        upload_padded(m, d->m1, n, n, n, ld, &m->linvT) || upload_padded(m, d->m2, n, n, n, ld, &m->chol))
        return -1;
    m->logp_const = -0.5 * (double)n * 1.8378770664093454836 - d->scalar0;  // -n/2 log 2pi - sum log L_ii
    return 0;
}

static int prepare_logistic(b200_model* m, const b200_model_desc* d) {
    if (!d->x || !d->y_u8 || d->n_obs <= 0) return fail("logistic: X and y are required");
    if (d->n > 128) return fail("logistic: n_features=%d exceeds the fused kernel's limit (128)", d->n);
    m->n_rows = d->n_obs;
    m->ld = (d->n + 3) & ~3;
    m->KP = d->n <= 8 ? 8 : (d->n <= 32 ? 32 : 128);
    const size_t n_pad = (size_t)((d->n_obs + kLogiRows - 1) / kLogiRows) * kLogiRows;
    if (upload_padded(m, d->x, (size_t)d->n_obs, (size_t)d->n, n_pad, (size_t)m->KP, &m->X) ||
        upload_raw(m, d->y_u8, (size_t)d->n_obs, &m->y8))
        return -1;
    return 0;
}


// ------------------------------------------------------------------------------------------------
// ModelSpec IR -> device tables (csrc/ir_model.cuh).  Validates the closed set, precomputes the constant parts of the
// densities on the host (lgamma, log 2pi ...) and builds, for every indexed factor, the CSR transpose of its gather index
// (element -> observations) that the gradient is pulled through (deterministic, no atomics).
// ------------------------------------------------------------------------------------------------
static int ir_param(const b200_ir_param& p, int n, IrParamD* out, const char* what) {
    if (p.kind != 0 && p.kind != 1) return fail("ir: %s: parameter kind %d", what, p.kind);
    if (p.kind == 1 && (p.ref < 0 || p.ref >= n)) return fail("ir: %s: parameter reference %d outside q[0..%d)", what, p.ref, n);
    out->kind = p.kind; out->ref = p.kind ? p.ref : 0; out->value = p.value;
    return 0;
}

static int prepare_ir(b200_model* m, const b200_model_desc* d) {
    const b200_ir* R = d->ir;
    if (!R) return fail("ir: desc.ir is null");
    if (R->n_vars <= 0 || !R->vars) return fail("ir: no value variables");
    const int n = d->n;
    std::vector<IrVarD> vars(R->n_vars);
    int off = 0;
    for (int v = 0; v < R->n_vars; ++v) {
        const b200_ir_var& V = R->vars[v];
        if (V.offset != off || V.size <= 0) return fail("ir: variable %d: offsets must be contiguous in registration order", v);
        if (V.transform < B200_IR_T_NONE || V.transform > B200_IR_T_INTERVAL) return fail("ir: variable %d: transform %d", v, V.transform);
        if (V.transform == B200_IR_T_INTERVAL && !(V.lo < V.hi)) return fail("ir: variable %d: interval needs lo < hi", v);
        vars[v] = IrVarD{V.offset, V.size, V.transform, 0, V.lo, V.hi};
        off += V.size;
    }
    if (off != n) return fail("ir: variables cover %d elements but n = %d", off, n);
    const double LOG_PI = 1.1447298858494001741, LOG_2 = 0.69314718055994530942;
    std::vector<IrPriorD> priors(std::max(R->n_priors, 0));
    for (int k = 0; k < R->n_priors; ++k) {
        const b200_ir_prior& F = R->priors[k];
        if (F.var < 0 || F.var >= R->n_vars) return fail("ir: prior %d: variable index %d", k, F.var);
        IrPriorD P{};
        P.dist = F.dist; P.offset = vars[F.var].offset; P.size = vars[F.var].size;
        for (int a = 0; a < 3; ++a)
            if (ir_param(F.p[a], n, &P.p[a], "prior")) return -1;
        auto cst = [&](int a) { return F.p[a].kind == 0; };
        switch (F.dist) {
            case B200_IR_P_FLAT: break;
            case B200_IR_P_NORMAL: case B200_IR_P_LOGNORMAL: P.c0 = -B200_HALF_LOG_2PI; break;
            case B200_IR_P_HALFNORMAL: P.c0 = 0.5 * (LOG_2 - LOG_PI); break;
            case B200_IR_P_CAUCHY: P.c0 = -LOG_PI; break;
            case B200_IR_P_HALFCAUCHY: P.c0 = LOG_2 - LOG_PI; break;
            case B200_IR_P_EXPONENTIAL: break;
            case B200_IR_P_STUDENTT: {
                if (!cst(0) || !(F.p[0].value > 0)) return fail("ir: prior %d: StudentT nu must be a positive constant", k);
                const double nu = F.p[0].value;
                P.c0 = std::lgamma(0.5 * (nu + 1.0)) - std::lgamma(0.5 * nu) - 0.5 * std::log(nu) - 0.5 * LOG_PI;
            } break;
            case B200_IR_P_UNIFORM:
                if (!cst(0) || !cst(1) || !(F.p[0].value < F.p[1].value)) return fail("ir: prior %d: Uniform bounds must be constants lo < hi", k);
                P.c0 = -std::log(F.p[1].value - F.p[0].value);
                break;
            case B200_IR_P_GAMMA:
                if (!cst(0) || !cst(1) || !(F.p[0].value > 0) || !(F.p[1].value > 0)) return fail("ir: prior %d: Gamma needs constant alpha, beta > 0", k);
                P.c0 = F.p[0].value * std::log(F.p[1].value) - std::lgamma(F.p[0].value);
                break;
            case B200_IR_P_BETA:
                if (!cst(0) || !cst(1) || !(F.p[0].value > 0) || !(F.p[1].value > 0)) return fail("ir: prior %d: Beta needs constant alpha, beta > 0", k);
                P.c0 = -(std::lgamma(F.p[0].value) + std::lgamma(F.p[1].value) - std::lgamma(F.p[0].value + F.p[1].value));
                break;
            default: return fail("ir: prior %d: density %d is not in the closed set", k, F.dist);
        }
        priors[k] = P;
    }
    std::vector<IrLikD> liks(std::max(R->n_liks, 0));
    std::vector<IrTermD> terms;
    long long max_obs = 0;
    for (int l = 0; l < R->n_liks; ++l) {
        const b200_ir_lik& L = R->liks[l];
        if (L.N <= 0 || L.N > 0x7fffffff || !L.y) return fail("ir: likelihood %d: missing observations", l);
        if (L.n_terms <= 0 || !L.terms) return fail("ir: likelihood %d: no linear-predictor terms", l);
        const long long N = L.N;
        max_obs = std::max(max_obs, N);
        IrLikD D{};
        D.dist = L.dist; D.n_terms = L.n_terms; D.term0 = (int)terms.size(); D.sigma_kind = L.sigma_kind; D.N = N; D.nu = L.nu;
        if (upload_raw(m, L.y, (size_t)N, &D.y)) return -1;
        if (ir_param(L.sigma, n, &D.sigma, "likelihood sigma")) return -1;
        if (L.sigma_kind == B200_IR_S_REF && L.sigma.kind != 1) return fail("ir: likelihood %d: sigma_kind REF needs a reference", l);
        if (L.sigma_kind == B200_IR_S_OBS) {
            if (!L.sigma_obs) return fail("ir: likelihood %d: sigma_obs missing", l);
            if (upload_raw(m, L.sigma_obs, (size_t)N, &D.sigma_obs)) return -1;
        }
        switch (L.dist) {
            case B200_IR_L_NORMAL: case B200_IR_L_NORMAL_LOGVAR: D.c0 = -(double)N * B200_HALF_LOG_2PI; break;
            case B200_IR_L_BERNOULLI_LOGIT: break;
            case B200_IR_L_POISSON_LOG: { double c = 0; for (long long i = 0; i < N; ++i) c -= std::lgamma(L.y[i] + 1.0); D.c0 = c; } break;
            case B200_IR_L_STUDENTT:
                if (!(L.nu > 0)) return fail("ir: likelihood %d: StudentT nu must be > 0", l);
                D.c0 = (double)N * (std::lgamma(0.5 * (L.nu + 1.0)) - std::lgamma(0.5 * L.nu) - 0.5 * std::log(L.nu) - 0.5 * LOG_PI);
                break;
            default: return fail("ir: likelihood %d: density %d is not in the closed set", l, L.dist);
        }
        if ((L.dist == B200_IR_L_NORMAL || L.dist == B200_IR_L_STUDENTT) && L.sigma_kind == B200_IR_S_NONE)
            return fail("ir: likelihood %d needs sigma", l);
        for (int t = 0; t < L.n_terms; ++t) {
            const b200_ir_term& T = L.terms[t];
            if (T.n_factors < 0 || T.n_factors > 3) return fail("ir: likelihood %d term %d: 0..3 variable factors", l, t);
            IrTermD TD{};
            TD.n_factors = T.n_factors;
            if (T.coef && upload_raw(m, T.coef, (size_t)N, &TD.coef)) return -1;
            for (int f = 0; f < T.n_factors; ++f) {
                const b200_ir_factor& F = T.f[f];
                if (F.offset < 0 || F.size <= 0 || F.offset + F.size > n) return fail("ir: likelihood %d term %d: factor slice outside q", l, t);
                IrFactorD FD{};
                FD.offset = F.offset; FD.size = F.size;
                if (F.idx) {
                    std::vector<int> rowptr(F.size + 1, 0), rowobs((size_t)N);
                    for (long long i = 0; i < N; ++i) {
                        if (F.idx[i] < 0 || F.idx[i] >= F.size) return fail("ir: likelihood %d term %d: index %d out of range at %lld", l, t, F.idx[i], i);
                        ++rowptr[F.idx[i] + 1];
                    }
                    for (int j = 0; j < F.size; ++j) rowptr[j + 1] += rowptr[j];
                    std::vector<int> fill(rowptr.begin(), rowptr.end() - 1);
                    for (long long i = 0; i < N; ++i) rowobs[fill[F.idx[i]]++] = (int)i;  // ascending i inside a row: fixed order
                    if (upload_raw(m, F.idx, (size_t)N, &FD.idx) || upload(m, rowptr, &FD.rowptr) || upload(m, rowobs, &FD.rowobs)) return -1;
                } else if (F.size != 1 && F.size != N) {
                    return fail("ir: likelihood %d term %d: a variable of size %d needs an index to enter %lld observations", l, t, F.size, N);
                }
                TD.f[f] = FD;
            }
            terms.push_back(TD);
        }
        liks[l] = D;
    }
    std::vector<IrAr1D> ars(std::max(R->n_ar1, 0));
    for (int k = 0; k < R->n_ar1; ++k) {
        const b200_ir_ar1& A = R->ar1[k];
        if (A.var < 0 || A.var >= R->n_vars || vars[A.var].size < 2) return fail("ir: ar1 %d: bad variable", k);
        if (!(A.init_sigma > 0)) return fail("ir: ar1 %d: init_sigma must be > 0", k);
        IrAr1D D{};
        D.offset = vars[A.var].offset; D.size = vars[A.var].size; D.init_sigma = A.init_sigma;
        if (ir_param(A.phi, n, &D.phi, "ar1 phi") || ir_param(A.sigma, n, &D.sigma, "ar1 sigma")) return -1;
        ars[k] = D;
    }
    IrModel::Params& P = m->ir;
    P.n_vars = R->n_vars; P.n_priors = (int)priors.size(); P.n_liks = (int)liks.size(); P.n_ar1 = (int)ars.size(); P.n = n;
    if (upload(m, vars, &P.vars) || upload(m, priors, &P.priors) || upload(m, liks, &P.liks) || upload(m, terms, &P.terms) ||
        upload(m, ars, &P.ar1))
        return -1;
    P.n_pad = (n + 3) & ~3;
    P.stride = P.n_pad + ((max_obs + 3) & ~3LL);
    m->ir_max_obs = max_obs;
    return 0;
}

extern "C" int b200_model_create(const b200_model_desc* desc, b200_model** out) {
    if (!desc || !out) return fail("b200_model_create: null argument");
    if (desc->n <= 0) return fail("b200_model_create: n must be positive");
    if (b200_device_count() == 0) return fail("b200_model_create: no CUDA device visible");
    b200_model* m = new b200_model();
    m->kind = desc->kind;
    m->n = desc->n;
    cudaGetDevice(&m->device);
    int rc = 0;
    switch (desc->kind) {
        case B200_MODEL_STD_NORMAL: m->std_normal.n = desc->n; break;
        case B200_MODEL_EIGHT_SCHOOLS: rc = prepare_eight(m, desc); break;
        case B200_MODEL_RADON: rc = prepare_radon(m, desc); break;
        case B200_MODEL_STOCHVOL: rc = prepare_stochvol(m, desc); break;
        case B200_MODEL_MVGAUSS: rc = prepare_mvgauss(m, desc); break;
        case B200_MODEL_LOGISTIC: rc = prepare_logistic(m, desc); break;
        case B200_MODEL_IR: rc = prepare_ir(m, desc); break;
        default: rc = fail("b200_model_create: model kind %d not implemented", desc->kind);
    }
    if (rc) {
        delete m;
        return rc;
    }
    *out = m;
    return 0;
}

extern "C" void b200_model_destroy(b200_model* m) { delete m; }

extern "C" int b200_model_set_dense_mass(b200_model* m, const double* cov, const double* mp0, const double* mv0) {
    if (!m || !cov || !mp0 || !mv0) return fail("b200_model_set_dense_mass: null argument");
    if (m->cov) return fail("b200_model_set_dense_mass: this handle already has a dense mass matrix");
    CU(cudaSetDevice(m->device));
    const size_t n = (size_t)m->n;
    if (!m->ld) m->ld = (long long)((n + 3) & ~(size_t)3);
    const size_t ld = (size_t)m->ld;
    if (upload_padded(m, cov, n, n, n, ld, &m->cov) || upload_padded(m, mp0, n, n, n, ld, &m->linvT) ||
        upload_padded(m, mv0, n, n, n, ld, &m->chol))
        return -1;
    return 0;
}

extern "C" int b200_model_set_transforms(b200_model* m, const int8_t* kind, const double* lo, const double* hi) {
    if (!m || !kind || !lo || !hi) return fail("b200_model_set_transforms: null argument");
    for (int i = 0; i < m->n; ++i) {
        if (kind[i] < 0 || kind[i] > 2) return fail("b200_model_set_transforms: element %d: unknown transform %d", i, (int)kind[i]);
        if (kind[i] == 2 && !(lo[i] < hi[i])) return fail("b200_model_set_transforms: element %d: interval needs lo < hi", i);
    }
    CU(cudaSetDevice(m->device));
    std::vector<signed char> k(kind, kind + m->n);
    std::vector<double> l(lo, lo + m->n), h(hi, hi + m->n);
    if (upload(m, k, &m->tr_kind) || upload(m, l, &m->tr_lo) || upload(m, h, &m->tr_hi)) return -1;
    return 0;
}
extern "C" int b200_model_n(const b200_model* m) { return m ? m->n : -1; }

// ------------------------------------------------------------------------------------------------
// dispatch helpers: (model kind, n) -> (Model, NPL elements per thread, W warps per chain)
//   n <= 256   : chain = warp  (W = 1), NPL in {1,2,4,6,8}
//   n <= 4096  : chain = CTA of 8 warps (W = 8), NPL in {2,4,8,12,16}   (models that implement the team path)
// ------------------------------------------------------------------------------------------------
static constexpr int kTeamW = 8;
static int npl_warp(int n) {
    const int need = (n + 31) / 32;
    const int opts[] = {1, 2, 4, 6, 8};
    for (int o : opts)
        if (need <= o) return o;
    return 0;
}
static int npl_team(int n) {
    const int need = (n + 32 * kTeamW - 1) / (32 * kTeamW);
    const int opts[] = {2, 4, 8, 12, 16};
    for (int o : opts)
        if (need <= o) return o;
    return 0;
}

// Calls f.template operator()<Model, NPL, W>(params) for the model's kind and size.
template <class F>
static int dispatch(const b200_model* m, F&& f) {
#define B200_WARP(MODEL, PARAMS)                                                  \
    switch (npl_warp(m->n)) {                                                     \
        case 1: return f.template operator()<MODEL, 1, 1>(PARAMS);                \
        case 2: return f.template operator()<MODEL, 2, 1>(PARAMS);                \
        case 4: return f.template operator()<MODEL, 4, 1>(PARAMS);                \
        case 6: return f.template operator()<MODEL, 6, 1>(PARAMS);                \
        case 8: return f.template operator()<MODEL, 8, 1>(PARAMS);                \
        default: break;                                                           \
    }
#define B200_TEAM(MODEL, PARAMS)                                                  \
    switch (npl_team(m->n)) {                                                     \
        case 2: return f.template operator()<MODEL, 2, kTeamW>(PARAMS);           \
        case 4: return f.template operator()<MODEL, 4, kTeamW>(PARAMS);           \
        case 8: return f.template operator()<MODEL, 8, kTeamW>(PARAMS);           \
        case 12: return f.template operator()<MODEL, 12, kTeamW>(PARAMS);         \
        case 16: return f.template operator()<MODEL, 16, kTeamW>(PARAMS);         \
        default: break;                                                           \
    }
    switch (m->kind) {
        case B200_MODEL_STD_NORMAL:
            B200_WARP(StdNormalModel, m->std_normal)  // n <= 256
            B200_TEAM(StdNormalModel, m->std_normal)
            return fail("std_normal: n=%d exceeds 4096", m->n);
        case B200_MODEL_EIGHT_SCHOOLS:
            B200_WARP(EightSchoolsModel, m->eight)
            return fail("eight_schools: n=%d exceeds the chain-per-warp limit (256)", m->n);
        case B200_MODEL_RADON:
            B200_WARP(RadonModel, m->radon)
            return fail("radon: n=%d exceeds the chain-per-warp limit (256)", m->n);
        case B200_MODEL_STOCHVOL:
            B200_TEAM(StochVolModel, m->stochvol)
            return fail("stochvol: n=%d exceeds 4096", m->n);
        case B200_MODEL_IR:
            B200_WARP(IrModel, m->ir)  // n <= 256
            B200_TEAM(IrModel, m->ir)
            return fail("ir: n=%d exceeds the chain-per-CTA limit (4096)", m->n);
    }
#undef B200_WARP
#undef B200_TEAM
    return fail("dispatch: model kind %d not implemented", m->kind);
}


// The generic IR device function keeps x (constrained values) and the per-observation residuals of the likelihood being
// processed in a per-team global scratch slice: size it for the launch (teams = CTAs x teams per CTA) and hand the kernel
// the Params copy that points at it.
template <class Model>
static int launch_params(const b200_model* m, const typename Model::Params& MP, long long teams, typename Model::Params* out) {
    *out = MP;
    if constexpr (std::is_same_v<Model, IrModel>) {
        b200_model* mm = const_cast<b200_model*>(m);
        CU(mm->ensure_ir_scratch(teams));
        *out = mm->ir;
    }
    return 0;
}

struct Timer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t s;
    explicit Timer(cudaStream_t s_) : s(s_) {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, s);
    }
    void stop(int launches) {
        cudaEventRecord(b, s);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        g_last_ms = ms;
        g_last_launches = launches;
    }
    ~Timer() {
        if (a) cudaEventDestroy(a);
        if (b) cudaEventDestroy(b);
    }
};

// Host<->device staging of one array.
struct Staged {
    DevBuf dev;
    void* lent = nullptr;  // device staging lent by the caller (an arena in the model handle) instead of `dev`
    void* user = nullptr;
    size_t bytes = 0;
    bool host = false, out = false;
    void* dptr() const { return lent ? lent : dev.p; }
    void* ptr() const { return host ? dptr() : user; }
};
// `direct`: an OUTPUT buffer in page-locked host memory (cudaHostAlloc / cudaHostRegister, e.g. a torch pinned tensor) is
// written by the kernel itself through its device alias (UVA), so the device->host transfer overlaps the run instead of
// following it (2.9 GB of draws per Radon bench step: 160 ms after the kernel vs ~0 inside it).
static int stage_in(Staged& s, const void* user, size_t bytes, int mem, bool copy_in, bool copy_out,
                    cudaStream_t st, bool direct = false) {
    s.user = const_cast<void*>(user);
    s.bytes = bytes;
    s.host = (mem == B200_MEM_HOST) && user != nullptr;
    s.out = copy_out;
    if (s.host && direct && !copy_in) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, user) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
            s.user = at.devicePointer;
            s.host = false;
            return 0;
        }
        cudaGetLastError();  // pageable memory: not an error, fall back to staging
    }
    if (s.host) {
        if (!s.lent) CU(s.dev.alloc(bytes));
        if (copy_in) CU(cudaMemcpyAsync(s.dptr(), user, bytes, cudaMemcpyHostToDevice, st));
    }
    return 0;
}
static int stage_out(Staged& s, cudaStream_t st) {
    if (s.host && s.out) CU(cudaMemcpyAsync(s.user, s.dptr(), s.bytes, cudaMemcpyDeviceToHost, st));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// b200_logp_dlogp
// ------------------------------------------------------------------------------------------------
struct LogpLaunch {
    const b200_model* m; int C; const double* q; double* logp; double* grad; cudaStream_t st;
    long long ldq = 0, ldg = 0;  // row strides (0: contiguous rows of n)
    template <class Model, int NPL, int W>
    int operator()(const typename Model::Params& MP) const {
        const int wpb = (W == 1) ? 8 : 1;  // chains per CTA
        const size_t data = (Model::shared_bytes(MP) + 15) & ~(size_t)15;
        const size_t smem = data + (size_t)wpb * (2 * 32 * W * NPL + (W > 1 ? 8 * W : 0)) * sizeof(double);
        auto kern = logp_grad_warp_kernel<Model, NPL, W>;
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int blocks = std::max(1, std::min((C + wpb - 1) / wpb, 148 * 8));
        typename Model::Params MPl;
        if (launch_params<Model>(m, MP, (long long)blocks * wpb, &MPl)) return -1;
        kern<<<blocks, (W == 1) ? wpb * 32 : 32 * W, smem, st>>>(MPl, m->n, C, q, logp, grad, ldq ? ldq : m->n, ldg ? ldg : m->n);
        CU(cudaGetLastError());
        return 0;
    }
};

extern "C" int b200_logp_dlogp(b200_model* m, const double* q, int32_t C, double* logp, double* grad,
                               int32_t mem, void* stream) {
    if (!m || !q || !logp || !grad) return fail("b200_logp_dlogp: null argument");
    if (C <= 0) return 0;
    CU(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t vb = (size_t)C * m->n * sizeof(double);
    Staged sq, sl, sg;
    if (stage_in(sq, q, vb, mem, true, false, st)) return -1;
    if (stage_in(sl, logp, (size_t)C * sizeof(double), mem, false, true, st)) return -1;
    if (stage_in(sg, grad, vb, mem, false, true, st)) return -1;
    Timer t(st);
    if (is_lockstep_kind(m->kind)) {
        if (lockstep_logp(m, (const double*)sq.ptr(), C, (double*)sl.ptr(), (double*)sg.ptr(), st)) return -1;
    } else {
        LogpLaunch L{m, C, (const double*)sq.ptr(), (double*)sl.ptr(), (double*)sg.ptr(), st};
        if (dispatch(m, L)) return -1;
    }
    t.stop(1);
    if (stage_out(sl, st) || stage_out(sg, st)) return -1;
    CU(cudaStreamSynchronize(st));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// b200_leapfrog
// ------------------------------------------------------------------------------------------------
struct LeapLaunch {
    const b200_model* m; int C, n_steps; const double *var, *eps; double *q, *p, *v, *grad, *energy, *logp;
    long long* idx; cudaStream_t st;
    template <class Model, int NPL, int W>
    int operator()(const typename Model::Params& MP) const {
        const int wpb = (W == 1) ? 8 : 1;
        const size_t data = (Model::shared_bytes(MP) + 15) & ~(size_t)15;
        const size_t smem = data + (size_t)wpb * (2 * 32 * W * NPL + (W > 1 ? 8 * W : 0)) * sizeof(double);
        auto kern = leapfrog_warp_kernel<Model, NPL, W>;
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int blocks = std::max(1, std::min((C + wpb - 1) / wpb, 148 * 8));
        typename Model::Params MPl;
        if (launch_params<Model>(m, MP, (long long)blocks * wpb, &MPl)) return -1;
        kern<<<blocks, (W == 1) ? wpb * 32 : 32 * W, smem, st>>>(MPl, m->n, C, var, eps, n_steps, q, p, v, grad, energy, logp, idx);
        CU(cudaGetLastError());
        return 0;
    }
};

extern "C" int b200_leapfrog(b200_model* m, const double* var, const double* eps, int32_t n_steps, int32_t C,
                             double* q, double* p, double* v, double* grad, double* energy, double* logp,
                             int64_t* idx, int32_t mem, void* stream) {
    if (!m || !var || !eps || !q || !p || !v || !grad || !energy || !logp || !idx)
        return fail("b200_leapfrog: null argument");
    if (n_steps < 0) return fail("b200_leapfrog: n_steps < 0");
    if (is_lockstep_kind(m->kind)) return fail("b200_leapfrog: GEMM-shaped models advance in lock step inside b200_nuts_run");
    if (C <= 0) return 0;
    CU(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t vb = (size_t)C * m->n * sizeof(double), sb = (size_t)C * sizeof(double);
    Staged s_var, s_eps, s_q, s_p, s_v, s_g, s_e, s_l, s_i;
    if (stage_in(s_var, var, vb, mem, true, false, st) || stage_in(s_eps, eps, sb, mem, true, false, st) ||
        stage_in(s_q, q, vb, mem, true, true, st) || stage_in(s_p, p, vb, mem, true, true, st) ||
        stage_in(s_v, v, vb, mem, true, true, st) || stage_in(s_g, grad, vb, mem, true, true, st) ||
        stage_in(s_e, energy, sb, mem, true, true, st) || stage_in(s_l, logp, sb, mem, true, true, st) ||
        stage_in(s_i, idx, (size_t)C * sizeof(int64_t), mem, true, true, st))
        return -1;
    Timer t(st);
    LeapLaunch L{m, C, n_steps, (const double*)s_var.ptr(), (const double*)s_eps.ptr(), (double*)s_q.ptr(),
                 (double*)s_p.ptr(), (double*)s_v.ptr(), (double*)s_g.ptr(), (double*)s_e.ptr(),
                 (double*)s_l.ptr(), (long long*)s_i.ptr(), st};
    if (dispatch(m, L)) return -1;
    t.stop(1);
    if (stage_out(s_q, st) || stage_out(s_p, st) || stage_out(s_v, st) || stage_out(s_g, st) ||
        stage_out(s_e, st) || stage_out(s_l, st) || stage_out(s_i, st))
        return -1;
    CU(cudaStreamSynchronize(st));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// GEMM-shaped models: batched evaluation of C points (rows of Q[C][ld]) -> G[C][ld] (+ logp[C]) with the
// hand-written DMMA kernels of dense.cuh.
// ------------------------------------------------------------------------------------------------
template <int WM, int NB>
static int launch_gemm(cudaStream_t st, const double* Q, long long ldq, int C, const double* M, long long ldm, int Nout, int K,
                       double alpha, double* D, long long ldd) {
    constexpr int NST = 3;
    const size_t smem = NST * gemm_stage_doubles<WM, NB>() * sizeof(double);
    auto kern = gemm_nt_dmma_kernel<WM, NB, NST>;
    // per call: the attribute belongs to the (function, device) pair and a process may own handles on several devices
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((Nout + 8 * NB - 1) / (8 * NB), (C + 16 * WM - 1) / (16 * WM));
    kern<<<grid, 32 * WM, smem, st>>>(Q, ldq, C, M, ldm, Nout, K, alpha, D, ldd);
    CU(cudaGetLastError());
    return 0;
}

// D[C][Nout] = alpha * Q[C][K] . M[Nout][K]^T.  Tile shape picked per call: chains per CTA from C, outputs per CTA
// (8 NB) so that the tile count fills whole waves of 148 SMs.
static int gemm_nt_tc(b200_model* m, cudaStream_t st, const double* Q, long long ldq, int C, const b200_model::TcMat& T, int Nout,
                      double alpha, double* D, long long ldd);

static int gemm_nt(b200_model* m, cudaStream_t st, const double* Q, long long ldq, int C, const double* M, long long ldm, int Nout, int K,
                   double alpha, double* D, long long ldd) {
    if (C <= 0 || Nout <= 0) return 0;
    if (m && m->precision == B200_PRECISION_TC_FP16X2) {
        for (const b200_model::TcMat& T : m->tc_mats)
            if (T.src == M && T.hi) return gemm_nt_tc(m, st, Q, ldq, C, T, Nout, alpha, D, ldd);
    }
    const int wm = C > 64 ? 8 : (C > 32 ? 4 : 2);
    const int cb = (C + 16 * wm - 1) / (16 * wm);
    int best_nb = 9;
    double best = -1.0;
    const int nbs[3] = {17, 9, 5};
    for (int i = 0; i < (wm == 8 ? 3 : 2); ++i) {
        const int nb = (wm == 8) ? nbs[i] : nbs[i + 1];
        const long long tiles = (long long)cb * ((Nout + 8 * nb - 1) / (8 * nb));
        const long long waves = (tiles + 147) / 148;
        // useful work / occupied SM time; small bonus for wider tiles (fewer fragment loads per DMMA)
        const double eff = (double)Nout * cb / ((double)waves * 148 * 8 * nb) + 1e-3 * nb;
        if (eff > best) { best = eff; best_nb = nb; }
    }
#define B200_GEMM(WM_, NB_) return launch_gemm<WM_, NB_>(st, Q, ldq, C, M, ldm, Nout, K, alpha, D, ldd)
    if (wm == 8) { if (best_nb == 17) B200_GEMM(8, 17); if (best_nb == 9) B200_GEMM(8, 9); B200_GEMM(8, 5); }
    if (wm == 4) { if (best_nb == 9) B200_GEMM(4, 9); B200_GEMM(4, 5); }
    if (best_nb == 9) B200_GEMM(2, 9);
    B200_GEMM(2, 5);
#undef B200_GEMM
}

struct BatchScratch {  // logistic partial results
    DevBuf gpart, lpart;
    int gx = 0, cpad = 0;
    long long cap_rows = 0;  // allocated gx * cpad (the product barely changes when the batch shrinks: more row CTAs per chain block)
};


// ------------------------------------------------------------------------------------------------
// tensor-core performance mode of the logistic GLM (tcgen05 + TMEM + TMA, split fp16): preparation and launch
// ------------------------------------------------------------------------------------------------
typedef CUresult (*b200_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                         const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                         CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// K-major fp16 matrix [rows][kpad] -> tensor map with boxes of 64 k (one 128-byte swizzle row) x box_rows rows
static int make_tc_map(CUtensorMap* map, const __half* base, long long rows, long long kpad, int box_rows) {
    static b200_encode_tiled_fn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        CU(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        if (!fn || q != cudaDriverEntryPointSuccess) return fail("cuTensorMapEncodeTiled is not available in this driver");
        encode = reinterpret_cast<b200_encode_tiled_fn>(fn);
    }
    const cuuint64_t dims[2] = {(cuuint64_t)kpad, (cuuint64_t)rows};         // innermost first
    const cuuint64_t strides[1] = {(cuuint64_t)kpad * sizeof(__half)};       // row pitch in bytes
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}
static int make_x_map(CUtensorMap* map, const __half* base, long long rows) { return make_tc_map(map, base, rows, kTcK, kTcRows); }

// dense Gaussian: split the four n x n matrices once
static int prepare_mvgauss_tc(b200_model* m) {
    if (m->tc_mats[0].hi) return 0;
    const long long n = m->n;
    m->tc_kpad = (n + kGtKB - 1) / kGtKB * kGtKB;
    m->tc_npad = (n + kGtN - 1) / kGtN * kGtN;
    const double* src[4] = {m->prec, m->cov, m->linvT, m->chol};
    for (int i = 0; i < 4; ++i) {
        void *h = nullptr, *l = nullptr;
        const size_t bytes = (size_t)m->tc_npad * m->tc_kpad * sizeof(__half);
        CU(cudaMalloc(&h, bytes));
        m->owned.push_back(h);
        CU(cudaMalloc(&l, bytes));
        m->owned.push_back(l);
        const long long total = m->tc_npad * m->tc_kpad;
        gemm_tc_split_kernel<<<(unsigned)((total + 255) / 256), 256>>>(src[i], n, n, m->ld, (__half*)h, (__half*)l, m->tc_npad, m->tc_kpad);
        CU(cudaGetLastError());
        b200_model::TcMat& T = m->tc_mats[i];
        T.src = src[i]; T.hi = (const __half*)h; T.lo = (const __half*)l;
        if (make_tc_map(&T.map_hi, T.hi, m->tc_npad, m->tc_kpad, kGtN) || make_tc_map(&T.map_lo, T.lo, m->tc_npad, m->tc_kpad, kGtN)) return -1;
    }
    CU(cudaDeviceSynchronize());
    return 0;
}

// D[C][Nout] = alpha Q . M^T on the tensor cores; M must be one of the model's pre-split matrices
static int gemm_nt_tc(b200_model* m, cudaStream_t st, const double* Q, long long ldq, int C, const b200_model::TcMat& T, int Nout,
                      double alpha, double* D, long long ldd) {
    const long long rows_pad = ((long long)C + kGtM - 1) / kGtM * kGtM;
    if (rows_pad > m->tc_a_rows) {
        if (m->tc_a_hi) cudaFree(m->tc_a_hi);
        if (m->tc_a_lo) cudaFree(m->tc_a_lo);
        m->tc_a_hi = m->tc_a_lo = nullptr;
        m->tc_a_rows = 0;
        CU(cudaMalloc((void**)&m->tc_a_hi, (size_t)rows_pad * m->tc_kpad * sizeof(__half)));
        CU(cudaMalloc((void**)&m->tc_a_lo, (size_t)rows_pad * m->tc_kpad * sizeof(__half)));
        m->tc_a_rows = rows_pad;
    }
    const long long total = rows_pad * m->tc_kpad;
    gemm_tc_split_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(Q, C, m->n, ldq, m->tc_a_hi, m->tc_a_lo, rows_pad, m->tc_kpad);
    CU(cudaGetLastError());
    CUtensorMap a_hi, a_lo;
    if (make_tc_map(&a_hi, m->tc_a_hi, rows_pad, m->tc_kpad, kGtM) || make_tc_map(&a_lo, m->tc_a_lo, rows_pad, m->tc_kpad, kGtM)) return -1;
    GemmTcArgs G{};
    G.C = C; G.Nout = Nout; G.n_kblocks = (int)(m->tc_kpad / kGtKB); G.alpha = alpha; G.D = D; G.ldd = ldd;
    G.n_tiles_n = (int)(m->tc_npad / kGtN);
    G.n_tiles = G.n_tiles_n * (int)(rows_pad / kGtM);
    auto kern = gemm_tc_kernel;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGtSmemBytes));
    const int grid = std::min(G.n_tiles, 148);
    kern<<<grid, kGtThreads, kGtSmemBytes, st>>>(a_hi, a_lo, T.map_hi, T.map_lo, G);
    CU(cudaGetLastError());
    return 0;
}

static int prepare_logistic_tc(b200_model* m) {
    if (m->Xh) return 0;
    m->tc_slabs = (m->n_rows + kTcRows - 1) / kTcRows;
    const long long rows_pad = m->tc_slabs * kTcRows;
    void *h = nullptr, *l = nullptr;
    CU(cudaMalloc(&h, (size_t)rows_pad * kTcK * sizeof(__half)));
    m->owned.push_back(h);
    CU(cudaMalloc(&l, (size_t)rows_pad * kTcK * sizeof(__half)));
    m->owned.push_back(l);
    const long long total = rows_pad * kTcK;
    logistic_tc_split_kernel<<<(unsigned)((total + 255) / 256), 256>>>(m->X, m->n_rows, m->n, m->KP, (__half*)h, (__half*)l, rows_pad);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    m->Xh = (const __half*)h;
    m->Xl = (const __half*)l;
    void* y32 = nullptr;  // labels as fp32, padded to whole slabs: travel with the slab (logistic_tc2_kernel)
    CU(cudaMalloc(&y32, (size_t)rows_pad * sizeof(float)));
    m->owned.push_back(y32);
    logistic_tc_y_kernel<<<(unsigned)((rows_pad + 255) / 256), 256>>>(m->y8, m->n_rows, (float*)y32, rows_pad);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    m->y32 = (const float*)y32;
    if (make_x_map(&m->map_hi, m->Xh, rows_pad) || make_x_map(&m->map_lo, m->Xl, rows_pad)) return -1;
    return 0;
}

extern "C" int b200_model_set_precision(b200_model* m, int32_t mode) {
    if (!m) return fail("b200_model_set_precision: null model");
    if (mode != B200_PRECISION_FP64 && mode != B200_PRECISION_TC_FP16X2) return fail("b200_model_set_precision: unknown mode %d", mode);
    if (mode == B200_PRECISION_TC_FP16X2) {
        if (m->kind != B200_MODEL_LOGISTIC && m->kind != B200_MODEL_MVGAUSS)
            return fail("tensor-core mode is implemented for the dense contractions: the logistic GLM and the dense Gaussian");
        CU(cudaSetDevice(m->device));
        if (m->kind == B200_MODEL_LOGISTIC ? prepare_logistic_tc(m) : prepare_mvgauss_tc(m)) return -1;
    }
    m->precision = mode;
    return 0;
}

static bool is_lockstep_kind(int kind) { return kind == B200_MODEL_MVGAUSS || kind == B200_MODEL_LOGISTIC; }

template <int KB>
static int launch_logistic(const b200_model* m, int C, const double* Q, long long ldq, BatchScratch& bs, cudaStream_t st) {
    auto kern = logistic_fused_kernel<KB>;
    const size_t smem = logistic_smem_bytes<KB>();
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<dim3(bs.gx, bs.cpad / kLogiChains), 32 * (kLogiChains / (8 * kLogiMB)), smem, st>>>(m->X, m->y8, m->n_rows, Q, ldq, C, m->n, bs.gpart.as<double>(),
                                                               bs.lpart.as<double>(), bs.cpad);
    CU(cudaGetLastError());
    return 0;
}

// G = grad logp(Q) for all C rows; logp written only for models that do not derive it from q.g
static int batch_eval(b200_model* m, int C, const double* Q, double* G, double* logp, BatchScratch& bs, cudaStream_t st,
                      int* launches) {
    const int n = m->n;
    const long long ld = m->ld;
    if (!is_lockstep_kind(m->kind)) {
        // any other model under a dense mass matrix: its own fused logp+grad device function, one team per requested point
        LogpLaunch L{m, C, Q, logp, G, st, ld, ld};
        if (launches) *launches += 1;
        return dispatch(m, L);
    }
    if (m->kind == B200_MODEL_MVGAUSS) {
        // grad = -P q  (MvNormal.logp multivariate.py:275-295; P symmetric)
        if (launches) *launches += 1;
        return gemm_nt(m, st, Q, ld, C, m->prec, ld, n, (int)ld, -1.0, G, ld);
    }
    // logistic: one fused pass over X, then the fixed-order reduction of the row-CTA partials
    const int cb = (C + kLogiChains - 1) / kLogiChains;
    const long long n_slabs = (m->n_rows + kLogiRows - 1) / kLogiRows;
    const int gx = (int)std::max<long long>(1, std::min<long long>(n_slabs, 148 / std::min(cb, 148)));
    bs.gx = gx;
    bs.cpad = cb * kLogiChains;
    if ((long long)gx * bs.cpad > bs.cap_rows) {
        if (bs.gpart.p) { cudaFree(bs.gpart.p); bs.gpart.p = nullptr; }
        if (bs.lpart.p) { cudaFree(bs.lpart.p); bs.lpart.p = nullptr; }
        bs.cap_rows = std::max<long long>((long long)gx * bs.cpad, 148LL * kLogiChains);
        CU(bs.gpart.alloc((size_t)bs.cap_rows * m->KP * sizeof(double)));
        CU(bs.lpart.alloc((size_t)bs.cap_rows * sizeof(double)));
    }
    int rc = 0;
    if (m->precision == B200_PRECISION_TC_FP16X2) {
        // tcgen05 path: the same partial-result layout ([gx][Cpad][128] fp64), so the fixed-order finish below is shared
        if (m->KP != kTcK) {  // partials are [.][.][KP]: the tensor-core kernel writes 128-wide rows
            return fail("tensor-core mode needs the 128-feature layout (65..128 features); this model has %d", m->n);
        }
        auto kern = logistic_tc2_kernel;
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTc2SmemBytes));
        LogisticTc2Args A{m->y32, m->n_rows, m->tc_slabs, Q, ld, C, m->n, bs.gpart.as<double>(), bs.lpart.as<double>(), bs.cpad};
        kern<<<dim3(bs.gx, bs.cpad / kLogiChains), kTc2Threads, kTc2SmemBytes, st>>>(m->map_hi, m->map_lo, A);
        CU(cudaGetLastError());
    } else
    switch (m->KP) {
        case 8: rc = launch_logistic<1>(m, C, Q, ld, bs, st); break;
        case 32: rc = launch_logistic<4>(m, C, Q, ld, bs, st); break;
        default: rc = launch_logistic<16>(m, C, Q, ld, bs, st); break;
    }
    if (rc) return rc;
    if (m->precision == B200_PRECISION_TC_FP16X2)  // feature-major partials: the coalesced reduction
        logistic_finish_fm_kernel<<<dim3((C + 31) / 32, (m->KP + 15) / 16), 256, 0, st>>>(Q, ld, G, ld, n, m->KP, C, bs.cpad, bs.gpart.as<double>(),
                                                                                         bs.lpart.as<double>(), gx, logp);
    else
        logistic_finish_kernel<<<(C + 3) / 4, 128, 0, st>>>(Q, ld, G, ld, n, m->KP, C, bs.cpad, bs.gpart.as<double>(),
                                                            bs.lpart.as<double>(), gx, logp, 0);
    CU(cudaGetLastError());
    if (launches) *launches += 2;
    return 0;
}

// b200_logp_dlogp for the GEMM-shaped models: user rows [C][n] <-> padded rows [C][ld]
static int lockstep_logp(b200_model* m, const double* q_dev, int C, double* logp_dev, double* grad_dev, cudaStream_t st) {
    const int n = m->n;
    const long long ld = m->ld;
    DevBuf Qp, Gp;
    CU(Qp.alloc((size_t)C * ld * sizeof(double)));
    CU(Gp.alloc((size_t)C * ld * sizeof(double)));
    CU(cudaMemsetAsync(Qp.p, 0, (size_t)C * ld * sizeof(double), st));
    CU(cudaMemcpy2DAsync(Qp.p, ld * sizeof(double), q_dev, n * sizeof(double), n * sizeof(double), C, cudaMemcpyDeviceToDevice, st));
    BatchScratch bs;
    if (batch_eval(m, C, Qp.as<double>(), Gp.as<double>(), logp_dev, bs, st, nullptr)) return -1;
    if (m->kind == B200_MODEL_MVGAUSS) {
        half_dot_logp_kernel<<<(C + 3) / 4, 128, 0, st>>>(Qp.as<double>(), Gp.as<double>(), ld, n, C, m->logp_const, logp_dev);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpy2DAsync(grad_dev, n * sizeof(double), Gp.p, ld * sizeof(double), n * sizeof(double), C, cudaMemcpyDeviceToDevice, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

// warps per chain of the lock-step advance kernel for long state vectors (n > 512): 16 is 5 % faster than 8 at n = 10^4
static constexpr int kLsAdvW = 16;

// The lock-step driver: advance <-> batched evaluation until every chain is done.
static int run_lockstep(b200_model* m, LsDev P, cudaStream_t st) {
    const int C = P.C, n = P.n;
    const bool dense = P.dense != 0;
    const long long ld = m->ld;
    const size_t mat = (size_t)C * ld * sizeof(double);
    // One arena in the model handle, kept between runs (VERDICT r1 weak #6: eleven cudaMalloc per run; the chain vectors alone
    // are 2.6 GB for config 5, and allocating / freeing them cost ~1 s of host time per run): state | vecs | 3-8 request
    // matrices | logp | counters | momentum list.
    P.ld = ld;
    P.vec_stride = ls_vec_count(P.max_td) * n;
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t b_state = up((size_t)C * sizeof(LsState)), b_vecs = up((size_t)C * P.vec_stride * sizeof(double)), b_mat = up(mat);
    const size_t b_l = up((size_t)C * sizeof(double)), b_cnt = up(4 * sizeof(int)), b_mom = up((size_t)C * sizeof(int));
    // compaction of the request rows once finished chains free a whole tile (128 rows) of them (lockstep.cuh: ls_compact_*).
    // B200_LS_COMPACT_TILE is a test seam, not a tuning option: 0 never compacts, and a small tile makes runs of a few dozen
    // chains compact, so that a test can check that compaction changes no result.
    const char* tile_env = getenv("B200_LS_COMPACT_TILE");
    const int ctile = tile_env ? atoi(tile_env) : 128;
    const bool compact = ctile > 0 && C > ctile;
    const int n_mats = (dense ? 8 : 2) + (compact ? 1 : 0);
    // DENSE_ADAPT: four n x n matrices per chain (covariance, Cholesky factor, two raw scatter matrices; dense_adapt.cuh)
    const bool fa = P.mass_kind == B200_MASS_DENSE_ADAPT;
    const size_t b_fa = fa ? up((size_t)C * n * n * sizeof(double)) : 0;
    CU(m->ensure_ls_arena(b_state + b_vecs + n_mats * b_mat + b_l + b_cnt + 3 * b_mom + 4 * b_fa));
    char* a = static_cast<char*>(m->ls_arena);
    auto take = [&](size_t b) { char* p = a; a += b; return p; };
    P.state = reinterpret_cast<LsState*>(take(b_state));
    P.vecs = reinterpret_cast<double*>(take(b_vecs));
    P.Qreq = reinterpret_cast<double*>(take(b_mat));
    P.Greq = reinterpret_cast<double*>(take(b_mat));
    double *Zb = nullptr, *P0b = nullptr, *V0b = nullptr;
    if (dense) {
        P.Wreq = reinterpret_cast<double*>(take(b_mat));
        P.P0n = reinterpret_cast<double*>(take(b_mat));
        P.V0n = reinterpret_cast<double*>(take(b_mat));
        Zb = reinterpret_cast<double*>(take(b_mat));
        P0b = reinterpret_cast<double*>(take(b_mat));
        V0b = reinterpret_cast<double*>(take(b_mat));
    }
    double* Qalt = compact ? reinterpret_cast<double*>(take(b_mat)) : nullptr;
    P.logp_req = reinterpret_cast<double*>(take(b_l));
    P.counters = reinterpret_cast<int*>(take(b_cnt));
    P.mom_list = reinterpret_cast<int*>(take(b_mom));
    P.slot = reinterpret_cast<int*>(take(b_mom));
    int* new_slot = reinterpret_cast<int*>(take(b_mom));
    if (!compact) P.slot = nullptr;
    if (fa) {
        P.fa_cov = reinterpret_cast<double*>(take(b_fa));
        P.fa_chol = reinterpret_cast<double*>(take(b_fa));
        P.fa_raw = reinterpret_cast<double*>(take(2 * b_fa));
    }
    // the padding columns of the request / result matrices must be zero (they are inside the GEMMs' k range) and the chain
    // vectors start from zero: clearing is bandwidth-trivial (2.6 GB at HBM speed = 0.4 ms), unlike allocating
    CU(cudaMemsetAsync(P.vecs, 0, b_vecs + n_mats * b_mat, st));
    P.logp_from_dot = (m->kind == B200_MODEL_MVGAUSS) ? 1 : 0;
    P.logp_const = m->logp_const;
    BatchScratch bs;
    const int blocks = (C + 3) / 4;
    Timer t(st);
    int launches = 0;
    ls_init_kernel<<<blocks, 128, 0, st>>>(P);
    CU(cudaGetLastError());
    ++launches;
    if (fa) {
        fa_init_kernel<<<C, kFaThreads, 0, st>>>(P);
        CU(cudaGetLastError());
        ++launches;
    }
    int n_mom = dense ? C : 0;  // every chain needs the momentum of draw 0
    bool serve = true;
    // Deferred momentum (fixed dense mass).  A chain asks for the momentum of draw it+1 when draw `it` begins, so the request
    // has the length of a draw to be served.  The two momentum GEMMs stream their n x n matrices whatever the number of
    // requesting rows (for n = 10^4 they cost as much as the gradient and mass GEMMs of ALL chains), so requests are queued on
    // the device and served in batches: when half of the live chains are waiting in the queue, or as soon as a chain reaches
    // the end of its draw without its momentum (it then idles for one round: LsState phase 3).  The noise z of (chain, draw)
    // does not depend on when it is served, so results are identical for every threshold.
    const double defer = fa ? 0.0 : 0.5;
    CU(cudaMemsetAsync(P.counters, 0, 4 * sizeof(int), st));
    int C_eval = C;             // rows of the request matrices in use (shrinks when finished chains free a tile)
    for (;;) {
        if (batch_eval(m, C_eval, P.Qreq, P.Greq, P.logp_req, bs, st, &launches)) return -1;
        if (fa) {
            // per-chain covariance: w = Sigma_c g is a matrix-vector product per chain; a chain that finished a draw gets its
            // potential updated (covariance, Cholesky) and the momentum of its next draw (dense_adapt.cuh)
            fa_symv_kernel<<<C, kFaThreads, fa_smem_bytes(n), st>>>(P);
            ++launches;
            if (n_mom > 0) {
                fa_update_momentum_kernel<<<n_mom, kFaThreads, fa_smem_bytes(n), st>>>(P, n_mom);
                ++launches;
                CU(cudaMemsetAsync(P.counters + 2, 0, sizeof(int), st));
            }
            CU(cudaGetLastError());
        } else if (dense) {
            // w = Sigma g for every requested point (QuadPotentialFull.velocity, quadpotential.py:705-707)
            if (gemm_nt(m, st, P.Greq, ld, C_eval, m->cov, ld, n, (int)ld, 1.0, P.Wreq, ld)) return -1;
            ++launches;
            if (serve && n_mom > 0) {
                ls_gather_z_kernel<<<n_mom, 256, 0, st>>>(P, n_mom, Zb);
                // p0 = L^-T z (solve_triangular(chol.T, z), quadpotential.py:710-713);  v0 = Sigma p0 = L z
                if (gemm_nt(m, st, Zb, ld, n_mom, m->linvT, ld, n, (int)ld, 1.0, P0b, ld)) return -1;
                if (gemm_nt(m, st, Zb, ld, n_mom, m->chol, ld, n, (int)ld, 1.0, V0b, ld)) return -1;
                ls_scatter_mom_kernel<<<n_mom, 256, 0, st>>>(P, n_mom, P0b, V0b);
                CU(cudaGetLastError());
                CU(cudaMemsetAsync(P.counters + 2, 0, sizeof(int), st));
                launches += 4;
            }
        }
        CU(cudaMemsetAsync(P.counters, 0, 2 * sizeof(int), st));
        if (n > 512) ls_advance_kernel<kLsAdvW><<<C, 32 * kLsAdvW, 0, st>>>(P);
        else ls_advance_kernel<1><<<blocks, 128, 0, st>>>(P);
        CU(cudaGetLastError());
        ++launches;
        int h[3];
        CU(cudaMemcpyAsync(h, P.counters, sizeof h, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (h[0] == 0) break;
        n_mom = dense ? h[2] : 0;
        serve = h[1] > 0 || n_mom >= std::max(1, (int)(defer * h[0]));
        if (compact && (h[0] + ctile - 1) / ctile < (C_eval + ctile - 1) / ctile) {
            ls_compact_slots_kernel<<<1, 1024, 0, st>>>(P, new_slot);
            ls_compact_move_kernel<<<C, 256, 0, st>>>(P, new_slot, Qalt);
            CU(cudaGetLastError());
            std::swap(P.Qreq, Qalt);
            C_eval = h[0];
            launches += 2;
        }
    }
    t.stop(launches);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// b200_nuts_run
// ------------------------------------------------------------------------------------------------
struct NutsLaunch {
    b200_model* m; NutsDev P; cudaStream_t st;
    template <class Model, int NPL, int W>
    int operator()(const typename Model::Params& MP) {
        constexpr int NP = 32 * W * NPL;
        constexpr bool SUBS = (W > 1);  // nuts_warp_kernel's default
        const int wpb = (W == 1) ? kNutsWarpChains : 1;  // chains per CTA
        int hot = std::min((W == 1) ? 2 : 1, P.max_td);
        const size_t data = (Model::shared_bytes(MP) + 15) & ~(size_t)15;
        size_t smem = data + (size_t)wpb * nuts_warp_smem_bytes(NP, hot, SUBS, W);
        while (smem > 227 * 1024 && hot > 0) {  // shrink the hot window until the CTA fits
            --hot;
            smem = data + (size_t)wpb * nuts_warp_smem_bytes(NP, hot, SUBS, W);
        }
        if (smem > 227 * 1024) return fail("nuts: shared memory request %zu B exceeds 227 KB", smem);
        P.hot_levels = hot;
        P.scratch_stride = nuts_scratch_doubles(NP, P.max_td);
        // tree scratch [C][stride] | ChainCtx [C] | done [C] | ticket
        const size_t tree_bytes = ((size_t)P.C * P.scratch_stride * sizeof(double) + 255) & ~(size_t)255;
        const size_t ctx_bytes = ((size_t)P.C * sizeof(ChainCtx) + 255) & ~(size_t)255;
        const size_t sched_bytes = ((size_t)(P.C + 1) * sizeof(int) + 255) & ~(size_t)255;
        CU(m->ensure_scratch(tree_bytes + ctx_bytes + sched_bytes));
        char* base = static_cast<char*>(m->scratch);
        P.scratch = reinterpret_cast<double*>(base);
        P.ctx = reinterpret_cast<ChainCtx*>(base + tree_bytes);
        P.done = reinterpret_cast<int*>(base + tree_bytes + ctx_bytes);
        P.ticket = reinterpret_cast<unsigned int*>(P.done + P.C);
        CU(cudaMemsetAsync(P.done, 0, sched_bytes, st));
        auto kern = nuts_warp_kernel<Model, NPL, W>;
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // persistent grid: every CTA resident (teams take (chain, segment) units from the ticket counter)
        const int threads = (W == 1) ? wpb * 32 : 32 * W;
        int per_sm = 0, sms = 148;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
        CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device));
        const int need = (P.C + wpb - 1) / wpb;
        const int blocks = std::max(1, std::min(need, std::max(1, per_sm) * sms));
        // iterations per work unit: fine enough to balance chains of different cost, coarse enough that the ~3 KB state
        // hand-over per unit is noise.  One unit per chain when every chain has its own resident team anyway.
        const int Ttot = P.n_iter;
        const int seg = (need <= blocks) ? Ttot : 50;  // 50 measured (r2): 10 -> 390 ms, 25 -> 370, 50 -> 361, 100 -> 367
        P.seg_iters = std::max(1, std::min(seg, Ttot));
        typename Model::Params MPl;
        if (launch_params<Model>(m, MP, (long long)blocks * wpb, &MPl)) return -1;
        Timer t(st);
        kern<<<blocks, threads, smem, st>>>(P, MPl);
        CU(cudaGetLastError());
        t.stop(1);
        CU(cudaStreamSynchronize(st));
        CU(cudaGetLastError());
        return 0;
    }
};

extern "C" int b200_nuts_run(b200_model* m, const b200_nuts_cfg* cfg, const double* q0, const double* var0,
                             const double* mean0, const double* eps0, b200_pcg64* rng, const double* z,
                             double* draws_out,
                             const b200_stats* stats, const b200_chain_summary* summary, int32_t mem,
                             void* stream) {
    if (!m || !cfg || !q0 || !rng || !draws_out) return fail("b200_nuts_run: null argument");
    const int C = cfg->chains, n = m->n;
    if (C <= 0) return fail("b200_nuts_run: chains must be positive");
    if (cfg->tune < 0 || cfg->draws < 0 || cfg->tune + cfg->draws <= 0) return fail("b200_nuts_run: bad tune/draws");
    if (cfg->max_treedepth < 1 || cfg->max_treedepth > kMaxLevels || cfg->early_max_treedepth < 1 ||
        cfg->early_max_treedepth > cfg->max_treedepth)
        return fail("b200_nuts_run: treedepth must satisfy 1 <= early <= max <= %d", kMaxLevels);
    // GEMM-shaped models always advance in lock step; so does any model under a dense mass matrix (v = Sigma p is a GEMM
    // over all chains on the fp64 tensor path instead of n^2 per chain per leapfrog inside a warp)
    const bool lockstep = is_lockstep_kind(m->kind) || cfg->mass_kind == B200_MASS_DENSE || cfg->mass_kind == B200_MASS_DENSE_ADAPT;
    if (cfg->mass_kind == B200_MASS_DENSE_ADAPT) {
        if (is_lockstep_kind(m->kind)) return fail("b200_nuts_run: DENSE_ADAPT is not wired for the GEMM-shaped models (use a diagonal mass)");
        if (n > kFaMaxN) return fail("b200_nuts_run: DENSE_ADAPT keeps four n x n matrices per chain and supports n <= %d (n = %d)", kFaMaxN, n);
        if (cfg->mass_update_window < 0) return fail("b200_nuts_run: mass_update_window must be >= 0");
        if (cfg->adaptation_window_multiplier < 0) return fail("b200_nuts_run: adaptation_window_multiplier must be >= 0");
        if (!m->ld) m->ld = (long long)((n + 3) & ~3);
    } else if (cfg->mass_kind == B200_MASS_DENSE) {
        if (!m->cov) return fail("b200_nuts_run: mass_kind DENSE needs b200_model_set_dense_mass first");
        if (m->kind == B200_MODEL_LOGISTIC) return fail("b200_nuts_run: dense mass for the logistic GLM is not wired (use a diagonal mass)");
    } else if (cfg->mass_kind == B200_MASS_DIAG_ADAPT_GRAD) {
        if (lockstep) return fail("b200_nuts_run: DIAG_ADAPT_GRAD is implemented by the persistent engine only");
        if (!(cfg->mass_alpha > 0 && cfg->mass_alpha < 1)) return fail("b200_nuts_run: mass_alpha must be in (0, 1)");
    } else if (cfg->mass_kind != B200_MASS_DIAG && cfg->mass_kind != B200_MASS_DIAG_ADAPT) {
        return fail("b200_nuts_run: mass kind %d not implemented", cfg->mass_kind);
    }
    if (cfg->sampler != B200_SAMPLER_NUTS && cfg->sampler != B200_SAMPLER_HMC) return fail("b200_nuts_run: unknown sampler %d", cfg->sampler);
    if (cfg->sampler == B200_SAMPLER_HMC) {
        if (lockstep) return fail("b200_nuts_run: HamiltonianMC is implemented by the persistent engine only");
        if (!(cfg->path_length > 0) || cfg->max_steps < 1) return fail("b200_nuts_run: HMC needs path_length > 0 and max_steps >= 1");
    }
    if (cfg->momentum_source == B200_MOMENTUM_HOST_BUFFER && !z)
        return fail("b200_nuts_run: momentum_source=HOST_BUFFER but z is null");
    if (!(cfg->step_scale > 0)) return fail("b200_nuts_run: step_scale must be > 0");
    if (cfg->adaptation_window < 1) return fail("b200_nuts_run: adaptation_window must be >= 1");
    CU(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // B200_TRACE=1: host-side wall time of the call's phases on stderr (staging | run | copy-out)
    const bool trace = getenv("B200_TRACE") != nullptr;
    const auto tr0 = std::chrono::steady_clock::now();
    auto since = [&](std::chrono::steady_clock::time_point t) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
    };

    // iterations of this call: [it0, it0 + n_iter) of the chain's tune + draws schedule (default: all of it)
    const long long Tsched = (long long)cfg->tune + cfg->draws;
    const long long it0 = cfg->iter_begin;
    if (it0 < 0 || it0 >= Tsched) return fail("b200_nuts_run: iter_begin %lld outside the schedule of %lld iterations", it0, Tsched);
    const long long Ttot = cfg->iter_count > 0 ? cfg->iter_count : Tsched - it0;  // iterations run by this call
    if (it0 + Ttot > Tsched) return fail("b200_nuts_run: iter_begin + iter_count exceeds tune + draws");
    if ((it0 > 0) != (cfg->resume != nullptr)) return fail("b200_nuts_run: iter_begin > 0 needs `resume` (and only then)");
    if ((cfg->resume || cfg->save || it0 > 0 || Ttot != Tsched) && lockstep)
        return fail("b200_nuts_run: partial schedules / chain-state export are implemented by the persistent engine only");
    const long long rec_lo = cfg->store_warmup ? it0 : std::max<long long>(cfg->tune, it0);
    const long long T = std::max<long long>(0, it0 + Ttot - rec_lo);
    const size_t vb = (size_t)C * n * sizeof(double);
    Staged s_q0, s_var0, s_mean0, s_eps0, s_rng, s_z, s_draws;
    // Device staging of host arrays comes from ONE arena kept in the model handle: a steady-state call makes no cudaMalloc /
    // cudaFree at all (measured on the bench boxes, call 8 of round 2: the per-call allocations of five small input arrays
    // cost 0.2-90 ms, and a public-API call took 20-770 ms longer than its kernel).  Everything except the draws (direct
    // host writes, or their own buffer) and a host momentum buffer (parity tests) is lent from it.
    const size_t ct_all = (size_t)C * (size_t)std::max<long long>(0, it0 + Ttot - rec_lo);
    char* lend_p = nullptr;
    size_t lend_left = 0;
    auto up256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
    if (mem == B200_MEM_HOST) {
        size_t need = 3 * up256(vb) + up256((size_t)C * sizeof(double)) + up256((size_t)C * sizeof(b200_pcg64));
        if (stats) need += 12 * up256(ct_all * sizeof(double));
        const size_t state_bytes = 6 * up256(vb) + 9 * up256((size_t)C * sizeof(double));
        if (cfg->resume) need += state_bytes;
        if (cfg->save) need += state_bytes;
        CU(m->ensure_stage(need));
        lend_p = static_cast<char*>(m->stage_arena);
        lend_left = m->stage_bytes;
    }
    auto lend = [&](Staged& s, const void* user, size_t bytes) {
        const size_t b = up256(bytes);
        if (user && lend_p && b <= lend_left) { s.lent = lend_p; lend_p += b; lend_left -= b; }
    };
    lend(s_q0, q0, vb); lend(s_var0, var0, vb); lend(s_mean0, mean0, vb);
    lend(s_eps0, eps0, (size_t)C * sizeof(double)); lend(s_rng, rng, (size_t)C * sizeof(b200_pcg64));
    if (stage_in(s_q0, q0, vb, mem, true, false, st) || stage_in(s_var0, var0, vb, mem, true, false, st) ||
        stage_in(s_mean0, mean0, vb, mem, true, false, st) ||
        stage_in(s_eps0, eps0, (size_t)C * sizeof(double), mem, true, false, st) ||
        stage_in(s_rng, rng, (size_t)C * sizeof(b200_pcg64), mem, true, true, st) ||
        stage_in(s_z, cfg->momentum_source == B200_MOMENTUM_HOST_BUFFER ? z : nullptr, vb * Ttot, mem, true, false, st) ||
        stage_in(s_draws, T > 0 ? draws_out : nullptr, vb * T, mem, false, true, st, /*direct=*/true))
        return -1;
    // stats / summary arrays
    b200_stats ds{};
    b200_chain_summary dsum{};
    Staged st_arr[12], sm_arr[5];
    const size_t ct = (size_t)C * T;
    if (stats) {
        // Sampler statistics are ONE 1-8 byte value per (chain, draw) and array: written straight into host memory they are
        // 12 x C x T single-value PCIe write transactions (24 M for the Radon bench), which costs more link time than the
        // draws themselves.  They are staged in HBM (one arena in the model handle) and leave with 12 DMA copies at the end
        // (143 MB for the Radon bench).  The draws -- 256-byte coalesced row segments -- keep the direct path.
#define B200_ST(i, field, type)                                                              \
    if (stats->field) {                                                                      \
        lend(st_arr[i], stats->field, ct * sizeof(type));                                    \
        if (stage_in(st_arr[i], stats->field, ct * sizeof(type), mem, false, true, st)) return -1; \
        ds.field = (type*)st_arr[i].ptr();                                                   \
    }
        B200_ST(0, depth, int32_t) B200_ST(1, tree_size, int32_t) B200_ST(2, index_in_trajectory, int32_t)
        B200_ST(3, diverging, uint8_t) B200_ST(4, reached_max_treedepth, uint8_t) B200_ST(5, step_size, double)
        B200_ST(6, step_size_bar, double) B200_ST(7, mean_tree_accept, double) B200_ST(8, energy, double)
        B200_ST(9, energy_error, double) B200_ST(10, max_energy_error, double) B200_ST(11, model_logp, double)
#undef B200_ST
    }
    if (summary) {
        if (summary->grad_evals) {
            if (stage_in(sm_arr[0], summary->grad_evals, (size_t)C * sizeof(int64_t), mem, false, true, st, true)) return -1;
            dsum.grad_evals = (int64_t*)sm_arr[0].ptr();
        }
        if (summary->bad_energy_at) {
            if (stage_in(sm_arr[1], summary->bad_energy_at, (size_t)C * sizeof(int32_t), mem, false, true, st, true)) return -1;
            dsum.bad_energy_at = (int32_t*)sm_arr[1].ptr();
        }
        if (summary->final_step_size) {
            if (stage_in(sm_arr[2], summary->final_step_size, (size_t)C * sizeof(double), mem, false, true, st, true)) return -1;
            dsum.final_step_size = (double*)sm_arr[2].ptr();
        }
        if (summary->final_var) {
            if (stage_in(sm_arr[3], summary->final_var, vb, mem, false, true, st, true)) return -1;
            dsum.final_var = (double*)sm_arr[3].ptr();
        }
        if (summary->final_cov && cfg->mass_kind == B200_MASS_DENSE_ADAPT) {
            if (stage_in(sm_arr[4], summary->final_cov, vb * n, mem, false, true, st, true)) return -1;
            dsum.final_cov = (double*)sm_arr[4].ptr();
        }
    }
    // draws of a frozen chain ("bad initial energy") from the failing iteration on are set to NaN by the kernels

    // per-chain state in / out (b200_chain_state): 15 arrays each, staged like every other buffer
    b200_chain_state d_resume{}, d_save{};
    Staged st_state[30];
    {
        const size_t sb = (size_t)C * sizeof(double), ib = (size_t)C * sizeof(int32_t), lb = (size_t)C * sizeof(int64_t);
        int slot = 0;
        auto stage_state = [&](const b200_chain_state* src, b200_chain_state* dst, bool in) -> int {
            if (!src) return 0;
#define B200_SF(field, bytes, type)                                                                       \
    if (!src->field) return fail("b200_nuts_run: chain state field `" #field "` is null");               \
    lend(st_state[slot], src->field, bytes);                                                             \
    if (stage_in(st_state[slot], src->field, bytes, mem, in, !in, st)) return -1;                        \
    dst->field = (type*)st_state[slot++].ptr();
            B200_SF(q, vb, double) B200_SF(log_step, sb, double) B200_SF(log_bar, sb, double) B200_SF(hbar, sb, double)
            B200_SF(da_count, ib, int32_t) B200_SF(n_samples, ib, int32_t) B200_SF(window, ib, int32_t) B200_SF(var, vb, double)
            B200_SF(fg_n, sb, double) B200_SF(fg_mean, vb, double) B200_SF(fg_m2, vb, double) B200_SF(bg_n, sb, double)
            B200_SF(bg_mean, vb, double) B200_SF(bg_m2, vb, double) B200_SF(n_grad, lb, int64_t)
#undef B200_SF
            return 0;
        };
        if (stage_state(cfg->resume, &d_resume, true) || stage_state(cfg->save, &d_save, false)) return -1;
    }

    NutsDev P{};
    P.it0 = (int)it0; P.n_iter = (int)Ttot; P.resume = d_resume; P.save = d_save;
    P.C = C; P.n = n; P.tune = cfg->tune; P.draws = cfg->draws;
    P.max_td = cfg->max_treedepth; P.early_td = cfg->early_max_treedepth;
    P.adapt_step = cfg->adapt_step_size; P.mass_kind = cfg->mass_kind;
    P.momentum_source = cfg->momentum_source; P.store_warmup = cfg->store_warmup;
    P.window = cfg->adaptation_window; P.discard = cfg->discard_window;
    P.eps0 = cfg->step_scale / std::pow((double)n, 0.25);  // base_hmc.py:161
    P.target = cfg->target_accept; P.gamma = cfg->gamma; P.kappa = cfg->k; P.t0 = cfg->t0;
    P.Emax = cfg->Emax; P.init_weight = cfg->mass_initial_weight;
    P.philox_seed = cfg->philox_seed; P.chain_offset = cfg->chain_offset;
    P.sampler = cfg->sampler; P.max_steps = cfg->max_steps; P.path_length = cfg->path_length;
    P.mass_alpha = cfg->mass_alpha; P.stop_adaptation = cfg->stop_adaptation < 0 ? 0x7fffffff : cfg->stop_adaptation;
    P.q0 = (const double*)s_q0.ptr(); P.var0 = (const double*)s_var0.ptr();
    P.mean0 = (const double*)s_mean0.ptr(); P.eps0c = (const double*)s_eps0.ptr(); P.z = (const double*)s_z.ptr();
    P.rng = (b200_pcg64*)s_rng.ptr(); P.draws_out = (double*)s_draws.ptr();
    P.st = ds; P.sm = dsum;
    if (cfg->constrain_draws) {
        if (!m->tr_kind) return fail("b200_nuts_run: constrain_draws needs b200_model_set_transforms first");
        P.tr_kind = m->tr_kind; P.tr_lo = m->tr_lo; P.tr_hi = m->tr_hi;
    }

    const double tr_stage = trace ? since(tr0) : 0.0;
    const auto tr1 = std::chrono::steady_clock::now();
    if (lockstep) {
        LsDev Q{};
        Q.C = C; Q.n = n; Q.tune = P.tune; Q.draws = P.draws; Q.max_td = P.max_td; Q.early_td = P.early_td;
        Q.adapt_step = P.adapt_step; Q.mass_kind = P.mass_kind; Q.momentum_source = P.momentum_source;
        Q.store_warmup = P.store_warmup; Q.window = P.window; Q.discard = P.discard; Q.chain_offset = P.chain_offset;
        Q.dense = (cfg->mass_kind == B200_MASS_DENSE || cfg->mass_kind == B200_MASS_DENSE_ADAPT) ? 1 : 0;
        Q.upd_window = cfg->mass_update_window > 0 ? cfg->mass_update_window : 1;
        Q.win_mult = cfg->adaptation_window_multiplier > 0 ? cfg->adaptation_window_multiplier : 2.0;
        Q.eps0 = P.eps0; Q.target = P.target; Q.gamma = P.gamma; Q.kappa = P.kappa; Q.t0 = P.t0; Q.Emax = P.Emax;
        Q.init_weight = P.init_weight; Q.philox_seed = P.philox_seed;
        Q.q0 = P.q0; Q.var0 = P.var0; Q.mean0 = P.mean0; Q.eps0c = P.eps0c; Q.z = P.z; Q.rng = P.rng;
        Q.draws_out = P.draws_out; Q.st = P.st; Q.sm = P.sm;
        Q.tr_kind = P.tr_kind; Q.tr_lo = P.tr_lo; Q.tr_hi = P.tr_hi;
        if (run_lockstep(m, Q, st)) return -1;
    } else {
        NutsLaunch L{m, P, st};
        // (a chain of the stochastic-volatility model spread over 16 warps instead of 8 was measured and rejected: 16.0 M vs
        // 17.5 M grad-evals/s, the extra cross-warp reduction traffic outweighs the halved per-thread work; profiles/r2_variants.md)
        if (dispatch(m, L)) return -1;
    }

    const double tr_run = trace ? since(tr1) : 0.0;
    const auto tr2 = std::chrono::steady_clock::now();
    if (stage_out(s_rng, st) || stage_out(s_draws, st)) return -1;
    for (auto& s : st_arr) if (stage_out(s, st)) return -1;
    for (auto& s : sm_arr) if (stage_out(s, st)) return -1;
    for (auto& s : st_state) if (stage_out(s, st)) return -1;
    CU(cudaStreamSynchronize(st));
    if (trace)
        fprintf(stderr, "[b200_nuts_run] staging %.2f ms | run %.2f ms (kernels %.2f ms) | copy-out %.2f ms | mem=%s\n", tr_stage, tr_run,
                g_last_ms, since(tr2), mem == B200_MEM_HOST ? "host" : "device");
    return 0;
}

extern "C" int b200_pointwise_loglik(b200_model* m, int32_t lik, const double* draws, int64_t D, double* out, int32_t mem,
                                     void* stream) {
    if (!m || !draws || !out) return fail("b200_pointwise_loglik: null argument");
    if (m->kind != B200_MODEL_IR) return fail("b200_pointwise_loglik: implemented for IR models (b200_ir likelihood factors)");
    if (lik < 0 || lik >= m->ir.n_liks) return fail("b200_pointwise_loglik: likelihood index %d out of range", lik);
    if (D <= 0) return 0;
    CU(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the IR tables live on the device: read the number of observations of this factor back
    IrLikD L;
    CU(cudaMemcpy(&L, m->ir.liks + lik, sizeof L, cudaMemcpyDeviceToHost));
    Staged s_in, s_out;
    if (stage_in(s_in, draws, (size_t)D * m->n * sizeof(double), mem, true, false, st) ||
        stage_in(s_out, out, (size_t)D * (size_t)L.N * sizeof(double), mem, false, true, st))
        return -1;
    const int wpb = 8;
    const int blocks = (int)std::max<long long>(1, std::min<long long>((D + wpb - 1) / wpb, 148 * 8));
    CU(m->ensure_ir_scratch((long long)blocks * wpb));
    Timer t(st);
    ir_pointwise_kernel<<<blocks, wpb * 32, 0, st>>>(m->ir, lik, D, (const double*)s_in.ptr(), (double*)s_out.ptr());
    CU(cudaGetLastError());
    t.stop(1);
    if (stage_out(s_out, st)) return -1;
    CU(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int b200_last_kernel_ms(double* ms, int32_t* launches) {
    if (ms) *ms = g_last_ms;
    if (launches) *launches = g_last_launches;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// fp64 FMA peak micro-benchmark
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
           a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

extern "C" int b200_measure_fp64_tflops(double* tflops) {
    if (!tflops) return fail("null argument");
    const int blocks = 148 * 8, threads = 256, iters = 1 << 14;
    DevBuf out;
    CU(out.alloc((size_t)blocks * threads * sizeof(double)));
    dfma_peak_kernel<<<blocks, threads>>>(out.as<double>(), 64);
    CU(cudaDeviceSynchronize());
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        Timer t(0);
        dfma_peak_kernel<<<blocks, threads>>>(out.as<double>(), iters);
        CU(cudaGetLastError());
        t.stop(1);
        const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
        best = std::max(best, flops / (g_last_ms * 1e-3) / 1e12);
    }
    *tflops = best;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// fp64 tensor-path (DMMA m8n8k4) peak micro-benchmark: roofline denominator of the GEMM-shaped configs
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = 0.0;
    const double a = threadIdx.x * 1e-9, b = 1.0000001;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dmma884(c[i][0], c[i][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" int b200_measure_dmma_tflops(double* tflops) {
    if (!tflops) return fail("null argument");
    const int blocks = 148 * 2, threads = 256, iters = 1 << 12;
    DevBuf out;
    CU(out.alloc((size_t)blocks * threads * sizeof(double)));
    dmma_peak_kernel<<<blocks, threads>>>(out.as<double>(), 16);
    CU(cudaDeviceSynchronize());
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        Timer t(0);
        dmma_peak_kernel<<<blocks, threads>>>(out.as<double>(), iters);
        CU(cudaGetLastError());
        t.stop(1);
        const double flops = 2.0 * 256.0 * 8.0 * (double)iters * blocks * (threads / 32);  // 8x8x4 FMAs per DMMA
        best = std::max(best, flops / (g_last_ms * 1e-3) / 1e12);
    }
    *tflops = best;
    return 0;
}
