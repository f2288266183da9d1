// rv_abi.cu -- the extern "C" boundary of librvgpu.so (see include/rvgpu.h).
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <new>
#include "../../include/rvgpu.h"
#include "rv_launch.h"
#include "rv_loglik.cuh"
#include "rv_model.h"
#include "rv_var.cuh"
#include "rv_map.cuh"
#include "rv_whfast.cuh"
#include "rv_rng.cuh"

struct rv_ctx {
    int device;
    int num_sms, cc_major, cc_minor, clock_khz;
    cudaStream_t stream;
    unsigned long long* d_item_counter;   // work-queue head
    unsigned long long* d_work;           // [2] force evaluations, step attempts
    int count_work;
    long long chain_walkers;              // samplers record only walkers [0, chain_walkers) in chain rows (0 = all)
    // grow-only scratch
    double* d_theta; size_t cap_theta;
    double* d_logp; size_t cap_logp;
    int* d_status; size_t cap_status;
    double* d_part; size_t cap_part;
    int* d_order; size_t cap_order;       // cost-ordered scheduling: order[W], then bin[W]
    int* d_costhist;                      // [2 * RV_COST_BINS]: histogram (kept zero between calls), cursors
    int* d_pstat; size_t cap_pstat;
    double* d_times; size_t cap_times;
    double* d_rv; size_t cap_rv;
    double* d_prop; size_t cap_prop;
    double* d_plogp; size_t cap_plogp;
    int* d_pstatus; size_t cap_pstatus;
    double* d_zz; size_t cap_zz;
    double* d_scales; size_t cap_scales;
    double* d_chain; size_t cap_chain;
    double* d_chainlp; size_t cap_chainlp;
    unsigned long long* d_nacc; size_t cap_nacc;
    unsigned char* d_acc; size_t cap_acc;
    double* d_vpart; size_t cap_vpart;
    double* d_grad; size_t cap_grad;
    double* d_hess; size_t cap_hess;
    double* d_pgrad; size_t cap_pgrad;
    double* d_phess; size_t cap_phess;
    double* d_qf; size_t cap_qf;
    double* d_lascr; size_t cap_lascr;
    int* d_geo; size_t cap_geo;
    int* d_flag; size_t cap_flag;
    double* d_vhist; size_t cap_vhist;
    // maximum-likelihood fit (rv_map_fit)
    double* d_mrows; size_t cap_mrows;    // trial rows [running walkers][n_trial + 1][nvars]
    double* d_mtlogp; size_t cap_mtlogp;
    int* d_mtstat; size_t cap_mtstat;
    double* d_mmu; size_t cap_mmu;        // per-walker damping
    int* d_mfit; size_t cap_mfit;         // fit code[W], n_iter[W]
    int* d_mlist; size_t cap_mlist;       // running list, next running list, evaluation list [W] each; counts[2]
    char err[512];
};
struct rv_obs {
    rv_ctx* ctx;
    double *d_t, *d_rv, *d_err;   // forward [0,nf) then backward [nf,nf+nb)
    int nf, nb;
    double npoints;
};
struct rv_model {
    rv_ctx* ctx;
    rv::Model h;
    rv::Model* d;
    int mapping;
    int cost_order;    // 1 (default): the likelihood kernel takes its items most expensive first (launch_cost_order)
};

static char g_err[512] = "";

static int fail(rv_ctx* ctx, int code, const char* fmt, ...) {
    char* dst = ctx ? ctx->err : g_err;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
    return code;
}
#define CU(ctx, call)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) return fail(ctx, -100, "%s: %s", #call, cudaGetErrorString(e__)); \
    } while (0)
// same, running `cleanup` before the early return (create functions: nothing half-built may leak)
#define CU_OR(ctx, call, cleanup)                                                                  \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            cleanup;                                                                               \
            return fail(ctx, -100, "%s: %s", #call, cudaGetErrorString(e__));                      \
        }                                                                                          \
    } while (0)

template <class T>
static int ensure(rv_ctx* ctx, T** p, size_t* cap, size_t n) {
    if (n <= *cap) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    size_t want = n + n / 4 + 64;
    CU(ctx, cudaMalloc((void**)p, want * sizeof(T)));
    *cap = want;
    return 0;
}

static inline int64_t chain_width(const rv_ctx* ctx, int64_t W) {
    return (ctx->chain_walkers > 0 && ctx->chain_walkers < W) ? (int64_t)ctx->chain_walkers : W;
}

extern "C" {

int rv_ctx_set_option(rv_ctx* ctx, const char* key, double value) {
    if (!ctx || !key) return -1;
    if (!strcmp(key, "chain_walkers")) ctx->chain_walkers = value > 0 ? (long long)value : 0;
    else if (!strcmp(key, "count_work")) ctx->count_work = value != 0.0;
    else return fail(ctx, -20, "rv_ctx_set_option: unknown key '%s'", key);
    return 0;
}

const char* rv_last_error(const rv_ctx* ctx) { return ctx ? ctx->err : g_err; }

int rv_ctx_create(int device, rv_ctx** out) {
    if (!out) return fail(nullptr, -1, "rv_ctx_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, -10, "rv_ctx_create: no CUDA device (%s); librvgpu has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= n) return fail(nullptr, -11, "rv_ctx_create: device %d out of range (0..%d)", device, n - 1);
    rv_ctx* c = new (std::nothrow) rv_ctx();
    if (!c) return fail(nullptr, -12, "rv_ctx_create: out of host memory");
    memset(c, 0, sizeof(*c));
    c->device = device;
    auto drop = [&]() {
        if (c->stream) cudaStreamDestroy(c->stream);
        cudaFree(c->d_item_counter); cudaFree(c->d_work);
        delete c;
    };
    CU_OR(nullptr, cudaSetDevice(device), drop());
    cudaDeviceProp prop;
    CU_OR(nullptr, cudaGetDeviceProperties(&prop, device), drop());
    c->num_sms = prop.multiProcessorCount;
    c->cc_major = prop.major; c->cc_minor = prop.minor;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
    c->clock_khz = khz;
    if (prop.major != 10) {
        delete c;
        return fail(nullptr, -13, "rv_ctx_create: device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major, prop.minor);
    }
    CU_OR(nullptr, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking), drop());
    CU_OR(nullptr, cudaMalloc((void**)&c->d_item_counter, sizeof(unsigned long long)), drop());
    CU_OR(nullptr, cudaMalloc((void**)&c->d_work, 2 * sizeof(unsigned long long)), drop());
    CU_OR(nullptr, cudaMemset(c->d_item_counter, 0, sizeof(unsigned long long)), drop());
    CU_OR(nullptr, cudaMemset(c->d_work, 0, 2 * sizeof(unsigned long long)), drop());
    *out = c;
    return 0;
}

int rv_ctx_destroy(rv_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    cudaFree(c->d_item_counter); cudaFree(c->d_work);
    cudaFree(c->d_theta); cudaFree(c->d_logp); cudaFree(c->d_status); cudaFree(c->d_part);
    cudaFree(c->d_pstat); cudaFree(c->d_times); cudaFree(c->d_rv); cudaFree(c->d_order); cudaFree(c->d_costhist);
    cudaFree(c->d_prop); cudaFree(c->d_plogp); cudaFree(c->d_pstatus); cudaFree(c->d_zz); cudaFree(c->d_scales);
    cudaFree(c->d_chain); cudaFree(c->d_chainlp); cudaFree(c->d_nacc); cudaFree(c->d_acc);
    cudaFree(c->d_vpart); cudaFree(c->d_grad); cudaFree(c->d_hess);
    cudaFree(c->d_pgrad); cudaFree(c->d_phess); cudaFree(c->d_qf); cudaFree(c->d_lascr); cudaFree(c->d_geo); cudaFree(c->d_flag); cudaFree(c->d_vhist);
    cudaFree(c->d_mrows); cudaFree(c->d_mtlogp); cudaFree(c->d_mtstat); cudaFree(c->d_mmu); cudaFree(c->d_mfit); cudaFree(c->d_mlist);
    cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

int rv_device_info(const rv_ctx* c, int* sm_count, int* cc_major, int* cc_minor, int* clock_khz) {
    if (!c) return -1;
    if (sm_count) *sm_count = c->num_sms;
    if (cc_major) *cc_major = c->cc_major;
    if (cc_minor) *cc_minor = c->cc_minor;
    if (clock_khz) *clock_khz = c->clock_khz;
    return 0;
}

int rv_obs_create(rv_ctx* ctx, const double* tf, const double* rvf, const double* errf, int nf,
                  const double* tb, const double* rvb, const double* errb, int nb, double npoints,
                  rv_obs** out) {
    if (!ctx || !out) return fail(ctx, -1, "rv_obs_create: NULL argument");
    if (nf < 0 || nb < 0 || nf + nb == 0) return fail(ctx, -2, "rv_obs_create: empty observation set");
    if ((long long)nf + nb > (1 << 24)) return fail(ctx, -3, "rv_obs_create: %lld epochs exceed the limit of 2^24", (long long)nf + nb);
    CU(ctx, cudaSetDevice(ctx->device));
    rv_obs* o = new (std::nothrow) rv_obs();
    if (!o) return fail(ctx, -12, "out of host memory");
    o->ctx = ctx; o->nf = nf; o->nb = nb; o->npoints = npoints; o->d_t = nullptr;
    const size_t n = (size_t)nf + nb;
    auto drop = [&]() { cudaFree(o->d_t); delete o; };
    CU_OR(ctx, cudaMalloc((void**)&o->d_t, 3 * n * sizeof(double)), drop());
    o->d_rv = o->d_t + n; o->d_err = o->d_t + 2 * n;
    const double* srcs[3][2] = {{tf, tb}, {rvf, rvb}, {errf, errb}};
    double* dsts[3] = {o->d_t, o->d_rv, o->d_err};
    for (int a = 0; a < 3; a++) {
        if (nf) CU_OR(ctx, cudaMemcpyAsync(dsts[a], srcs[a][0], nf * sizeof(double), cudaMemcpyHostToDevice, ctx->stream), drop());
        if (nb) CU_OR(ctx, cudaMemcpyAsync(dsts[a] + nf, srcs[a][1], nb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream), drop());
    }
    CU_OR(ctx, cudaStreamSynchronize(ctx->stream), drop());
    *out = o;
    return 0;
}

int rv_obs_destroy(rv_obs* o) {
    if (!o) return 0;
    cudaSetDevice(o->ctx->device);
    cudaFree(o->d_t);
    delete o;
    return 0;
}

int rv_model_create(rv_ctx* ctx, int n_planets, const double* fixed, int nvars, const int32_t* free_planet,
                    const int32_t* free_elem, double hill_factor, int dims, rv_model** out) {
    if (!ctx || !out || !fixed) return fail(ctx, -1, "rv_model_create: NULL argument");
    rv_model* m = new (std::nothrow) rv_model();
    if (!m) return fail(ctx, -12, "out of host memory");
    m->ctx = ctx; m->mapping = 0; m->cost_order = 1; m->d = nullptr;
    const int rc = rv::build_model(&m->h, n_planets, fixed, nvars, free_planet, free_elem, hill_factor, dims);
    if (rc) {
        delete m;
        return fail(ctx, rc, "rv_model_create: invalid model (code %d): planets must be 1..%d, slots unique and in range, dims 0/2/3", rc, rv::MAXP);
    }
    auto drop = [&]() { cudaFree(m->d); delete m; };
    CU_OR(ctx, cudaSetDevice(ctx->device), drop());
    CU_OR(ctx, cudaMalloc((void**)&m->d, sizeof(rv::Model)), drop());
    CU_OR(ctx, cudaMemcpy(m->d, &m->h, sizeof(rv::Model), cudaMemcpyHostToDevice), drop());
    *out = m;
    return 0;
}

int rv_model_destroy(rv_model* m) {
    if (!m) return 0;
    cudaSetDevice(m->ctx->device);
    cudaFree(m->d);
    delete m;
    return 0;
}

int rv_model_set_option(rv_model* m, const char* key, double value) {
    if (!m || !key) return -1;
    rv_ctx* ctx = m->ctx;
    if (!strcmp(key, "dt0")) m->h.dt0 = value;
    else if (!strcmp(key, "epsilon")) m->h.epsilon = value;
    else if (!strcmp(key, "max_attempts")) m->h.max_attempts = (int)value;
    else if (!strcmp(key, "hill_factor")) m->h.hill_factor = value;
    else if (!strcmp(key, "mapping")) m->mapping = (int)value;
    else if (!strcmp(key, "cost_order")) m->cost_order = value != 0.0;
    else if (!strcmp(key, "check_prior")) m->h.check_prior = value != 0.0;
    else if (!strcmp(key, "monotone_backward")) m->h.monotone_backward = value != 0.0;
    else if (!strcmp(key, "dense_output")) m->h.dense_output = value != 0.0;
    else if (!strcmp(key, "integrator")) {
        if (value != 0.0 && value != 1.0) return fail(ctx, -21, "rv_model_set_option: integrator must be 0 (IAS15) or 1 (WHFast)");
        m->h.integrator = (int)value;
    }
    else return fail(ctx, -20, "rv_model_set_option: unknown key '%s'", key);
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpy(m->d, &m->h, sizeof(rv::Model), cudaMemcpyHostToDevice));
    return 0;
}

static int loglik_dev_impl(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* d_theta,
                           int64_t W, double* d_logp, int32_t* d_status, cudaStream_t s) {
    if (W == 0) return 0;
    if (int rc = ensure(ctx, &ctx->d_part, &ctx->cap_part, (size_t)(2 * W))) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstat, &ctx->cap_pstat, (size_t)(2 * W))) return rc;
    if (model->h.integrator == 1) {
        rv::WhArgs wa;
        memset(&wa, 0, sizeof wa);
        wa.model = model->d; wa.theta = d_theta; wa.W = W;
        wa.ot = obs->d_t; wa.orv = obs->d_rv; wa.oerr = obs->d_err; wa.nf = obs->nf; wa.nb = obs->nb;
        wa.part_chi2 = ctx->d_part; wa.part_status = ctx->d_pstat;
        wa.work_counters = ctx->count_work ? ctx->d_work : nullptr;
        CU(ctx, rv::launch_whfast(wa, model->h.P, model->h.D, ctx->num_sms, s));
        CU(ctx, rv::launch_finalize(ctx->d_part, ctx->d_pstat, W, obs->npoints, d_logp, d_status, ctx->d_item_counter, s));
        return 0;
    }
    rv::LoglikArgs a;
    memset(&a, 0, sizeof a);
    a.model = model->d; a.theta = d_theta; a.W = W;
    a.ot = obs->d_t; a.orv = obs->d_rv; a.oerr = obs->d_err; a.nf = obs->nf; a.nb = obs->nb;
    a.times = nullptr; a.nt = 0; a.rv_out = nullptr;
    a.part_chi2 = ctx->d_part; a.part_status = ctx->d_pstat;
    a.item_counter = ctx->d_item_counter;
    a.work_counters = ctx->count_work ? ctx->d_work : nullptr;
    // batches of more than one wave of items: most expensive walkers first, similar walkers adjacent
    if (model->cost_order && W >= 4096 && W < (int64_t)1 << 31) {
        if (int rc = ensure(ctx, &ctx->d_order, &ctx->cap_order, (size_t)(2 * W))) return rc;
        if (!ctx->d_costhist) {
            CU(ctx, cudaMalloc((void**)&ctx->d_costhist, 2 * rv::RV_COST_BINS * sizeof(int)));
            CU(ctx, cudaMemsetAsync(ctx->d_costhist, 0, 2 * rv::RV_COST_BINS * sizeof(int), s));
        }
        CU(ctx, rv::launch_cost_order(model->d, d_theta, W, ctx->d_order + W, ctx->d_costhist, ctx->d_costhist + rv::RV_COST_BINS,
                                      ctx->d_order, s));
        a.order = ctx->d_order;
    }
    CU(ctx, rv::launch_loglik(a, model->h.P, model->h.D, model->mapping, model->h.dense_output, ctx->num_sms, s));
    CU(ctx, rv::launch_finalize(ctx->d_part, ctx->d_pstat, W, obs->npoints, d_logp, d_status, ctx->d_item_counter, s));
    return 0;
}

int rv_loglik_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* d_theta, int64_t W,
                  double* d_logp, int32_t* d_status, void* stream) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_loglik_dev: NULL handle");
    if (W < 0) return fail(ctx, -2, "rv_loglik_dev: negative W");
    CU(ctx, cudaSetDevice(ctx->device));
    return loglik_dev_impl(ctx, model, obs, d_theta, W, d_logp, d_status, (cudaStream_t)stream);
}

int rv_loglik(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* theta, int64_t W,
              double* logp, int32_t* status) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_loglik: NULL handle");
    if (W < 0) return fail(ctx, -2, "rv_loglik: negative W");
    if (W == 0) return 0;
    if (!theta || !logp || !status) return fail(ctx, -1, "rv_loglik: NULL buffer");
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t nv = (size_t)(model->h.nvars > 0 ? model->h.nvars : 1);
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nv)) return rc;
    if (int rc = ensure(ctx, &ctx->d_logp, &ctx->cap_logp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    cudaStream_t s = ctx->stream;
    if (model->h.nvars > 0)
        CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * model->h.nvars * sizeof(double), cudaMemcpyHostToDevice, s));
    if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_theta, W, ctx->d_logp, ctx->d_status, s)) return rc;
    CU(ctx, cudaMemcpyAsync(logp, ctx->d_logp, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(status, ctx->d_status, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

int rv_rv_curve(rv_ctx* ctx, const rv_model* model, const double* theta, int64_t W, const double* times,
                int nt, double* rv, int32_t* status) {
    if (!ctx || !model) return fail(ctx, -1, "rv_rv_curve: NULL handle");
    if (W < 0 || nt < 0) return fail(ctx, -2, "rv_rv_curve: negative size");
    if (W == 0) return 0;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t nv = (size_t)(model->h.nvars > 0 ? model->h.nvars : 1);
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nv)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstat, &ctx->cap_pstat, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_times, &ctx->cap_times, (size_t)(nt > 0 ? nt : 1))) return rc;
    if (int rc = ensure(ctx, &ctx->d_rv, &ctx->cap_rv, (size_t)W * (size_t)(nt > 0 ? nt : 1))) return rc;
    cudaStream_t s = ctx->stream;
    if (model->h.nvars > 0)
        CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * model->h.nvars * sizeof(double), cudaMemcpyHostToDevice, s));
    if (nt) CU(ctx, cudaMemcpyAsync(ctx->d_times, times, (size_t)nt * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemsetAsync(ctx->d_rv, 0, (size_t)W * (size_t)(nt > 0 ? nt : 1) * sizeof(double), s));
    if (model->h.integrator == 1) {
        rv::WhArgs wa;
        memset(&wa, 0, sizeof wa);
        wa.model = model->d; wa.theta = ctx->d_theta; wa.W = W;
        wa.times = ctx->d_times; wa.nt = nt; wa.rv_out = ctx->d_rv; wa.part_status = ctx->d_pstat;
        wa.work_counters = ctx->count_work ? ctx->d_work : nullptr;
        CU(ctx, rv::launch_whfast(wa, model->h.P, model->h.D, ctx->num_sms, s));
        if (nt) CU(ctx, cudaMemcpyAsync(rv, ctx->d_rv, (size_t)W * nt * sizeof(double), cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaMemcpyAsync(status, ctx->d_pstat, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaStreamSynchronize(s));
        return 0;
    }
    rv::LoglikArgs a;
    memset(&a, 0, sizeof a);
    a.model = model->d; a.theta = ctx->d_theta; a.W = W;
    a.nf = 0; a.nb = 0;
    a.times = ctx->d_times; a.nt = nt; a.rv_out = ctx->d_rv;
    a.part_chi2 = nullptr; a.part_status = ctx->d_pstat;
    a.item_counter = ctx->d_item_counter;
    a.work_counters = ctx->count_work ? ctx->d_work : nullptr;
    CU(ctx, rv::launch_loglik(a, model->h.P, model->h.D, model->mapping, model->h.dense_output, ctx->num_sms, s));
    CU(ctx, rv::launch_curve_finalize(ctx->d_item_counter, s));
    if (nt) CU(ctx, cudaMemcpyAsync(rv, ctx->d_rv, (size_t)W * nt * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(status, ctx->d_pstat, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

int rv_initial_conditions(rv_ctx* ctx, const rv_model* model, const double* theta, int64_t W, double* particles,
                          int32_t* status) {
    if (!ctx || !model) return fail(ctx, -1, "rv_initial_conditions: NULL handle");
    if (W < 0) return fail(ctx, -2, "rv_initial_conditions: negative W");
    if (W == 0) return 0;
    if (!particles || !status) return fail(ctx, -1, "rv_initial_conditions: NULL buffer");
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t nv = (size_t)(model->h.nvars > 0 ? model->h.nvars : 1);
    const size_t np7 = (size_t)(model->h.P + 1) * 7;
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nv)) return rc;
    if (int rc = ensure(ctx, &ctx->d_rv, &ctx->cap_rv, (size_t)W * np7)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    cudaStream_t s = ctx->stream;
    if (model->h.nvars > 0)
        CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * model->h.nvars * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(ctx, rv::launch_initial_conditions(model->d, ctx->d_theta, W, ctx->d_rv, ctx->d_status, s));
    CU(ctx, cudaMemcpyAsync(particles, ctx->d_rv, (size_t)W * np7 * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(status, ctx->d_status, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// value + gradient + Hessian

// 0 when launch_var has a configuration for this model, else -31 (WHFast) or -30 (too many planets / parameters)
static int var_refusal(rv_ctx* ctx, const rv_model* model) {
    const int nv = model->h.nvars;
    if (model->h.integrator != 0)
        return fail(ctx, -31, "the variational (gradient + Hessian) path integrates with IAS15 only; set integrator = 0");
    if (model->h.P > rv::MAXP_VAR)
        return fail(ctx, -30, "variational kernel: built for up to %d planets (this model has %d); the plain likelihood, MH and the stretch move take up to %d",
                    rv::MAXP_VAR, model->h.P, rv::MAXP);
    // models whose (set, planet) threads do not fit one CTA run their second-order sets in chunks (launch_var_chunked); what must
    // fit is the real + first-order group beside at least one pair -- true for everything the schema allows (5 planets x 7 elements:
    // 180 threads of 320)
    if (!rv::var_model_fits(model->h.P, model->h.D, nv))
        return fail(ctx, -30, "variational kernel: %d planets x %d free parameters: the real and first-order sets alone need %d threads of one block",
                    model->h.P, nv, (nv + 1) * model->h.P);
    return 0;
}

// check_prior is a per-call argument: the samplers always test priorHard (mcmc.py:171), whatever the model option says;
// the plain entry points follow the model option (default 1), rv_loglik_d_dd_opt takes it from the caller.
static int var_dev_impl(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* d_theta, int64_t W,
                        double* d_logp, double* d_grad, double* d_hess, int32_t* d_status, int check_prior, cudaStream_t s) {
    if (W == 0) return 0;
    if (int rc = var_refusal(ctx, model)) return rc;
    const int nv = model->h.nvars;
    const int nsets = rv::var_nsets(nv);
    if (int rc = ensure(ctx, &ctx->d_vpart, &ctx->cap_vpart, (size_t)(2 * W) * nsets)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstat, &ctx->cap_pstat, (size_t)(2 * W))) return rc;
    rv::VarArgs a;
    memset(&a, 0, sizeof a);
    a.model = model->d; a.theta = d_theta; a.W = W;
    a.ot = obs->d_t; a.orv = obs->d_rv; a.oerr = obs->d_err; a.nf = obs->nf; a.nb = obs->nb;
    a.npoints = obs->npoints;
    a.check_prior = check_prior ? 1 : 0;
    a.part = ctx->d_vpart; a.part_status = ctx->d_pstat;
    a.item_counter = ctx->d_item_counter;
    a.work_counters = ctx->count_work ? ctx->d_work : nullptr;
    const size_t nh = rv::var_hist_doubles_needed(model->h.P, model->h.D, nv, ctx->num_sms);
    if (nh) { if (int rc = ensure(ctx, &ctx->d_vhist, &ctx->cap_vhist, nh)) return rc; }
    a.hist = ctx->d_vhist; a.hist_doubles = ctx->cap_vhist;
    CU(ctx, rv::launch_var(a, model->h.P, model->h.D, nv, ctx->num_sms, s));
    CU(ctx, rv::launch_var_finalize(ctx->d_vpart, ctx->d_pstat, W, nv, d_logp, d_grad, d_hess, d_status, ctx->d_item_counter, s));
    return 0;
}

int rv_loglik_d_dd_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* d_theta, int64_t W,
                       double* d_logp, double* d_grad, double* d_hess, int32_t* d_status, void* stream) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_loglik_d_dd_dev: NULL handle");
    if (W < 0) return fail(ctx, -2, "rv_loglik_d_dd_dev: negative W");
    CU(ctx, cudaSetDevice(ctx->device));
    return var_dev_impl(ctx, model, obs, d_theta, W, d_logp, d_grad, d_hess, d_status, model->h.check_prior, (cudaStream_t)stream);
}

int rv_loglik_d_dd(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* theta, int64_t W,
                   double* logp, double* grad, double* hess, int32_t* status) {
    if (!model) return fail(ctx, -1, "rv_loglik_d_dd: NULL handle");
    return rv_loglik_d_dd_opt(ctx, model, obs, theta, W, model->h.check_prior, logp, grad, hess, status);
}

int rv_loglik_d_dd_opt(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* theta, int64_t W,
                       int check_prior, double* logp, double* grad, double* hess, int32_t* status) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_loglik_d_dd: NULL handle");
    if (W < 0) return fail(ctx, -2, "rv_loglik_d_dd: negative W");
    if (W == 0) return 0;
    if (!theta || !logp || !grad || !hess || !status) return fail(ctx, -1, "rv_loglik_d_dd: NULL buffer");
    CU(ctx, cudaSetDevice(ctx->device));
    const int nv = model->h.nvars;
    const size_t nvs = (size_t)(nv > 0 ? nv : 1);
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_logp, &ctx->cap_logp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_grad, &ctx->cap_grad, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_hess, &ctx->cap_hess, (size_t)W * nvs * nvs)) return rc;
    cudaStream_t s = ctx->stream;
    if (nv > 0) CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * nv * sizeof(double), cudaMemcpyHostToDevice, s));
    if (int rc = var_dev_impl(ctx, model, obs, ctx->d_theta, W, ctx->d_logp, ctx->d_grad, ctx->d_hess, ctx->d_status, check_prior, s)) return rc;
    CU(ctx, cudaMemcpyAsync(logp, ctx->d_logp, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(status, ctx->d_status, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (nv > 0) {
        CU(ctx, cudaMemcpyAsync(grad, ctx->d_grad, (size_t)W * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaMemcpyAsync(hess, ctx->d_hess, (size_t)W * nv * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// maximum-likelihood fit: damped saddle-free Newton per walker, batched line search (DESIGN.md 3.6)

// One iteration: (1) the variational evaluation of the walkers whose theta moved (or that are new), gathered into one
// contiguous batch and scattered back; (2) the Newton step of every running walker, n_trial + 1 rows each; (3) one plain
// likelihood launch over all rows; (4) selection + compaction into the next running / evaluation lists.  The host reads
// the two list lengths once per iteration; the loop ends when no walker runs.
static int map_fit_impl(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, int64_t W, int max_iter, int n_trial,
                        double tol, double damping0, cudaStream_t s) {
    const int nv = model->h.nvars;
    const size_t nvs = (size_t)nv, R = (size_t)n_trial + 1;
    if (int rc = ensure(ctx, &ctx->d_prop, &ctx->cap_prop, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_plogp, &ctx->cap_plogp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstatus, &ctx->cap_pstatus, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pgrad, &ctx->cap_pgrad, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_phess, &ctx->cap_phess, (size_t)W * nvs * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_lascr, &ctx->cap_lascr, (size_t)W * 2 * nvs * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_mrows, &ctx->cap_mrows, (size_t)W * R * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_mtlogp, &ctx->cap_mtlogp, (size_t)W * R)) return rc;
    if (int rc = ensure(ctx, &ctx->d_mtstat, &ctx->cap_mtstat, (size_t)W * R)) return rc;
    if (int rc = ensure(ctx, &ctx->d_mmu, &ctx->cap_mmu, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_mfit, &ctx->cap_mfit, (size_t)2 * W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_mlist, &ctx->cap_mlist, (size_t)3 * W + 2)) return rc;
    int* code = ctx->d_mfit;
    int* iters = ctx->d_mfit + W;
    int* run = ctx->d_mlist;
    int* run_next = ctx->d_mlist + W;
    int* eval = ctx->d_mlist + 2 * W;
    int* counts = ctx->d_mlist + 3 * W;
    CU(ctx, rv::launch_map_init(W, damping0, code, iters, ctx->d_mmu, run, eval, s));
    long long n_run = W, n_eval = W;
    while (n_run > 0) {
        if (n_eval > 0) {
            CU(ctx, rv::launch_map_gather(eval, n_eval, ctx->d_theta, nv, ctx->d_prop, s));
            if (int rc = var_dev_impl(ctx, model, obs, ctx->d_prop, n_eval, ctx->d_plogp, ctx->d_pgrad, ctx->d_phess,
                                      ctx->d_pstatus, 1, s)) return rc;
            CU(ctx, rv::launch_map_scatter(eval, n_eval, nv, ctx->d_plogp, ctx->d_pgrad, ctx->d_phess, ctx->d_pstatus,
                                           ctx->d_logp, ctx->d_grad, ctx->d_hess, ctx->d_status, code, iters, s));
        }
        CU(ctx, rv::launch_map_step(run, n_run, nv, ctx->d_theta, ctx->d_grad, ctx->d_hess, ctx->d_mmu, iters, code, max_iter,
                                    tol, n_trial, ctx->d_mrows, ctx->d_lascr, s));
        if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_mrows, n_run * (int64_t)R, ctx->d_mtlogp, ctx->d_mtstat, s)) return rc;
        CU(ctx, cudaMemsetAsync(counts, 0, 2 * sizeof(int), s));
        CU(ctx, rv::launch_map_select(run, n_run, nv, n_trial, ctx->d_mrows, ctx->d_mtlogp, ctx->d_mtstat, ctx->d_theta,
                                      ctx->d_mmu, iters, code, run_next, eval, counts, s));
        int h[2];
        CU(ctx, cudaMemcpyAsync(h, counts, sizeof h, cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaStreamSynchronize(s));
        n_run = h[0]; n_eval = h[1];
        int* t = run; run = run_next; run_next = t;
    }
    return 0;
}

int rv_map_fit(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, int64_t W, int max_iter, int n_trial,
               double tol, double damping0, double* logp, double* grad, double* hess, int32_t* status, int32_t* fit_code,
               int32_t* n_iter) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_map_fit: NULL handle");
    if (W < 0 || W >= ((int64_t)1 << 31)) return fail(ctx, -2, "rv_map_fit: W = %lld out of range [0, 2^31)", (long long)W);
    if (n_trial < 1 || n_trial > rv::MAP_MAX_TRIAL)
        return fail(ctx, -2, "rv_map_fit: n_trial = %d out of range 1..%d", n_trial, rv::MAP_MAX_TRIAL);
    if (max_iter < 0) return fail(ctx, -2, "rv_map_fit: negative max_iter");
    if (!(tol >= 0.0) || !(damping0 >= 0.0) || !isfinite(damping0))
        return fail(ctx, -2, "rv_map_fit: tol and damping must be finite and >= 0");
    const int nv = model->h.nvars;
    if (nv < 1) return fail(ctx, -2, "rv_map_fit: the model has no free parameter");
    if (int rc = var_refusal(ctx, model)) return rc;
    if (W == 0) return 0;
    if (!theta || !logp || !status || !fit_code || !n_iter) return fail(ctx, -1, "rv_map_fit: NULL buffer");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t nvs = (size_t)nv;
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_logp, &ctx->cap_logp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_grad, &ctx->cap_grad, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_hess, &ctx->cap_hess, (size_t)W * nvs * nvs)) return rc;
    CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * nvs * sizeof(double), cudaMemcpyHostToDevice, s));
    if (int rc = map_fit_impl(ctx, model, obs, W, max_iter, n_trial, tol, damping0, s)) return rc;
    CU(ctx, cudaMemcpyAsync(theta, ctx->d_theta, (size_t)W * nvs * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(logp, ctx->d_logp, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(status, ctx->d_status, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(fit_code, ctx->d_mfit, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(n_iter, ctx->d_mfit + W, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (grad) CU(ctx, cudaMemcpyAsync(grad, ctx->d_grad, (size_t)W * nvs * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (hess) CU(ctx, cudaMemcpyAsync(hess, ctx->d_hess, (size_t)W * nvs * nvs * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// samplers

static int mh_steps_impl(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* d_theta, double* d_logp,
                         const double* d_scales, double step_size, uint64_t seed, uint64_t first_id, uint32_t first_step,
                         int nsteps, int thin, int64_t W, unsigned long long* d_nacc, unsigned char* d_acc_rows,
                         double* d_chain, double* d_chainlp, cudaStream_t s) {
    const int nv = model->h.nvars;
    const int64_t CW = chain_width(ctx, W);
    if (int rc = ensure(ctx, &ctx->d_prop, &ctx->cap_prop, (size_t)W * (nv > 0 ? nv : 1))) return rc;
    if (int rc = ensure(ctx, &ctx->d_plogp, &ctx->cap_plogp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstatus, &ctx->cap_pstatus, (size_t)W)) return rc;
    long long row = 0;
    for (int k = 0; k < nsteps; k++) {
        const unsigned step = first_step + (unsigned)k;
        CU(ctx, rv::launch_mh_propose(d_theta, d_scales, step_size, nv, W, seed, first_id, step, ctx->d_prop, s));
        if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_prop, W, ctx->d_plogp, ctx->d_pstatus, s)) return rc;
        const bool rec = d_chain && thin > 0 && ((k + 1) % thin == 0);
        CU(ctx, rv::launch_mh_accept(d_theta, d_logp, ctx->d_prop, ctx->d_plogp, ctx->d_pstatus, nv, W, seed, first_id, step,
                                     d_nacc, d_acc_rows ? d_acc_rows + (size_t)k * W : nullptr,
                                     rec ? d_chain + (size_t)row * CW * nv : nullptr,
                                     rec ? d_chainlp + (size_t)row * CW : nullptr, CW, s));
        if (rec) row++;
    }
    return 0;
}

int rv_mh_steps_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* d_theta, double* d_logp,
                    const double* d_scales, double step_size, uint64_t seed, uint64_t first_chain_id,
                    uint32_t first_step, int nsteps, int64_t W, uint64_t* d_n_accept, void* stream) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_mh_steps_dev: NULL handle");
    if (W <= 0 || nsteps < 0) return fail(ctx, -2, "rv_mh_steps_dev: bad size");
    CU(ctx, cudaSetDevice(ctx->device));
    return mh_steps_impl(ctx, model, obs, d_theta, d_logp, d_scales, step_size, seed, first_chain_id, first_step, nsteps, 0,
                         W, (unsigned long long*)d_n_accept, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int rv_mh_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, int have_logp,
              const double* scales, double step_size, uint64_t seed, uint64_t first_chain_id, uint32_t first_step,
              int nsteps, int thin, int64_t W, double* chain, double* chain_logp, uint64_t* n_accept,
              uint8_t* accepted) {
    if (!ctx || !model || !obs || !theta || !logp || !scales) return fail(ctx, -1, "rv_mh_run: NULL argument");
    if (W <= 0 || nsteps < 0) return fail(ctx, -2, "rv_mh_run: bad size");
    if (thin < 1) thin = 1;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int nv = model->h.nvars;
    const size_t nvs = (size_t)(nv > 0 ? nv : 1);
    const long long rows = chain ? nsteps / thin : 0;
    const int64_t CW = chain_width(ctx, W);
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_logp, &ctx->cap_logp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_scales, &ctx->cap_scales, nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_nacc, &ctx->cap_nacc, (size_t)W)) return rc;
    if (rows) {
        if (int rc = ensure(ctx, &ctx->d_chain, &ctx->cap_chain, (size_t)rows * CW * nvs)) return rc;
        if (int rc = ensure(ctx, &ctx->d_chainlp, &ctx->cap_chainlp, (size_t)rows * CW)) return rc;
    }
    if (accepted) if (int rc = ensure(ctx, &ctx->d_acc, &ctx->cap_acc, (size_t)nsteps * W + 1)) return rc;
    CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * nv * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemcpyAsync(ctx->d_scales, scales, (size_t)nv * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemsetAsync(ctx->d_nacc, 0, (size_t)W * sizeof(unsigned long long), s));
    if (have_logp) {
        CU(ctx, cudaMemcpyAsync(ctx->d_logp, logp, (size_t)W * sizeof(double), cudaMemcpyHostToDevice, s));
    } else {
        if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_theta, W, ctx->d_logp, ctx->d_status, s)) return rc;
        CU(ctx, rv::launch_mask_logp(ctx->d_logp, ctx->d_status, W, s));
    }
    if (int rc = mh_steps_impl(ctx, model, obs, ctx->d_theta, ctx->d_logp, ctx->d_scales, step_size, seed, first_chain_id,
                               first_step, nsteps, thin, W, ctx->d_nacc, accepted ? ctx->d_acc : nullptr,
                               rows ? ctx->d_chain : nullptr, rows ? ctx->d_chainlp : nullptr, s)) return rc;
    CU(ctx, cudaMemcpyAsync(theta, ctx->d_theta, (size_t)W * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(logp, ctx->d_logp, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (rows) {
        CU(ctx, cudaMemcpyAsync(chain, ctx->d_chain, (size_t)rows * CW * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (chain_logp) CU(ctx, cudaMemcpyAsync(chain_logp, ctx->d_chainlp, (size_t)rows * CW * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    if (n_accept) CU(ctx, cudaMemcpyAsync(n_accept, ctx->d_nacc, (size_t)W * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (accepted) CU(ctx, cudaMemcpyAsync(accepted, ctx->d_acc, (size_t)nsteps * W, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

static int stretch_half_impl(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* d_S, int64_t nS,
                             uint64_t id0_S, const double* d_C, int64_t nC, double* d_lnp_S, double a, uint64_t seed,
                             uint32_t step, uint32_t half, unsigned long long* d_nacc, unsigned char* d_acc,
                             cudaStream_t s) {
    const int nv = model->h.nvars;
    if (int rc = ensure(ctx, &ctx->d_prop, &ctx->cap_prop, (size_t)nS * (nv > 0 ? nv : 1))) return rc;
    if (int rc = ensure(ctx, &ctx->d_plogp, &ctx->cap_plogp, (size_t)nS)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstatus, &ctx->cap_pstatus, (size_t)nS)) return rc;
    if (int rc = ensure(ctx, &ctx->d_zz, &ctx->cap_zz, (size_t)nS)) return rc;
    CU(ctx, rv::launch_stretch_propose(d_S, d_C, nv, nS, nC, a, seed, id0_S, step, half, ctx->d_prop, ctx->d_zz, s));
    if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_prop, nS, ctx->d_plogp, ctx->d_pstatus, s)) return rc;
    CU(ctx, rv::launch_stretch_accept(d_S, d_lnp_S, ctx->d_prop, ctx->d_plogp, ctx->d_pstatus, ctx->d_zz, nv, nS, seed, id0_S,
                                      step, half, d_nacc, d_acc, s));
    return 0;
}

int rv_stretch_half_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* d_S, int64_t nS,
                        uint64_t id0_S, const double* d_C, int64_t nC, double* d_lnp_S, double a, uint64_t seed,
                        uint32_t step, uint32_t half, uint64_t* d_n_accept, uint8_t* d_accepted, void* stream) {
    if (!ctx || !model || !obs) return fail(ctx, -1, "rv_stretch_half_dev: NULL handle");
    if (nS <= 0 || nC <= 0) return fail(ctx, -2, "rv_stretch_half_dev: empty half");
    CU(ctx, cudaSetDevice(ctx->device));
    return stretch_half_impl(ctx, model, obs, d_S, nS, id0_S, d_C, nC, d_lnp_S, a, seed, step, half,
                             (unsigned long long*)d_n_accept, d_accepted, (cudaStream_t)stream);
}

int rv_stretch_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* lnp, int have_lnp,
                   double a, uint64_t seed, uint32_t first_step, int nsteps, int thin, int64_t W, double* chain,
                   double* chain_lnp, uint64_t* n_accept, uint8_t* accepted) {
    if (!ctx || !model || !obs || !theta || !lnp) return fail(ctx, -1, "rv_stretch_run: NULL argument");
    if (W < 2 || (W & 1)) return fail(ctx, -2, "rv_stretch_run: the number of walkers must be even (emcee asserts the same)");
    if (nsteps < 0) return fail(ctx, -2, "rv_stretch_run: negative nsteps");
    if (thin < 1) thin = 1;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int nv = model->h.nvars;
    const size_t nvs = (size_t)(nv > 0 ? nv : 1);
    const long long rows = chain ? nsteps / thin : 0;
    const int64_t h = W / 2;
    const int64_t CW = chain_width(ctx, W);
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_logp, &ctx->cap_logp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_nacc, &ctx->cap_nacc, (size_t)W)) return rc;
    if (rows) {
        if (int rc = ensure(ctx, &ctx->d_chain, &ctx->cap_chain, (size_t)rows * CW * nvs)) return rc;
        if (int rc = ensure(ctx, &ctx->d_chainlp, &ctx->cap_chainlp, (size_t)rows * CW)) return rc;
    }
    if (accepted) if (int rc = ensure(ctx, &ctx->d_acc, &ctx->cap_acc, (size_t)nsteps * W + 1)) return rc;
    CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * nv * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemsetAsync(ctx->d_nacc, 0, (size_t)W * sizeof(unsigned long long), s));
    if (have_lnp) {
        CU(ctx, cudaMemcpyAsync(ctx->d_logp, lnp, (size_t)W * sizeof(double), cudaMemcpyHostToDevice, s));
    } else {
        if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_theta, W, ctx->d_logp, ctx->d_status, s)) return rc;
        CU(ctx, rv::launch_mask_logp(ctx->d_logp, ctx->d_status, W, s));
    }
    long long row = 0;
    for (int k = 0; k < nsteps; k++) {
        const unsigned step = first_step + (unsigned)k;
        for (unsigned half = 0; half < 2; half++) {
            double* S = ctx->d_theta + (half == 0 ? 0 : (size_t)h * nv);
            const double* C = ctx->d_theta + (half == 0 ? (size_t)h * nv : 0);
            const uint64_t id0 = half == 0 ? 0 : (uint64_t)h;
            if (int rc = stretch_half_impl(ctx, model, obs, S, h, id0, C, h, ctx->d_logp + id0, a, seed, step, half,
                                           ctx->d_nacc + id0, accepted ? ctx->d_acc + (size_t)k * W + id0 : nullptr, s)) return rc;
        }
        if (rows && ((k + 1) % thin == 0)) {
            CU(ctx, cudaMemcpyAsync(ctx->d_chain + (size_t)row * CW * nv, ctx->d_theta, (size_t)CW * nv * sizeof(double), cudaMemcpyDeviceToDevice, s));
            CU(ctx, cudaMemcpyAsync(ctx->d_chainlp + (size_t)row * CW, ctx->d_logp, (size_t)CW * sizeof(double), cudaMemcpyDeviceToDevice, s));
            row++;
        }
    }
    CU(ctx, cudaMemcpyAsync(theta, ctx->d_theta, (size_t)W * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(lnp, ctx->d_logp, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (rows) {
        CU(ctx, cudaMemcpyAsync(chain, ctx->d_chain, (size_t)rows * CW * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (chain_lnp) CU(ctx, cudaMemcpyAsync(chain_lnp, ctx->d_chainlp, (size_t)rows * CW * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    if (n_accept) CU(ctx, cudaMemcpyAsync(n_accept, ctx->d_nacc, (size_t)W * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (accepted) CU(ctx, cudaMemcpyAsync(accepted, ctx->d_acc, (size_t)nsteps * W, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// The stretch ensemble over several GPUs of ONE process (SURVEY 8(b): a context group driving several GPUs).
// Every GPU holds the whole ensemble (theta[W][nv], lnp[W]); GPU g owns the g-th slice of each half.  Per half-step each GPU
// proposes for its slice against the complementary half of ITS copy, integrates, and its accept kernel stores accepted walkers
// into all copies over peer memory.  A half-step on GPU g may start once every GPU has finished the previous one (events).
int rv_stretch_run_multi(int n_gpus, rv_ctx* const* ctxs, const rv_model* const* models, const rv_obs* const* obss,
                         double* theta, double* lnp, int have_lnp, double a, uint64_t seed, uint32_t first_step, int nsteps,
                         int thin, int64_t W, double* chain, double* chain_lnp, uint64_t* n_accept) {
    rv_ctx* c0 = (n_gpus > 0 && ctxs) ? ctxs[0] : nullptr;
    if (n_gpus < 1 || n_gpus > rv::RV_MAX_GROUP || !ctxs || !models || !obss || !theta || !lnp)
        return fail(c0, -1, "rv_stretch_run_multi: bad argument (1..%d GPUs)", rv::RV_MAX_GROUP);
    for (int g = 0; g < n_gpus; g++)
        if (!ctxs[g] || !models[g] || !obss[g]) return fail(c0, -1, "rv_stretch_run_multi: NULL handle for GPU %d", g);
    const int G = n_gpus;
    if (W < 2 || (W & 1) || (W / 2) % G) return fail(c0, -2, "rv_stretch_run_multi: %lld walkers do not split into two halves of %d equal slices", (long long)W, G);
    if (nsteps < 0) return fail(c0, -2, "rv_stretch_run_multi: negative nsteps");
    if (thin < 1) thin = 1;
    const int nv = models[0]->h.nvars;
    for (int g = 1; g < G; g++)
        if (models[g]->h.nvars != nv || models[g]->h.P != models[0]->h.P) return fail(c0, -2, "rv_stretch_run_multi: the models differ");
    const size_t nvs = (size_t)(nv > 0 ? nv : 1);
    const int64_t h = W / 2, n_loc = h / G;
    const long long rows = chain ? nsteps / thin : 0;
    rv::PeerCopies pc;
    memset(&pc, 0, sizeof pc);
    pc.n = G;
    unsigned long long* d_nacc[rv::RV_MAX_GROUP] = {nullptr};
    cudaEvent_t ev[rv::RV_MAX_GROUP][2];
    memset(ev, 0, sizeof ev);
    double *d_chain = nullptr, *d_chainlp = nullptr;
    int rc = 0;
    auto cleanup = [&]() {
        for (int g = 0; g < G; g++) {
            cudaSetDevice(ctxs[g]->device);
            cudaStreamSynchronize(ctxs[g]->stream);
            cudaFree(pc.theta[g]); cudaFree(pc.lnp[g]); cudaFree(d_nacc[g]);
            for (int k = 0; k < 2; k++) if (ev[g][k]) cudaEventDestroy(ev[g][k]);
        }
        cudaSetDevice(ctxs[0]->device);
        cudaFree(d_chain); cudaFree(d_chainlp);
    };
#define CUM(ctx, call)                                                                                 \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            rc = fail(ctx, -100, "%s: %s", #call, cudaGetErrorString(e__));                            \
            cleanup();                                                                                 \
            return rc;                                                                                 \
        }                                                                                              \
    } while (0)
    // peer access, buffers, events
    for (int g = 0; g < G; g++) {
        rv_ctx* c = ctxs[g];
        CUM(c, cudaSetDevice(c->device));
        for (int q = 0; q < G; q++) {
            if (q == g || ctxs[q]->device == c->device) continue;
            int can = 0;
            CUM(c, cudaDeviceCanAccessPeer(&can, c->device, ctxs[q]->device));
            if (!can) { rc = fail(c0, -40, "rv_stretch_run_multi: GPU %d cannot map GPU %d's memory (no peer access)", c->device, ctxs[q]->device); cleanup(); return rc; }
            cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) { rc = fail(c0, -100, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); cleanup(); return rc; }
        }
        CUM(c, cudaMalloc((void**)&pc.theta[g], (size_t)W * nvs * sizeof(double)));
        CUM(c, cudaMalloc((void**)&pc.lnp[g], (size_t)W * sizeof(double)));
        CUM(c, cudaMalloc((void**)&d_nacc[g], (size_t)2 * n_loc * sizeof(unsigned long long)));
        CUM(c, cudaEventCreateWithFlags(&ev[g][0], cudaEventDisableTiming));
        CUM(c, cudaEventCreateWithFlags(&ev[g][1], cudaEventDisableTiming));
        CUM(c, cudaMemcpyAsync(pc.theta[g], theta, (size_t)W * nv * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        CUM(c, cudaMemsetAsync(d_nacc[g], 0, (size_t)2 * n_loc * sizeof(unsigned long long), c->stream));
        if (int r2 = ensure(c, &c->d_prop, &c->cap_prop, (size_t)n_loc * nvs)) { cleanup(); return r2; }
        if (int r2 = ensure(c, &c->d_plogp, &c->cap_plogp, (size_t)n_loc)) { cleanup(); return r2; }
        if (int r2 = ensure(c, &c->d_pstatus, &c->cap_pstatus, (size_t)W)) { cleanup(); return r2; }
        if (int r2 = ensure(c, &c->d_zz, &c->cap_zz, (size_t)n_loc)) { cleanup(); return r2; }
    }
    if (rows) {
        CUM(c0, cudaSetDevice(c0->device));
        CUM(c0, cudaMalloc((void**)&d_chain, (size_t)rows * W * nvs * sizeof(double)));
        CUM(c0, cudaMalloc((void**)&d_chainlp, (size_t)rows * W * sizeof(double)));
    }
    // lnprob0: every GPU evaluates the whole ensemble copy it holds?  No -- its own two slices, then the slices are exchanged
    // by plain peer copies (once); with have_lnp the caller's values are uploaded to every copy.
    for (int g = 0; g < G; g++) {
        rv_ctx* c = ctxs[g];
        CUM(c, cudaSetDevice(c->device));
        if (have_lnp) {
            CUM(c, cudaMemcpyAsync(pc.lnp[g], lnp, (size_t)W * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        } else {
            for (int half = 0; half < 2; half++) {
                const int64_t lo = half * h + g * n_loc;
                if (int r2 = loglik_dev_impl(c, models[g], obss[g], pc.theta[g] + (size_t)lo * nv, n_loc, pc.lnp[g] + lo,
                                             c->d_pstatus + lo, c->stream)) { cleanup(); return r2; }
                CUM(c, rv::launch_mask_logp(pc.lnp[g] + lo, c->d_pstatus + lo, n_loc, c->stream));
            }
        }
    }
    if (!have_lnp) {
        for (int g = 0; g < G; g++) { CUM(ctxs[g], cudaSetDevice(ctxs[g]->device)); CUM(ctxs[g], cudaStreamSynchronize(ctxs[g]->stream)); }
        for (int g = 0; g < G; g++)
            for (int q = 0; q < G; q++) {
                if (q == g) continue;
                for (int half = 0; half < 2; half++) {
                    const int64_t lo = half * h + g * n_loc;
                    CUM(ctxs[g], cudaMemcpyPeerAsync(pc.lnp[q] + lo, ctxs[q]->device, pc.lnp[g] + lo, ctxs[g]->device,
                                                     (size_t)n_loc * sizeof(double), ctxs[g]->stream));
                }
            }
    }
    for (int g = 0; g < G; g++) { CUM(ctxs[g], cudaSetDevice(ctxs[g]->device)); CUM(ctxs[g], cudaStreamSynchronize(ctxs[g]->stream)); }
    // the sampling loop: asynchronous on G streams, ordered across devices by events
    long long row = 0;
    int phase = 0;
    bool have_prev = false;
    for (int k = 0; k < nsteps; k++) {
        const unsigned step = first_step + (unsigned)k;
        for (unsigned half = 0; half < 2; half++, phase ^= 1) {
            for (int g = 0; g < G; g++) {
                rv_ctx* c = ctxs[g];
                CUM(c, cudaSetDevice(c->device));
                if (have_prev)
                    for (int q = 0; q < G; q++)
                        if (q != g) CUM(c, cudaStreamWaitEvent(c->stream, ev[q][phase ^ 1], 0));
                const int64_t lo = (int64_t)half * h + g * n_loc;
                const double* C = pc.theta[g] + (half == 0 ? (size_t)h * nv : 0);
                CUM(c, rv::launch_stretch_propose(pc.theta[g] + (size_t)lo * nv, C, nv, n_loc, h, a, seed, (uint64_t)lo, step, half,
                                                  c->d_prop, c->d_zz, c->stream));
                if (int r2 = loglik_dev_impl(c, models[g], obss[g], c->d_prop, n_loc, c->d_plogp, c->d_pstatus, c->stream)) { cleanup(); return r2; }
                CUM(c, rv::launch_stretch_accept_peer(pc, g, lo, c->d_prop, c->d_plogp, c->d_pstatus, c->d_zz, nv, n_loc, seed,
                                                      (uint64_t)lo, step, half, d_nacc[g] + half * n_loc, c->stream));
                CUM(c, cudaEventRecord(ev[g][phase], c->stream));
            }
            have_prev = true;
        }
        if (rows && ((k + 1) % thin == 0)) {
            // GPU 0's copy is complete once every GPU has finished this step's second half-step
            CUM(c0, cudaSetDevice(c0->device));
            for (int q = 1; q < G; q++) CUM(c0, cudaStreamWaitEvent(c0->stream, ev[q][phase ^ 1], 0));
            CUM(c0, cudaMemcpyAsync(d_chain + (size_t)row * W * nv, pc.theta[0], (size_t)W * nv * sizeof(double), cudaMemcpyDeviceToDevice, c0->stream));
            CUM(c0, cudaMemcpyAsync(d_chainlp + (size_t)row * W, pc.lnp[0], (size_t)W * sizeof(double), cudaMemcpyDeviceToDevice, c0->stream));
            // the other GPUs must not overwrite GPU 0's copy before the snapshot is taken: they wait on this event next
            CUM(c0, cudaEventRecord(ev[0][phase ^ 1], c0->stream));
            row++;
        }
    }
    for (int g = 0; g < G; g++) { CUM(ctxs[g], cudaSetDevice(ctxs[g]->device)); CUM(ctxs[g], cudaStreamSynchronize(ctxs[g]->stream)); }
    CUM(c0, cudaSetDevice(c0->device));
    CUM(c0, cudaMemcpyAsync(theta, pc.theta[0], (size_t)W * nv * sizeof(double), cudaMemcpyDeviceToHost, c0->stream));
    CUM(c0, cudaMemcpyAsync(lnp, pc.lnp[0], (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, c0->stream));
    if (rows) {
        CUM(c0, cudaMemcpyAsync(chain, d_chain, (size_t)rows * W * nv * sizeof(double), cudaMemcpyDeviceToHost, c0->stream));
        if (chain_lnp) CUM(c0, cudaMemcpyAsync(chain_lnp, d_chainlp, (size_t)rows * W * sizeof(double), cudaMemcpyDeviceToHost, c0->stream));
    }
    CUM(c0, cudaStreamSynchronize(c0->stream));
    if (n_accept)
        for (int g = 0; g < G; g++) {
            CUM(ctxs[g], cudaSetDevice(ctxs[g]->device));
            for (int half = 0; half < 2; half++)
                CUM(ctxs[g], cudaMemcpy(n_accept + half * h + g * n_loc, d_nacc[g] + half * n_loc, (size_t)n_loc * sizeof(uint64_t), cudaMemcpyDeviceToHost));
        }
    cleanup();
#undef CUM
    return 0;
}

// SMALA (bern_a < 0) and ALSMALA (bern_a >= 0: step i is a full SMALA step with probability exp(-bern_a*i/niter_total),
// driver.py:181, else a MALA step on the stale derivatives) share one implementation.
static int smala_impl(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, double eps,
                      double alpha, double bern_a, int64_t niter_total, uint64_t seed, uint64_t first_chain_id,
                      uint32_t first_step, int nsteps, int thin, int64_t W, double* chain, double* chain_logp,
                      uint64_t* n_accept, uint8_t* accepted, int32_t* status, uint8_t* full_step) {
    if (!ctx || !model || !obs || !theta || !logp) return fail(ctx, -1, "rv_smala_run: NULL argument");
    if (W <= 0 || nsteps < 0) return fail(ctx, -2, "rv_smala_run: bad size");
    const int nv = model->h.nvars;
    if (nv < 1) return fail(ctx, -2, "rv_smala_run: the model has no free parameter");
    if (thin < 1) thin = 1;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t nvs = (size_t)nv;
    const long long rows = chain ? nsteps / thin : 0;
    const int64_t CW = chain_width(ctx, W);
    if (int rc = ensure(ctx, &ctx->d_theta, &ctx->cap_theta, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_logp, &ctx->cap_logp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_status, &ctx->cap_status, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_grad, &ctx->cap_grad, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_hess, &ctx->cap_hess, (size_t)W * nvs * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_prop, &ctx->cap_prop, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_plogp, &ctx->cap_plogp, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pstatus, &ctx->cap_pstatus, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_pgrad, &ctx->cap_pgrad, (size_t)W * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_phess, &ctx->cap_phess, (size_t)W * nvs * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_qf, &ctx->cap_qf, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_lascr, &ctx->cap_lascr, (size_t)W * 5 * nvs * nvs)) return rc;
    if (int rc = ensure(ctx, &ctx->d_geo, &ctx->cap_geo, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_flag, &ctx->cap_flag, (size_t)W)) return rc;
    if (int rc = ensure(ctx, &ctx->d_nacc, &ctx->cap_nacc, (size_t)W)) return rc;
    if (rows) {
        if (int rc = ensure(ctx, &ctx->d_chain, &ctx->cap_chain, (size_t)rows * CW * nvs)) return rc;
        if (int rc = ensure(ctx, &ctx->d_chainlp, &ctx->cap_chainlp, (size_t)rows * CW)) return rc;
    }
    if (accepted) if (int rc = ensure(ctx, &ctx->d_acc, &ctx->cap_acc, (size_t)nsteps * W + 1)) return rc;
    CU(ctx, cudaMemcpyAsync(ctx->d_theta, theta, (size_t)W * nv * sizeof(double), cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemsetAsync(ctx->d_nacc, 0, (size_t)W * sizeof(unsigned long long), s));
    // state.get_logp_d_dd at the start state (mcmc.py:145)
    if (int rc = var_dev_impl(ctx, model, obs, ctx->d_theta, W, ctx->d_logp, ctx->d_grad, ctx->d_hess, ctx->d_status, 1, s)) return rc;
    CU(ctx, cudaMemcpyAsync(ctx->d_flag, ctx->d_status, (size_t)W * sizeof(int), cudaMemcpyDeviceToDevice, s));
    long long row = 0;
    for (int k = 0; k < nsteps; k++) {
        const unsigned step = first_step + (unsigned)k;
        CU(ctx, rv::launch_smala_propose(ctx->d_theta, ctx->d_grad, ctx->d_hess, ctx->d_status, nv, W, eps, alpha, seed,
                                         first_chain_id, step, ctx->d_prop, ctx->d_qf, ctx->d_geo, ctx->d_lascr, s));
        bool mala = false;
        if (bern_a >= 0.0) {       // one schedule draw per iteration, shared by all chains (driver.py:181)
            const rv::U4 r = rv::philox4x32_10(seed, ~0ull, step, rv::RNG_SCHEDULE);
            const double total = niter_total > 0 ? (double)niter_total : (double)nsteps;
            mala = !(exp(-bern_a * (double)step / total) > rv::u53(r.x, r.y));
        }
        if (full_step) full_step[k] = mala ? 0 : 1;
        if (mala) {
            if (int rc = loglik_dev_impl(ctx, model, obs, ctx->d_prop, W, ctx->d_plogp, ctx->d_pstatus, s)) return rc;
        } else {
            if (int rc = var_dev_impl(ctx, model, obs, ctx->d_prop, W, ctx->d_plogp, ctx->d_pgrad, ctx->d_phess, ctx->d_pstatus, 1, s)) return rc;
        }
        const bool rec = rows && ((k + 1) % thin == 0);
        CU(ctx, rv::launch_smala_accept(ctx->d_theta, ctx->d_logp, ctx->d_grad, ctx->d_hess, ctx->d_prop, ctx->d_plogp,
                                        ctx->d_pgrad, ctx->d_phess, ctx->d_pstatus, ctx->d_geo, ctx->d_qf, nv, W, eps, alpha,
                                        seed, first_chain_id, step, ctx->d_nacc, accepted ? ctx->d_acc + (size_t)k * W : nullptr,
                                        ctx->d_flag, rec ? ctx->d_chain + (size_t)row * CW * nv : nullptr,
                                        rec ? ctx->d_chainlp + (size_t)row * CW : nullptr, CW, ctx->d_lascr, mala ? 1 : 0, s));
        if (rec) row++;
    }
    CU(ctx, cudaMemcpyAsync(theta, ctx->d_theta, (size_t)W * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(logp, ctx->d_logp, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (rows) {
        CU(ctx, cudaMemcpyAsync(chain, ctx->d_chain, (size_t)rows * CW * nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (chain_logp) CU(ctx, cudaMemcpyAsync(chain_logp, ctx->d_chainlp, (size_t)rows * CW * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    if (n_accept) CU(ctx, cudaMemcpyAsync(n_accept, ctx->d_nacc, (size_t)W * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (accepted) CU(ctx, cudaMemcpyAsync(accepted, ctx->d_acc, (size_t)nsteps * W, cudaMemcpyDeviceToHost, s));
    if (status) CU(ctx, cudaMemcpyAsync(status, ctx->d_flag, (size_t)W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return 0;
}

int rv_smala_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, double eps,
                 double alpha, uint64_t seed, uint64_t first_chain_id, uint32_t first_step, int nsteps, int thin, int64_t W,
                 double* chain, double* chain_logp, uint64_t* n_accept, uint8_t* accepted, int32_t* status) {
    return smala_impl(ctx, model, obs, theta, logp, eps, alpha, -1.0, 0, seed, first_chain_id, first_step, nsteps, thin, W,
                      chain, chain_logp, n_accept, accepted, status, nullptr);
}

int rv_alsmala_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, double eps,
                   double alpha, double bern_a, int64_t niter_total, uint64_t seed, uint64_t first_chain_id,
                   uint32_t first_step, int nsteps, int thin, int64_t W, double* chain, double* chain_logp,
                   uint64_t* n_accept, uint8_t* accepted, int32_t* status, uint8_t* full_step) {
    if (bern_a < 0.0) return fail(ctx, -2, "rv_alsmala_run: bern_a must be >= 0");
    return smala_impl(ctx, model, obs, theta, logp, eps, alpha, bern_a, niter_total, seed, first_chain_id, first_step, nsteps,
                      thin, W, chain, chain_logp, n_accept, accepted, status, full_step);
}

int rv_dev_alloc(rv_ctx* ctx, int64_t nbytes, void** out) {
    if (!ctx || !out || nbytes < 0) return fail(ctx, -1, "rv_dev_alloc: bad argument");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMalloc(out, (size_t)(nbytes > 0 ? nbytes : 1)));
    return 0;
}

int rv_dev_free(rv_ctx* ctx, void* p) {
    if (!ctx) return -1;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaFree(p));
    return 0;
}

int rv_dev_upload(rv_ctx* ctx, void* dst_dev, const void* src_host, int64_t nbytes) {
    if (!ctx || (nbytes > 0 && (!dst_dev || !src_host))) return fail(ctx, -1, "rv_dev_upload: bad argument");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst_dev, src_host, (size_t)nbytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rv_dev_download(rv_ctx* ctx, void* dst_host, const void* src_dev, int64_t nbytes) {
    if (!ctx || (nbytes > 0 && (!dst_host || !src_dev))) return fail(ctx, -1, "rv_dev_download: bad argument");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst_host, src_dev, (size_t)nbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rv_dev_copy_peer(rv_ctx* dst_ctx, void* dst_dev, rv_ctx* src_ctx, const void* src_dev, int64_t nbytes) {
    if (!dst_ctx || !src_ctx || (nbytes > 0 && (!dst_dev || !src_dev))) return fail(src_ctx, -1, "rv_dev_copy_peer: bad argument");
    CU(src_ctx, cudaSetDevice(src_ctx->device));
    CU(src_ctx, cudaMemcpyPeerAsync(dst_dev, dst_ctx->device, src_dev, src_ctx->device, (size_t)nbytes, src_ctx->stream));
    CU(src_ctx, cudaStreamSynchronize(src_ctx->stream));
    return 0;
}

int rv_count_work(rv_ctx* ctx, int enable) {
    if (!ctx) return -1;
    ctx->count_work = enable ? 1 : 0;
    return 0;
}

int rv_work_counters(rv_ctx* ctx, uint64_t out[2], int reset) {
    if (!ctx) return -1;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    CU(ctx, cudaDeviceSynchronize());
    unsigned long long h[2];
    CU(ctx, cudaMemcpy(h, ctx->d_work, sizeof h, cudaMemcpyDeviceToHost));
    if (out) { out[0] = h[0]; out[1] = h[1]; }
    if (reset) CU(ctx, cudaMemset(ctx->d_work, 0, sizeof h));
    return 0;
}

int rv_fp64_peak(rv_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return -1;
    CU(ctx, cudaSetDevice(ctx->device));
    double* d = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto drop = [&]() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); cudaFree(d); };
    CU_OR(ctx, cudaMalloc((void**)&d, 64), drop());
    CU_OR(ctx, cudaEventCreate(&e0), drop());
    CU_OR(ctx, cudaEventCreate(&e1), drop());
    const int blocks = ctx->num_sms * 8, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        CU_OR(ctx, cudaEventRecord(e0, ctx->stream), drop());
        CU_OR(ctx, rv::launch_fp64_peak(d, blocks, iters, ctx->stream), drop());
        CU_OR(ctx, cudaEventRecord(e1, ctx->stream), drop());
        CU_OR(ctx, cudaEventSynchronize(e1), drop());
        float ms = 0;
        CU_OR(ctx, cudaEventElapsedTime(&ms, e0, e1), drop());
        const double flops = 2.0 * 64.0 * (double)iters * 256.0 * (double)blocks;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    drop();
    *tflops = best;
    return 0;
}

void* rv_ctx_stream(rv_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int rv_sync(rv_ctx* ctx) {
    if (!ctx) return -1;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // extern "C"
