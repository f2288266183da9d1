// rv_kernels.cu -- sm_100a kernels for the batched RV log-likelihood (plain path: MH / affine sampler).
//
// loglik_kernel: persistent grid (resident CTAs x SM count); every lane group pulls (walker, leg)
// items from a global counter and runs the IAS15 state machine of rv_loglik.cuh.  Observation epochs,
// velocities and errors are staged once per CTA into shared memory; the once-per-step coefficients (e, and the
// rejected-step history br/er) and the state the predictor-corrector loop never reads (x0 and the compensated-summation
// carries) live in shared memory, strided per lane; x0 - csx, v0, a0/2 and the seven g coefficients per coordinate are in
// registers.
#include <cuda_runtime.h>
#include <stdio.h>
#include "rv_launch.h"
#include "rv_loglik.cuh"
#include "rv_core_g.cuh"

namespace rv {

struct DevFetch {
    unsigned long long* ctr;
    template <class G>
    __device__ __forceinline__ long long operator()(const G& g) const {
        unsigned long long v = 0;
        if (g.rank == 0) v = atomicAdd(ctr, 1ull);
        if (G::lanes > 1) v = __shfl_sync(g.mask, v, g.base);
        return (long long)v;
    }
};
struct DevAll {
    __device__ __forceinline__ bool operator()(bool f) const { return __all_sync(0xffffffffu, f) != 0; }
};

template <int P, int D, int PL, int NT, int MINB, int VAR>
__global__ void __launch_bounds__(NT, MINB) loglik_kernel(const LoglikArgs a) {
    extern __shared__ double sm[];
    const int nobs = a.nf + a.nb;
    // observation epochs / velocities / errors: staged in shared memory when that does not cost occupancy
    // (launch_one decides), else read from global memory (one read per epoch reached, L1/L2-resident)
    const double *st = a.ot, *srv = a.orv, *serr = a.oerr;
    double* hist = sm;
    if (a.stage_obs) {
        double* so = sm;
        for (int i = threadIdx.x; i < nobs; i += NT) {
            so[i] = a.ot[i];
            so[nobs + i] = a.orv[i];
            so[2 * nobs + i] = a.oerr[i];
        }
        st = so; srv = so + nobs; serr = so + 2 * nobs;
        hist = sm + 3 * nobs;
        __syncthreads();
    }
    using W = WalkerG<P, D, PL, VAR>;
    W w;
    const int lane = threadIdx.x & 31;
    w.grp.init(lane);
    w.hist.p = hist + threadIdx.x;
    w.hist.stride = NT;
    const bool lane_active = (w.grp.base + W::G) <= 32;
    DevFetch fetch{a.item_counter};
    DevAll all;
    run_items(w, a, st, srv, serr, fetch, all, lane_active);
}

__global__ void finalize_kernel(const double* __restrict__ part_chi2, const int* __restrict__ part_status,
                                long long W, double npoints, double* __restrict__ logp,
                                int* __restrict__ status, unsigned long long* item_counter) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) *item_counter = 0ull;
    if (w >= W) return;
    const int sb = part_status[w], sf = part_status[W + w];
    const int s = (sf != ST_OK) ? sf : sb;   // the reference integrates the forward leg first
    status[w] = s;
    // state.py:98: (chi2b + chi2f) / Npoints ; state.py:109: logp = -chi2
    logp[w] = (s == ST_OK) ? -((part_chi2[w] + part_chi2[W + w]) / npoints) : -INFINITY;
}

__global__ void curve_finalize_kernel(unsigned long long* item_counter) { *item_counter = 0ull; }

template <int P, int D, int PL, int NT, int MINB, int VAR = 0>
static cudaError_t launch_one(const LoglikArgs& a, int num_sms, cudaStream_t stream) {
    auto kern = loglik_kernel<P, D, PL, NT, MINB, VAR>;
    const int nobs = a.nf + a.nb;
    constexpr int NC = PL * D;
    constexpr int LANE_DOUBLES = WalkerG<P, D, PL, VAR>::LANE_DOUBLES;
    const size_t smem_hist = sizeof(double) * (size_t)LANE_DOUBLES * NT;
    const size_t smem_obs = sizeof(double) * (size_t)3 * nobs;
    LoglikArgs args = a;
    // stage the observations only while MINB CTAs still fit in the SM's 227 KB of shared memory.  Per lane (Walker::SLOT_*):
    // e / er / br (21 NC doubles), x0, csx, csv (3 NC), t, dt_last_done, tmax, last_full_dt (4); + 9 per own planet in the
    // dense-output instantiation.  The headline shape (P = 2, D = 2, one lane per planet: NC = 2) at 4 CTAs x 128 threads:
    // 52 doubles x 8 B x 128 = 53 248 B, + 2 928 B of HD155358's 122 epochs + 1 KB reserved = 57 200 B per CTA,
    // x 4 = 228 800 B <= 232 448 B (one double more per lane would stop the staging).
    args.stage_obs = ((smem_hist + smem_obs + 1024) * MINB <= (size_t)227 * 1024) ? 1 : 0;
    const size_t smem = smem_hist + (args.stage_obs ? smem_obs : 0);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorLaunchOutOfResources;
    constexpr int G = P / PL;
    const long long groups_per_block = (long long)(NT / 32) * (32 / G);
    const long long n_items = a.times ? a.W : 2 * a.W;
    long long blocks = (long long)num_sms * occ;
    const long long need = (n_items + groups_per_block - 1) / groups_per_block;
    if (need < blocks) blocks = need;
    if (blocks < 1) blocks = 1;
    kern<<<(unsigned)blocks, NT, smem, stream>>>(args);
    return cudaGetLastError();
}

// mapping: 0 = one lane per planet (default), 1 = one thread per walker; dense: the dense-output instantiations
template <int VAR>
static cudaError_t launch_loglik_var(const LoglikArgs& a, int P, int D, int mapping, int num_sms, cudaStream_t stream) {
    const int key = P * 100 + D * 10 + mapping;
    switch (key) {
        case 120: case 121: return launch_one<1, 2, 1, 128, 3, VAR>(a, num_sms, stream);
        case 130: case 131: return launch_one<1, 3, 1, 128, 2, VAR>(a, num_sms, stream);
        case 220:
            // the headline shape: 4 CTAs x 128 threads at <= 128 registers without spills, +7 % over 3 CTAs on B200 (mapping 11)
            if constexpr (VAR == 0) return launch_one<2, 2, 1, 128, 4, VAR>(a, num_sms, stream);
            else return launch_one<2, 2, 1, 128, 3, VAR>(a, num_sms, stream);
        case 221: return launch_one<2, 2, 2, 128, 2, VAR>(a, num_sms, stream);
        case 230: return launch_one<2, 3, 1, 128, 2, VAR>(a, num_sms, stream);
        case 231: return launch_one<2, 3, 1, 128, 2, VAR>(a, num_sms, stream);
        case 320: case 321: return launch_one<3, 2, 1, 128, 3, VAR>(a, num_sms, stream);
        case 330: case 331: return launch_one<3, 3, 1, 128, 2, VAR>(a, num_sms, stream);
        // four and five planets: lane per planet only (8 / 6 walkers per warp)
        case 420: case 421: return launch_one<4, 2, 1, 128, 2, VAR>(a, num_sms, stream);
        case 430: case 431: return launch_one<4, 3, 1, 128, 2, VAR>(a, num_sms, stream);
        case 520: case 521: return launch_one<5, 2, 1, 128, 2, VAR>(a, num_sms, stream);
        case 530: case 531: return launch_one<5, 3, 1, 128, 2, VAR>(a, num_sms, stream);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_loglik(const LoglikArgs& a, int P, int D, int mapping, int dense, int num_sms, cudaStream_t stream) {
    // tuning variants of the headline instantiation (tools/bench_variants.py): model option "mapping" >= 10
    if (mapping >= 10) {
        // the variants exist for the headline instantiation only; every other shape and the dense-output mode run the
        // default mapping (mapping + 10 would otherwise select another shape's kernel in launch_loglik_var)
        if (!(P == 2 && D == 2 && !dense)) return launch_loglik(a, P, D, 0, dense, num_sms, stream);
        switch (mapping) {
            case 10: return launch_one<2, 2, 1, 128, 3, 2>(a, num_sms, stream);     // IAS15 tables from the constant bank
            case 11: return launch_one<2, 2, 1, 128, 3, 0>(a, num_sms, stream);     // 3 CTAs per SM (the default up to round 2)
            case 12: return launch_one<2, 2, 1, 128, 4, 2>(a, num_sms, stream);
            case 13: return launch_one<2, 2, 1, 256, 2, 0>(a, num_sms, stream);     // 2 CTAs x 256 threads (<= 128 registers)
            default: return cudaErrorInvalidValue;
        }
    }
    if (dense && !a.times) return launch_loglik_var<4>(a, P, D, mapping, num_sms, stream);
    return launch_loglik_var<0>(a, P, D, mapping, num_sms, stream);
}

cudaError_t launch_finalize(const double* part_chi2, const int* part_status, long long W, double npoints,
                            double* logp, int* status, unsigned long long* item_counter, cudaStream_t stream) {
    const int nt = 256;
    const unsigned nb = (unsigned)((W + nt - 1) / nt);
    finalize_kernel<<<nb ? nb : 1, nt, 0, stream>>>(part_chi2, part_status, W, npoints, logp, status, item_counter);
    return cudaGetLastError();
}

cudaError_t launch_curve_finalize(unsigned long long* item_counter, cudaStream_t stream) {
    curve_finalize_kernel<<<1, 1, 0, stream>>>(item_counter);
    return cudaGetLastError();
}

// ---- cost-ordered scheduling ---------------------------------------------------------------------------------------
// The number of IAS15 steps of a walker is set by its fastest pericentre passage: max_p a_p^-3/2 (1 - e_p)^-3/2 tracks the
// measured step count of posterior walkers with rank correlation 0.95 (HD155358 ensemble).  Walkers are binned by that key
// (1/32 octave), most expensive first, and the likelihood kernel takes its items in that order: the lane groups of a warp
// then integrate walkers of similar cost and stay in step (a warp runs every predictor-corrector loop for the slowest of its
// groups: lane efficiency 0.77 -> 0.88 on the equilibrated ensemble), and the launch ends on its cheapest items.  A counting
// sort in three small kernels; the order inside a bin is whatever the atomics give -- it affects scheduling only, results are
// stored by walker.
constexpr int COST_BINS = RV_COST_BINS;

__global__ void cost_bin_kernel(const Model* __restrict__ md, const double* __restrict__ theta, long long W,
                                int* __restrict__ bin, int* __restrict__ hist) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const int P = md->P, nv = md->nvars;
    float key = 0.0f;
    bool bad = false;
    for (int i = 0; i < P; i++) {
        float el[3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const int e = EL_A + k;                        // a, h, k
            const int sidx = md->src[i * NELEM + e];
            el[k] = (float)((sidx >= 0) ? theta[w * nv + sidx] : md->fixed[i * NELEM + e]);
        }
        const float e2 = el[1] * el[1] + el[2] * el[2];
        if (!(el[0] > 0.02f) || !(e2 < 1.0f)) bad = true;  // hard prior: the item returns at once
        const float q = el[0] * (1.0f - sqrtf(fminf(e2, 0.9801f)));          // pericentre distance
        const float c = rsqrtf(q) / q;                     // q^-3/2
        key = fmaxf(key, c);
    }
    int b = COST_BINS - 1;                                 // cheapest bin: prior violations, non-finite keys
    if (!bad && key > 0.0f && key < 3.0e38f) {
        const float l = (log2f(key) + 12.0f) * 32.0f;      // 2^-12 .. 2^20 in 1/32 octaves
        const int i = l < 0.0f ? 0 : (l > (float)(COST_BINS - 2) ? COST_BINS - 2 : (int)l);
        b = COST_BINS - 2 - i;                             // most expensive first
    }
    bin[w] = b;
    // one atomic per distinct bin of the warp (a start ball puts every walker into the same two or three bins)
    const unsigned peers = __match_any_sync(__activemask(), b);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[b], __popc(peers));
}

// exclusive prefix sum of the histogram -> per-bin cursors; clears the histogram for the next call
__global__ void __launch_bounds__(COST_BINS) cost_scan_kernel(int* __restrict__ hist, int* __restrict__ cursor) {
    __shared__ int sh[COST_BINS];
    const int t = threadIdx.x;
    const int v = hist[t];
    sh[t] = v;
    __syncthreads();
    for (int o = 1; o < COST_BINS; o <<= 1) {
        const int x = t >= o ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += x;
        __syncthreads();
    }
    cursor[t] = sh[t] - v;
    hist[t] = 0;
}

__global__ void cost_scatter_kernel(const int* __restrict__ bin, long long W, int* __restrict__ cursor, int* __restrict__ order) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const int b = bin[w];
    const unsigned peers = __match_any_sync(__activemask(), b);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(&cursor[b], __popc(peers));
    base = __shfl_sync(peers, base, leader);
    order[base + __popc(peers & ((1u << lane) - 1u))] = (int)w;
}

// order[W] from theta; bin[W], hist[COST_BINS] (zero on entry, zero on exit), cursor[COST_BINS]: scratch
cudaError_t launch_cost_order(const Model* md, const double* theta, long long W, int* bin, int* hist, int* cursor, int* order,
                              cudaStream_t stream) {
    const int nt = 256;
    const unsigned nb = (unsigned)((W + nt - 1) / nt);
    cost_bin_kernel<<<nb, nt, 0, stream>>>(md, theta, W, bin, hist);
    cost_scan_kernel<<<1, COST_BINS, 0, stream>>>(hist, cursor);
    cost_scatter_kernel<<<nb, nt, 0, stream>>>(bin, W, cursor, order);
    return cudaGetLastError();
}

// ---- State.setup_sim (state.py:36-47) made visible: barycentric particles [W][P+1][7] = m, x, y, z, vx, vy, vz ----
// One thread per walker; the same Pal -> cartesian and move_to_com arithmetic the integrating kernels start from.
__global__ void initial_conditions_kernel(const Model* __restrict__ md, const double* __restrict__ theta, long long W,
                                          double* __restrict__ out, int* __restrict__ status) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const int P = md->P;
    const double m0 = md->m_star;
    double xr[MAXP][3], vr[MAXP][3], mp[MAXP];
    double cx[3] = {0, 0, 0}, cv[3] = {0, 0, 0}, mtot = m0;
    bool bad = false;
    for (int i = 0; i < P; i++) {
        double el[NELEM];
        for (int k = 0; k < NELEM; k++) {
            const int s = md->src[i * NELEM + k];
            el[k] = (s >= 0) ? theta[w * md->nvars + s] : md->fixed[i * NELEM + k];
        }
        bad = bad || prior_hard(el);
        pal_to_cart(el, m0, xr[i], vr[i]);
        mp[i] = el[EL_M];
        mtot += mp[i];
        for (int d = 0; d < 3; d++) { cx[d] += mp[i] * xr[i][d]; cv[d] += mp[i] * vr[i][d]; }
    }
    double* o = out + w * (P + 1) * 7;
    o[0] = m0;
    for (int d = 0; d < 3; d++) { o[1 + d] = -cx[d] / mtot; o[4 + d] = -cv[d] / mtot; }
    for (int i = 0; i < P; i++) {
        double* q = o + (i + 1) * 7;
        q[0] = mp[i];
        for (int d = 0; d < 3; d++) { q[1 + d] = xr[i][d] - cx[d] / mtot; q[4 + d] = vr[i][d] - cv[d] / mtot; }
    }
    status[w] = bad ? ST_PRIOR : ST_OK;
}

cudaError_t launch_initial_conditions(const Model* md, const double* theta, long long W, double* out, int* status,
                                      cudaStream_t stream) {
    const int nt = 128;
    initial_conditions_kernel<<<(unsigned)((W + nt - 1) / nt), nt, 0, stream>>>(md, theta, W, out, status);
    return cudaGetLastError();
}

// ---- FP64 FMA-pipe peak microbenchmark (roofline denominator; MEASURED_PEAKS.json has no FP64 entry) ----
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) out[0] = s;  // keep the chain alive
}

cudaError_t launch_fp64_peak(double* d_out, int blocks, int iters, cudaStream_t stream) {
    fp64_peak_kernel<<<blocks, 256, 0, stream>>>(d_out, iters, 1.0);
    return cudaGetLastError();
}

}  // namespace rv
