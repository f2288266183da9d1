// rv_var_kernels.cu -- sm_100a kernel for State.get_logp_d_dd (value + gradient + Hessian, SMALA).
//
// var_kernel: persistent grid; every CTA pulls (walker, leg) items and integrates the real system together
// with its first- and second-order variational sets, one thread per (set, planet) -- see rv_var.cuh.  var2_kernel: the same
// algorithm with one lane per second-order set, for one planet and two coplanar planets -- see rv_var2.cuh.
#include <cuda_runtime.h>
#include "rv_launch.h"
#include "rv_var.cuh"
#include "rv_var2.cuh"

namespace rv {

template <int P, int D>
struct DevVarExec {
    VarThread<P, D>& th;
    double* red;                 // [2][64] ping-pong maxima, then the item broadcast slot
    int parity;
    int nwarps;
    template <class F>
    __device__ __forceinline__ void each(F&& f) { f(th); }
    __device__ __forceinline__ void sync() { __syncthreads(); }
    __device__ __forceinline__ void stage_max(const VarThread<P, D>&, double a, double b) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a = fmax(a, __shfl_xor_sync(0xffffffffu, a, o));
            b = fmax(b, __shfl_xor_sync(0xffffffffu, b, o));
        }
        if ((threadIdx.x & 31) == 0) {
            red[parity * 64 + 2 * (threadIdx.x >> 5)] = a;
            red[parity * 64 + 2 * (threadIdx.x >> 5) + 1] = b;
        }
    }
    __device__ __forceinline__ void read_max(double& a, double& b) {
        a = 0.0; b = 0.0;
        for (int w = 0; w < nwarps; w++) {
            a = fmax(a, red[parity * 64 + 2 * w]);
            b = fmax(b, red[parity * 64 + 2 * w + 1]);
        }
        parity ^= 1;
    }
    __device__ __forceinline__ long long fetch(unsigned long long* ctr) {
        unsigned long long* slot = reinterpret_cast<unsigned long long*>(red + 128);
        __syncthreads();
        if (threadIdx.x == 0) *slot = atomicAdd(ctr, 1ull);
        __syncthreads();
        return (long long)*slot;
    }
    __device__ __forceinline__ void add_work(unsigned long long* wc, unsigned long long nf, unsigned long long na) {
        if (wc && threadIdx.x == 0) { atomicAdd(&wc[0], nf); atomicAdd(&wc[1], na); }
    }
};

template <int P, int D, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) var_kernel(const VarArgs a, const VarLayout L) {
    extern __shared__ __align__(16) double sm[];
    VarThread<P, D> th;
    var_assign(th, (int)threadIdx.x, L);
    DevVarExec<P, D> ex{th, sm + L.o_red, 0, NT / 32};
    var_run_items<P, D>(ex, a, L, sm);
}

// ---- "warp group per walker leg" layout (rv_var2.cuh): several independent groups per CTA, producer warp + mbarriers ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

template <int P, int D>
struct DevVar2Exec {
    Var2Thread<P, D>& th;
    double* red;                 // [2][16] ping-pong group maxima, then the item broadcast slot
    unsigned mbar;               // shared address of the group's seven substep mbarriers
    int parity, nwarps, nt, bar_id;
    unsigned round;              // predictor-corrector iterations so far: every substep mbarrier completes once per iteration
    bool producer;               // this thread's warp is the group's producer warp (real + first-order sets)
    template <class F>
    __device__ __forceinline__ void each(F&& f) { f(th); }
    // group barrier: one named barrier per group (id 0 stays free for __syncthreads)
    __device__ __forceinline__ void sync() { asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nt) : "memory"); }
    __device__ __forceinline__ void producer_sync() { if (producer) __syncwarp(); }
    __device__ __forceinline__ void signal(int n) {
        if (producer) {
            asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(mbar + 8u * (unsigned)(n - 1)) : "memory");
            if (n == 7) round++;
        }
    }
    __device__ __forceinline__ void wait(int n) {
        if (!producer) {
            const unsigned addr = mbar + 8u * (unsigned)(n - 1), ph = round & 1u;
            unsigned done = 0;
            for (unsigned spin = 0; !done; spin++) {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(done) : "r"(addr), "r"(ph) : "memory");
                if (spin > (1u << 26)) __trap();          // a lost signal must fail loudly, never hang the GPU
            }
            if (n == 7) round++;
        }
    }
    __device__ __forceinline__ void stage_max(const Var2Thread<P, D>&, double a, double b) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a = fmax(a, __shfl_xor_sync(0xffffffffu, a, o));
            b = fmax(b, __shfl_xor_sync(0xffffffffu, b, o));
        }
        if ((th.tid & 31) == 0) {
            red[parity * 16 + 2 * (th.tid >> 5)] = a;
            red[parity * 16 + 2 * (th.tid >> 5) + 1] = b;
        }
    }
    __device__ __forceinline__ void read_max(double& a, double& b) {
        a = 0.0; b = 0.0;
        for (int w = 0; w < nwarps; w++) {
            a = fmax(a, red[parity * 16 + 2 * w]);
            b = fmax(b, red[parity * 16 + 2 * w + 1]);
        }
        parity ^= 1;
    }
    __device__ __forceinline__ long long fetch(unsigned long long* ctr) {
        unsigned long long* slot = reinterpret_cast<unsigned long long*>(red + 32);
        sync();
        if (th.tid == 0) *slot = atomicAdd(ctr, 1ull);
        sync();
        return (long long)*slot;
    }
    __device__ __forceinline__ void add_work(unsigned long long* wc, unsigned long long nf, unsigned long long na) {
        if (wc && th.tid == 0) { atomicAdd(&wc[0], nf); atomicAdd(&wc[1], na); }
    }
};

// NTG threads per group, G groups per CTA; MAXR: register cap per thread (__maxnreg__: the register file is allocated per
// CTA in 128-thread units, so G * NTG should be a multiple of 128 and MAXR <= 65536 / (CTA threads x CTAs per SM))
template <int P, int D, int NTG, int G, int MAXR>
__global__ void __maxnreg__(MAXR) var2_kernel(const VarArgs a, const Var2Layout L) {
    extern __shared__ __align__(16) double sm_all[];
    const int group = (int)threadIdx.x / NTG, gtid = (int)threadIdx.x - group * NTG;
    double* sm = sm_all + (size_t)group * L.total;
    Var2Thread<P, D> th;
    var2_assign(th, gtid, L);
    unsigned long long* mb = reinterpret_cast<unsigned long long*>(sm + L.o_mbar);
    if (gtid == 0) {
#pragma unroll
        for (int k = 0; k < 7; k++)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 32;" ::"r"(smem_u32(mb + k)) : "memory");
    }
    __syncthreads();
    DevVar2Exec<P, D> ex{th, sm + L.o_red, smem_u32(mb), 0, NTG / 32, NTG, 1 + group, 0u, (gtid >> 5) == L.nso_warps};
    double* hist = a.hist + ((size_t)blockIdx.x * G + group) * var2_hist_doubles(P, D, L.nv);
    var2_run_items<P, D>(ex, a, L, sm, hist);
}

template <int P, int D, int NTG, int G, int MAXR>
static cudaError_t launch_var2_one(const VarArgs& a, int nv, int num_sms, cudaStream_t stream) {
    auto kern = var2_kernel<P, D, NTG, G, MAXR>;
    const Var2Layout L = var2_layout(P, D, nv, NTG);
    if (var2_min_threads(nv) > NTG) return cudaErrorInvalidConfiguration;
    const size_t smem = sizeof(double) * (size_t)L.total * G;
    if (smem > (size_t)227 * 1024) return cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NTG * G, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorLaunchOutOfResources;
    long long blocks = (long long)num_sms * occ;
    const long long need = (2 * a.W + G - 1) / G;
    if (need < blocks) blocks = need;
    if (blocks < 1) blocks = 1;
    if (!a.hist || a.hist_doubles < (size_t)blocks * G * var2_hist_doubles(P, D, nv)) return cudaErrorInvalidValue;
    kern<<<(unsigned)blocks, NTG * G, smem, stream>>>(a, L);
    return cudaGetLastError();
}

// groups of one CTA that fit the SM's shared memory (227 KB), at most gmax
static int var2_groups(int P, int D, int nv, int ntg, int gmax) {
    const Var2Layout L = var2_layout(P, D, nv, ntg);
    const size_t per = sizeof(double) * (size_t)L.total;
    int g = (int)(((size_t)227 * 1024) / per);
    return g < 1 ? 0 : (g > gmax ? gmax : g);
}

// logp = -(chi2b + chi2f), grad = -(db + df), hess symmetric (state.py:285,292-293)
__global__ void var_finalize_kernel(const double* __restrict__ part, const int* __restrict__ pstat, long long W, int nv,
                                    int nsets, double* __restrict__ logp, double* __restrict__ grad,
                                    double* __restrict__ hess, int* __restrict__ status,
                                    unsigned long long* item_counter) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0) *item_counter = 0ull;
    if (idx >= W * nsets) return;
    const long long w = idx / nsets;
    const int s = (int)(idx - w * nsets);
    const int sb = pstat[w], sf = pstat[W + w];
    const int st = (sf != ST_OK) ? sf : sb;
    const bool ok = st == ST_OK;
    const double v = ok ? -(part[w * nsets + s] + part[(W + w) * nsets + s]) : 0.0;
    if (s == 0) {
        status[w] = st;
        logp[w] = ok ? v : -INFINITY;
    } else if (s <= nv) {
        grad[w * nv + (s - 1)] = v;
    } else {
        const int k = s - 1 - nv;
        int a = 0;
        while ((a + 1) * (a + 2) / 2 <= k) a++;
        const int b = k - a * (a + 1) / 2;
        hess[(w * nv + a) * nv + b] = v;
        hess[(w * nv + b) * nv + a] = v;
    }
}

template <int P, int D, int NT, int MINB>
static cudaError_t launch_var_one(const VarArgs& a, int nv, int num_sms, cudaStream_t stream, int k2_lo = 0, int k2_n = -1) {
    auto kern = var_kernel<P, D, NT, MINB>;
    const VarLayout L = var_layout(P, D, nv, NT, k2_lo, k2_n);
    if (L.need > NT) return cudaErrorInvalidConfiguration;
    const size_t smem = sizeof(double) * (size_t)L.total;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorLaunchOutOfResources;
    long long blocks = (long long)num_sms * occ;
    if (2 * a.W < blocks) blocks = 2 * a.W;
    if (blocks < 1) blocks = 1;
    kern<<<(unsigned)blocks, NT, smem, stream>>>(a, L);
    return cudaGetLastError();
}

// Models whose sets do not fit one CTA: several launches, each with the real set, the first-order sets and a chunk of the
// second-order pairs (var_layout).  The work-queue counter is reset between the launches (the finalize kernel resets it
// after the last one).
template <int P, int D, int NT>
static cudaError_t launch_var_chunked(const VarArgs& a, int nv, int num_sms, cudaStream_t stream) {
    const int n2 = nv * (nv + 1) / 2, chunk = var_chunk_pairs(P, nv, NT);
    if (chunk < 1) return cudaErrorInvalidConfiguration;
    for (int lo = 0; lo < n2 || lo == 0; lo += chunk) {
        if (lo > 0) {
            cudaError_t e = cudaMemsetAsync(a.item_counter, 0, sizeof(unsigned long long), stream);
            if (e != cudaSuccess) return e;
        }
        const int n = (n2 - lo < chunk) ? n2 - lo : chunk;
        cudaError_t e = launch_var_one<P, D, NT, 1>(a, nv, num_sms, stream, lo, n);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// 1 when launch_var has a configuration for this model (one or two planets: always; more: one launch or chunks of pairs)
int var_model_fits(int P, int D, int nv) {
    if (P < 1 || P > MAXP_VAR) return 0;
    if (P <= 2) return 1;                                    // at most 14 free parameters: always one launch
    return var_chunk_pairs(P, nv, D == 3 ? 320 : 448) >= 1 || nv == 0;
}

// threads needed by a model (host-side check shared with the ABI)
int var_threads_needed(int P, int nv) {
    const VarLayout L = var_layout(P, 2, nv, 32);
    return L.need;
}

// global history scratch (doubles) the warp-group kernel needs for this model on this GPU; 0 when the other layout runs
size_t var_hist_doubles_needed(int P, int D, int nv, int num_sms) {
    if (!var2_supported(P, nv)) return 0;
    return (size_t)num_sms * 8 * var2_hist_doubles(P, D, nv);       // at most 8 resident groups per SM
}

// One planet, or two coplanar planets: the warp-group kernel (a coplanar two-planet model has at most 10 free parameters and
// a one-planet model at most 7, so 96 and 64 threads per group always suffice).  Two inclined planets and three to five
// planets: one thread per (set, planet).
cudaError_t launch_var(const VarArgs& a, int P, int D, int nv, int num_sms, cudaStream_t stream) {
    if (var2_supported(P, nv)) {
        const int nt = var2_min_threads(nv);
        if (P == 2 && D == 2 && nt <= 96) {                       // nv <= 10 (HD155358): 4 x 96 = 384 threads, 168 registers
            if (var2_groups(2, 2, nv, 96, 4) >= 4) return launch_var2_one<2, 2, 96, 4, 168>(a, nv, num_sms, stream);
        }
        if (P == 1 && D == 2 && nt <= 64) return launch_var2_one<1, 2, 64, 4, 128>(a, nv, num_sms, stream);
        if (P == 1 && D == 3 && nt <= 64) return launch_var2_one<1, 3, 64, 4, 168>(a, nv, num_sms, stream);
    }
    const int need = var_threads_needed(P, nv);
    if (P == 2 && D == 3 && need <= 256) return launch_var_one<2, 3, 256, 1>(a, nv, num_sms, stream);
    if (P == 3 && D == 2 && need <= 448) return launch_var_one<3, 2, 448, 1>(a, nv, num_sms, stream);
    // (inclined models: 320 threads -- the per-thread shared-memory history, 21 D doubles, is what fills the SM's 227 KB)
    if (P == 3 && D == 3 && need <= 320) return launch_var_one<3, 3, 320, 1>(a, nv, num_sms, stream);
    // everything else the schema allows (state.py:8-31 is open-ended): the second-order sets in chunks of what one CTA holds
    if (P == 3 && D == 2) return launch_var_chunked<3, 2, 448>(a, nv, num_sms, stream);
    if (P == 3 && D == 3) return launch_var_chunked<3, 3, 320>(a, nv, num_sms, stream);
    if (P == 4 && D == 2) return launch_var_chunked<4, 2, 448>(a, nv, num_sms, stream);
    if (P == 4 && D == 3) return launch_var_chunked<4, 3, 320>(a, nv, num_sms, stream);
    if (P == 5 && D == 2) return launch_var_chunked<5, 2, 448>(a, nv, num_sms, stream);
    if (P == 5 && D == 3) return launch_var_chunked<5, 3, 320>(a, nv, num_sms, stream);
    return cudaErrorInvalidConfiguration;
}

cudaError_t launch_var_finalize(const double* part, const int* pstat, long long W, int nv, double* logp, double* grad,
                                double* hess, int* status, unsigned long long* item_counter, cudaStream_t stream) {
    const int nsets = var_nsets(nv);
    const int nt = 256;
    const long long n = W * nsets;
    const unsigned nb = (unsigned)((n + nt - 1) / nt);
    var_finalize_kernel<<<nb ? nb : 1, nt, 0, stream>>>(part, pstat, W, nv, nsets, logp, grad, hess, status, item_counter);
    return cudaGetLastError();
}

}  // namespace rv
