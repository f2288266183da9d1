// rv_var2.cuh -- value + gradient + Hessian of the RV log-likelihood, "warp-group per walker leg" layout.
//
// Same contract as rv_var.cuh (State.get_logp_d_dd, state.py:290-294; setup_sim_vars state.py:229-248; get_chi2_d_dd
// state.py:253-285; one item = one leg of one walker, all sets share one IAS15 step sequence, real-only step-size
// norm), for systems of one or two planets.  The mapping:
//   * a GROUP of warps integrates one (walker, leg); a CTA holds several independent groups, so the register file is
//     allocated in full 128-thread units while each leg only occupies the warps it needs (96 threads for HD155358);
//   * second-order ("so") lanes own a whole variational SET -- all P planets of it: nothing is exchanged between so
//     lanes, pair terms are computed once (Newton's third law), their predicted positions never leave the registers;
//   * the real set and the nv first-order sets live in ONE producer warp, one lane per (set, planet).  They do not
//     depend on the second-order sets and carry half the work per lane, so the producer runs ahead of the so warps inside
//     a predictor-corrector iteration: per Gauss-Radau substep it publishes its predicted positions and star sums to
//     shared memory and arrives on that substep's mbarrier; the so warps wait on the mbarrier only;
//   * group-wide barriers (named barriers, one id per group) remain for the convergence monitor (once per iteration) and
//     the once-per-step bookkeeping; nothing is CTA-wide.
// Registers hold the seven g coefficients per coordinate and the predicted positions; x0, the carries, x0 - csx, v0, a0 and
// e live in shared memory (strided per planet slot); the rejected-step history br / er, written once per accepted step and
// read only after a rejection, lives in a per-group global scratch (L2-resident).  Written against an executor like rv_var.cuh, so the CPU test-suite runs the same source sequentially.
#pragma once
#include "rv_var.cuh"

namespace rv {

struct Var2Layout {
    int P, D, nv, n2, nsets;
    int nso_warps;     // warps of second-order lanes (lane t of these warps owns second-order set t)
    int NT;            // threads of one group = 32 * (nso_warps + 1); the last warp is the producer
    int nps;           // planet slots: nsets * P (so lane t, planet p -> p * n2 + t; producer lane (s, p) -> n2 * P + s * P + p)
    int CB;            // doubles per producer-set block in a buffer: P*D positions + D star sum
    int cstride;       // doubles per buffer: (nv + 1) * CB, rounded up to even
    int o_cbuf, o_dm, o_dg, o_red, o_real, o_mbar, o_uni, o_state, total;   // offsets in doubles (per group)
};
constexpr int VAR2_STATE_PER_COORD = 13;   // shared memory, per coordinate: x0, csx, csv, x0c, v0, a0, e[7]
// Each planet slot owns one contiguous block [entry k][axis d] of an ODD number of doubles: a lane reaches every entry from
// one base pointer with compile-time offsets (no address arithmetic in the substep loop), and consecutive lanes' 8-byte
// accesses fall into distinct bank pairs.
RV_HD int var2_slot_stride(int D) { return (VAR2_STATE_PER_COORD * D) | 1; }
constexpr int VAR2_HIST_PER_COORD = 14;    // global scratch (L2-resident), per coordinate: er[7], br[7] -- written once per
                                           // accepted step, read only when a step is rejected

RV_HD int var2_min_threads(int nv) { return 32 * ((nv * (nv + 1) / 2 + 31) / 32 + 1); }
// NT = 0: the smallest group that fits; otherwise the launched group size (a multiple of 32, >= var2_min_threads)
RV_HD Var2Layout var2_layout(int P, int D, int nv, int NT = 0) {
    Var2Layout L;
    L.P = P; L.D = D; L.nv = nv; L.n2 = nv * (nv + 1) / 2; L.nsets = 1 + nv + L.n2;
    L.NT = NT > 0 ? NT : var2_min_threads(nv);
    L.nso_warps = L.NT / 32 - 1;
    L.nps = L.nsets * P;
    L.CB = P * D + D;
    L.cstride = (nv + 1) * L.CB;
    if (L.cstride & 1) L.cstride++;
    int o = 0;
    L.o_cbuf = o; o += 8 * L.cstride;      // buffer 0: positions at x0; 1..7: predicted at substep n (1.. reused for the epoch exchange)
    L.o_dm = o; o += (nv > 0 ? nv : 1) * P; if (o & 1) o++;
    L.o_dg = o; o += (nv > 0 ? nv : 1) * P; if (o & 1) o++;   // d(G m_j) / d(parameter): 1 where the parameter is that mass
    L.o_red = o; o += 2 * 2 * 8 + 2;        // ping-pong group maxima (up to 8 warps) + the item broadcast slot
    L.o_real = o; o += P * D; if (o & 1) o++;      // the real lanes' last force (step-size control)
    L.o_mbar = o; o += 8;                   // seven substep mbarriers (8 bytes each)
    L.o_uni = o; o += 8;                    // the walker's masses (VarUniform): read from shared memory where they are used
    L.o_state = o; o += var2_slot_stride(D) * L.nps;
    if (o & 1) o++;
    L.total = o;
    return L;
}
// one or two planets; real + first-order sets must fit one warp at one lane per (set, planet); at most 8 warps per group
// doubles of global history scratch one group needs
RV_HD size_t var2_hist_doubles(int P, int D, int nv) { return (size_t)VAR2_HIST_PER_COORD * D * (size_t)var_nsets(nv) * P; }
RV_HD bool var2_supported(int P, int nv) { return P <= 2 && (nv + 1) * P <= 32 && var2_min_threads(nv) <= 256; }

template <int P, int D>
struct Var2Thread {
    static constexpr int NC = P * D;
    int tid;                       // thread index inside the group
    int role;                      // 0 real, 1 first-order (producer warp; own D coordinates), 2 second-order (all P*D), -1 idle
    int set, planet, pa, pb;
    int slot0;                     // planet slot of coordinate block 0 (so lanes: planet p at slot0 + p * n2)
    int nps, n2;                   // planet slots of the group, second-order sets (strides of the per-coordinate state)
    int ou, oa, ob;                // block offsets inside a producer buffer: own set, parents
    double* st;                    // the group's per-coordinate state in shared memory (see var2_state)
    double q[7][NC];               // b between step attempts, g inside the predictor-corrector loop
    double xn[NC];
    double mon_g, mon_a;           // convergence-monitor contributions of the last substep 7
    double acc;                    // running chi2 / d[a] / dd[a][b] (planet-0 lane of a producer set; so lanes)
};

// entry k of coordinate c (block p = c / D, axis d) of a lane: st[slot * stride + k * D + d], slot = slot0 + p * n2 for so
// lanes and slot0 for producer lanes (block 0 only)
enum : int { VK_X0 = 0, VK_CSX = 1, VK_CSV = 2, VK_X0C = 3, VK_V0 = 4, VK_A0 = 5, VK_E = 6 };
template <int P, int D>
RV_D double& var2_state(const Var2Thread<P, D>& th, int k, int c) {
    constexpr int STRIDE = (VAR2_STATE_PER_COORD * D) | 1;
    const int p = c / D, d = c - p * D;
    return th.st[(th.slot0 + p * th.n2) * STRIDE + k * D + d];
}

template <int P, int D>
RV_D void var2_assign(Var2Thread<P, D>& th, int tid, const Var2Layout& L) {
    th.tid = tid; th.role = -1; th.set = 0; th.planet = 0; th.pa = th.pb = 0; th.slot0 = 0;
    th.nps = L.nps; th.n2 = L.n2; th.st = nullptr;
    const int warp = tid >> 5, lane = tid & 31;
    if (warp < L.nso_warps) {
        if (tid < L.n2) {
            th.role = 2; th.set = 1 + L.nv + tid; th.slot0 = tid;
            int a = 0;
            while ((a + 1) * (a + 2) / 2 <= tid) a++;
            th.pa = a; th.pb = tid - a * (a + 1) / 2;
        }
    } else if (lane < (L.nv + 1) * P) {
        th.set = lane / P; th.planet = lane - th.set * P;
        th.role = th.set == 0 ? 0 : 1;
        th.slot0 = L.n2 * P + lane;
        th.pa = th.pb = th.set == 0 ? 0 : th.set - 1;
    }
    th.ou = th.set * L.CB;
    th.oa = (1 + th.pa) * L.CB; th.ob = (1 + th.pb) * L.CB;
}

// ---- force on ONE planet of a producer set (real or first-order), one code path for both -------------------------------
// real set:         a_p  = -m0 f(x_p + S) - sum_{j != p} m_j f(x_p - x_j),  f(d) = d / r^3,  S = sum mu_j x_j (= -r_star)
// first-order set:  da_p = -sum_j { m_j Df[U_pj] + dm_j f(d_pj) },  Df[u] = u / r^3 - 3 d (d.u) / r^5; star terms with
//                   d = x0_p + S, u = xu_p + SU, dm_star = 0
// Both need the same pair geometry (d, 1/r^3) of the REAL positions, so every producer lane evaluates both and keeps the one
// its set needs: the real lanes do not diverge from the first-order lanes of their warp (for them XU = X0, result unused).
template <int P, int D>
RV_D void var2_force_producer_planet(bool real, int p, const double* __restrict__ X0, const double* __restrict__ XU,
                                     const double (&S)[D], const double (&SU)[D], const double* __restrict__ dmu,
                                     const VarUniform<P>& u, double (&an)[P * D]) {
    double x0p[D], xup[D], ar[D], af[D];
#pragma unroll
    for (int d = 0; d < D; d++) {
        x0p[d] = X0[d]; xup[d] = XU[d];
#pragma unroll
        for (int k = 1; k < P; k++) { x0p[d] = (p == k) ? X0[k * D + d] : x0p[d]; xup[d] = (p == k) ? XU[k * D + d] : xup[d]; }
    }
    {
        double dd[D], U[D], r2 = 0.0, du = 0.0;
#pragma unroll
        for (int d = 0; d < D; d++) {
            dd[d] = x0p[d] + S[d]; U[d] = xup[d] + SU[d];
            r2 = fma(dd[d], dd[d], r2); du = fma(dd[d], U[d], du);
        }
        const double y = rinv1(r2), y2 = y * y, r3i = y * y2, r5i = r3i * y2;
        const double kU = -u.gm0 * r3i, kd = u.gm0 * 3.0 * r5i * du;
#pragma unroll
        for (int d = 0; d < D; d++) { ar[d] = kU * dd[d]; af[d] = fma(kU, U[d], kd * dd[d]); }
    }
#pragma unroll
    for (int j = 0; j < P; j++) {
        if (P == 1) break;
        double dd[D], U[D], r2 = 0.0, du = 0.0;
#pragma unroll
        for (int d = 0; d < D; d++) {
            dd[d] = x0p[d] - X0[j * D + d]; U[d] = xup[d] - XU[j * D + d];
            r2 = fma(dd[d], dd[d], r2); du = fma(dd[d], U[d], du);
        }
        const double y = rinv1(j == p ? 1.0 : r2), y2 = y * y, r3i = y * y2, r5i = r3i * y2;
        const double mj = (j == p) ? 0.0 : u.gm[j], dmj = (j == p) ? 0.0 : dmu[j] * u.gm0;
        const double kU = mj * r3i;
        const double kd = fma(mj * (-3.0 * r5i), du, dmj * r3i);
#pragma unroll
        for (int d = 0; d < D; d++) { ar[d] = fma(-kU, dd[d], ar[d]); af[d] -= fma(kU, U[d], kd * dd[d]); }
    }
#pragma unroll
    for (int d = 0; d < D; d++) an[d] = real ? ar[d] : af[d];
}

// ---- force on a whole second-order set (so lanes) ------------------------------------------------------------------
// d2a_i = -sum_j { m_j (Df[U] + D2f[A,B]) + dm_j^a Df[B] + dm_j^b Df[A] },  (d2 m = 0)
// D2f[u,w] = -3 [u (d.w) + w (d.u) + d (u.w)] / r^5 + 15 d (d.u)(d.w) / r^7.  X0 / XA / XB: producer blocks (positions of
// the real set and of the two parents, each followed by its star sum).
// Register pressure: the producer blocks are re-read from shared memory pair by pair (a compiler fence keeps the loads next to
// their uses) instead of being held across the whole evaluation -- shared-memory loads are cheap, spills to local memory
// (long-scoreboard stalls) are not.
RV_D void var2_fence() {
#if defined(__CUDA_ARCH__)
    asm volatile("" ::: "memory");
#endif
}
template <int P, int D>
RV_D void var2_force_second(const double (&xu)[P * D], const double* __restrict__ X0, const double* __restrict__ XA,
                            const double* __restrict__ XB, const double* __restrict__ dma, const double* __restrict__ dmb,
                            const double* __restrict__ dga, const double* __restrict__ dgb,
                            const VarUniform<P>& u, double (&an)[P * D]) {
    double SU[D];
#pragma unroll
    for (int d = 0; d < D; d++) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < P; j++) s = fma(u.mu[j], xu[j * D + d], fma(dma[j], XB[j * D + d], fma(dmb[j], XA[j * D + d], s)));
        SU[d] = s;
    }
    var2_fence();
    // star pairs (dm_star = 0)
#pragma unroll
    for (int i = 0; i < P; i++) {
        double dd[D], A[D], B[D], U[D], r2 = 0.0, da = 0.0, db = 0.0, ab = 0.0, du = 0.0;
#pragma unroll
        for (int d = 0; d < D; d++) {
            dd[d] = X0[i * D + d] + X0[P * D + d]; A[d] = XA[i * D + d] + XA[P * D + d];
            B[d] = XB[i * D + d] + XB[P * D + d]; U[d] = xu[i * D + d] + SU[d];
            r2 = fma(dd[d], dd[d], r2); da = fma(dd[d], A[d], da); db = fma(dd[d], B[d], db);
            ab = fma(A[d], B[d], ab); du = fma(dd[d], U[d], du);
        }
        // m / r^3, -3 m / r^5 and 15 m / r^7 = (-3 m / r^5)(-5 / r^2): the mass rides on the first power (12 scalar
        // operations instead of 15)
        const double y = rinv1(r2), y2 = y * y;
        const double kU = (y * u.gm0) * y2;
        const double c5m = kU * (-3.0 * y2);
        const double kA = c5m * db, kB = c5m * da;
        const double kd = c5m * fma(-5.0 * y2, da * db, du + ab);
#pragma unroll
        for (int d = 0; d < D; d++) an[i * D + d] = -fma(kU, U[d], fma(kA, A[d], fma(kB, B[d], kd * dd[d])));
        var2_fence();
    }
    // planet pairs, both sides from one set of geometric scalars
#pragma unroll
    for (int i = 0; i < P; i++)
#pragma unroll
        for (int j = i + 1; j < P; j++) {
            double dd[D], A[D], B[D], U[D], r2 = 0.0, da = 0.0, db = 0.0, ab = 0.0, du = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) {
                dd[d] = X0[i * D + d] - X0[j * D + d]; A[d] = XA[i * D + d] - XA[j * D + d]; B[d] = XB[i * D + d] - XB[j * D + d];
                U[d] = xu[i * D + d] - xu[j * D + d];
                r2 = fma(dd[d], dd[d], r2); da = fma(dd[d], A[d], da); db = fma(dd[d], B[d], db);
                ab = fma(A[d], B[d], ab); du = fma(dd[d], U[d], du);
            }
            const double y = rinv1(r2), y2 = y * y, r3i = y * y2;
            const double c5 = r3i * (-3.0 * y2);
            const double g0 = c5 * fma(-5.0 * y2, da * db, du + ab);      // coefficient of m d
            const double c5db = c5 * db, c5da = c5 * da;
            // dga / dgb: derivative of G m_j with respect to the parents' parameters (1 where the parameter is that mass)
            const double dgaj = dga[j], dgbj = dgb[j], dgai = dga[i], dgbi = dgb[i];
            {   // side i: masses of j
                const double m = u.gm[j];
                const double kU = m * r3i, kA = fma(m, c5db, dgbj * r3i), kB = fma(m, c5da, dgaj * r3i);
                const double kd = fma(m, g0, fma(dgaj, c5db, dgbj * c5da));
#pragma unroll
                for (int d = 0; d < D; d++) an[i * D + d] -= fma(kU, U[d], fma(kA, A[d], fma(kB, B[d], kd * dd[d])));
            }
            {   // side j: masses of i, opposite sign
                const double m = u.gm[i];
                const double kU = m * r3i, kA = fma(m, c5db, dgbi * r3i), kB = fma(m, c5da, dgai * r3i);
                const double kd = fma(m, g0, fma(dgai, c5db, dgbi * c5da));
#pragma unroll
                for (int d = 0; d < D; d++) an[j * D + d] += fma(kU, U[d], fma(kA, A[d], fma(kB, B[d], kd * dd[d])));
            }
            var2_fence();
        }
}

// ---- predictor / corrector over the first N coordinates of a lane ------------------------------------------------------
template <int N, int P, int D>
RV_D void var2_predict_positions(Var2Thread<P, D>& th, int n, double dt) {
    const double dth = dt * rvtabm::H[n];
    const double c0 = rvtabm::PG[n][0], c1 = rvtabm::PG[n][1], c2 = rvtabm::PG[n][2], c3 = rvtabm::PG[n][3],
                 c4 = rvtabm::PG[n][4], c5 = rvtabm::PG[n][5], c6 = rvtabm::PG[n][6];
#pragma unroll
    for (int c = 0; c < N; c++) {
        double p0 = fma(c0, th.q[0][c], 0.5 * var2_state(th, VK_A0, c));
        p0 = fma(c1, th.q[1][c], p0);
        p0 = fma(c2, th.q[2][c], p0);
        double p1 = c3 * th.q[3][c];
        p1 = fma(c4, th.q[4][c], p1);
        p1 = fma(c5, th.q[5][c], p1);
        p1 = fma(c6, th.q[6][c], p1);
        const double inner = fma(dth, p0 + p1, var2_state(th, VK_V0, c));
        th.xn[c] = fma(dth, inner, var2_state(th, VK_X0C, c));
    }
}

template <int n, int N, int P, int D>
RV_D void var2_corrector_n(Var2Thread<P, D>& th, const double (&an)[P * D]) {
    double mg = 0.0, ma = 0.0;
#pragma unroll
    for (int c = 0; c < N; c++) {
        const double gk = an[c] - var2_state(th, VK_A0, c);
        double gn;
        if (n <= 2) {
            gn = gk * rvtab::GA[n];
            if (n == 2) gn = fma(-th.q[0][c], rvtab::GB[n][0], gn);
        } else {
            double s0 = gk * rvtab::GA[n], s1 = -th.q[1][c] * rvtab::GB[n][1];
#pragma unroll
            for (int i = 0; i < n - 1; i++) {
                if (i == 1) continue;
                if (i & 1) s1 = fma(-th.q[i][c], rvtab::GB[n][i], s1);
                else s0 = fma(-th.q[i][c], rvtab::GB[n][i], s0);
            }
            gn = s0 + s1;
        }
        if (n == 7) {
            const double ak = fabs(an[c]), dg = fabs(gn - th.q[6][c]);
            norm_max(ak, ma);
            norm_max(dg, mg);
        }
        th.q[n - 1][c] = gn;
    }
    if (n == 7) { th.mon_g = mg; th.mon_a = ma; }
}
template <int N, int P, int D>
RV_D void var2_corrector(Var2Thread<P, D>& th, int n, const double (&an)[P * D]) {
    switch (n) {
        case 1: var2_corrector_n<1, N>(th, an); break;
        case 2: var2_corrector_n<2, N>(th, an); break;
        case 3: var2_corrector_n<3, N>(th, an); break;
        case 4: var2_corrector_n<4, N>(th, an); break;
        case 5: var2_corrector_n<5, N>(th, an); break;
        case 6: var2_corrector_n<6, N>(th, an); break;
        default: var2_corrector_n<7, N>(th, an); break;
    }
}

// Initial conditions of the lane's coordinates: the jet of the barycentric state with respect to the set's parameters
// (state.py:229-248: add_variation + vary + move_to_com).  Producer lanes keep their own planet in block 0.
template <int P, int D>
RV_D void var2_initial(const Var2Thread<P, D>& th, const Model* __restrict__ md, const double (&el)[P][NELEM],
                       double (&x0)[P * D], double (&v0)[P * D]) {
    const double m0 = md->m_star;
    Jet mt = J(m0), cx[3], cv[3];
#pragma unroll
    for (int d = 0; d < 3; d++) { cx[d] = J(0.0); cv[d] = J(0.0); }
    JState own[P];
    for (int i = 0; i < P; i++) {
        Jet ej[NELEM];
#pragma unroll
        for (int k = 0; k < NELEM; k++) ej[k] = J(el[i][k]);
        if (th.role >= 1 && md->free_planet[th.pa] == i) ej[md->free_elem[th.pa]].d1 = 1.0;
        if (th.role == 2 && md->free_planet[th.pb] == i) ej[md->free_elem[th.pb]].d2 = 1.0;
        const JState s = pal_to_cart_jet(ej, m0);
        mt = mt + s.m;
#pragma unroll
        for (int d = 0; d < 3; d++) { cx[d] = cx[d] + s.m * s.x[d]; cv[d] = cv[d] + s.m * s.v[d]; }
        own[i] = s;
    }
    const Jet im = jinv(mt);
#pragma unroll
    for (int i = 0; i < P; i++)
#pragma unroll
        for (int d = 0; d < D; d++) {
            const Jet x = own[i].x[d] - cx[d] * im, v = own[i].v[d] - cv[d] * im;
            x0[i * D + d] = th.role == 0 ? x.v : (th.role == 1 ? x.d1 : x.d12);
            v0[i * D + d] = th.role == 0 ? v.v : (th.role == 1 ? v.d1 : v.d12);
        }
    if (th.role <= 1) {      // producer lane: its own planet moves to block 0
#pragma unroll
        for (int d = 0; d < D; d++) {
            double xs = x0[d], vs = v0[d];
#pragma unroll
            for (int k = 1; k < P; k++) { xs = (th.planet == k) ? x0[k * D + d] : xs; vs = (th.planet == k) ? v0[k * D + d] : vs; }
            x0[d] = xs; v0[d] = vs;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// The group algorithm.  Exec provides (device / sequential host emulation):
//   each(f)            run f(Var2Thread&) for every thread of the group
//   sync()             group barrier
//   producer_sync()    barrier among the lanes of the producer warp (no-op for the others)
//   signal(n)          producer warp: substep n is published
//   wait(n)            second-order warps: wait until substep n is published
//   stage_max / read_max / fetch / add_work   as in rv_var.cuh (group-wide)
// hist: this group's global scratch of var2_hist_doubles() doubles (br, er: the rejected-step history)
template <int P, int D, class Exec>
RV_D void var2_run_items(Exec& ex, const VarArgs& a, const Var2Layout& L, double* __restrict__ sm, double* __restrict__ hist) {
    constexpr int NC = P * D;
    const Model* __restrict__ md = a.model;
    const int nv = md->nvars;
    const int n2 = L.n2;
    double* const cbuf = sm + L.o_cbuf;
    double* const vxs = cbuf + L.cstride;          // the epoch exchange reuses the substep buffers (dead between steps)
    double* const dm = sm + L.o_dm;
    double* const dg = sm + L.o_dg;
    double* const realv = sm + L.o_real;
    double* const state = sm + L.o_state;
    const double m0 = md->m_star;
    const long long n_items = 2 * a.W;
    // group-uniform masses live in shared memory (every thread writes the same values): values read through this
    // reference are re-loaded after each barrier instead of occupying registers across the whole integration
    static_assert(sizeof(VarUniform<P>) <= 8 * sizeof(double), "VarUniform must fit its shared-memory slot");
    VarUniform<P>& u = *reinterpret_cast<VarUniform<P>*>(sm + L.o_uni);
    const double epsilon = md->epsilon;
    // per-coordinate state: shared memory through var2_state(th, VK_*, c); the rejected-step history (k = 0..6 er, 7..13 br,
    // as var_accept_coord stores it) in the group's global scratch with the same slot striding
    auto ST = [&](const Var2Thread<P, D>& th, int k, int c) -> double& { return var2_state(th, k, c); };
    auto HS = [&](const Var2Thread<P, D>& th, int k, int c) -> double& {
        const int p = c / D, d = c - p * D;
        return hist[(size_t)(th.slot0 + p * n2) * (VAR2_HIST_PER_COORD * D) + k * D + d];
    };
    enum { K_X0 = VK_X0, K_CSX = VK_CSX, K_CSV = VK_CSV, K_X0C = VK_X0C, K_V0 = VK_V0, K_A0 = VK_A0, K_E = VK_E };
    ex.each([&](Var2Thread<P, D>& th) { th.st = state; });
    // a lane's coordinate count: producer lanes carry one planet, so lanes the whole set
    auto NCOF = [](const Var2Thread<P, D>& th) { return th.role == 2 ? NC : D; };

    ex.each([&](Var2Thread<P, D>& th) {
        if (th.tid < nv * P) {
            const int q = th.tid / P, j = th.tid - q * P;
            dm[th.tid] = (md->free_planet[q] == j && md->free_elem[q] == EL_M) ? 1.0 / m0 : 0.0;
            dg[th.tid] = (md->free_planet[q] == j && md->free_elem[q] == EL_M) ? 1.0 : 0.0;
        }
    });

    for (;;) {
        const long long item = ex.fetch(a.item_counter);
        if (item >= n_items) break;
        const long long wi = item < a.W ? item : item - a.W;
        double el[P][NELEM];
        const bool bad = var_item_setup<P>(md, a.theta, wi, nv, el);
        int final_status = ST_PRIOR;
        unsigned long long n_force = 0, n_attempt = 0;
        if (!(bad && a.check_prior)) {
            const double min2 = var_exit_min2<P>(el, m0, md->hill_factor);
            ex.sync();                                  // nobody still reads the previous item's masses
#pragma unroll
            for (int i = 0; i < P; i++) { u.gm[i] = el[i][EL_M]; u.mu[i] = el[i][EL_M] / m0; }
            u.gm0 = m0; u.epsilon = epsilon; u.min2 = min2;
            ex.sync();

            // Producer lanes publish their planet's position into buffer b (x0 or the predicted xn), and -- after a
            // producer-warp sync -- the planet-0 lane of each set adds the set's star sum:
            //   real set   S  = sum_j mu_j x_j            first-order set a   SA = sum_j (mu_j xa_j + dmu^a_j x_j)
            auto publish_positions = [&](int b, bool from_xn) {
                double* Xw = cbuf + b * L.cstride;
                ex.each([&](Var2Thread<P, D>& th) {
                    if (th.role != 0 && th.role != 1) return;
                    double* blk = Xw + th.ou + th.planet * D;
#pragma unroll
                    for (int d = 0; d < D; d++) blk[d] = from_xn ? th.xn[d] : ST(th, K_X0, d);
                });
                ex.producer_sync();
                ex.each([&](Var2Thread<P, D>& th) {
                    if ((th.role != 0 && th.role != 1) || th.planet != 0) return;
                    double* blk = Xw + th.ou;
                    const double* dma = dm + th.pa * P;
#pragma unroll
                    for (int d = 0; d < D; d++) {
                        double s = 0.0;
#pragma unroll
                        for (int j = 0; j < P; j++) {
                            s = fma(u.mu[j], blk[j * D + d], s);
                            if (th.role == 1) s = fma(dma[j], Xw[j * D + d], s);
                        }
                        blk[NC + d] = s;
                    }
                });
            };
            // force on the lane's coordinates at positions x with the producer data of buffer b.  Producer lanes need
            // their own set's star sum, which the planet-0 lane wrote after the producer sync: callers sync again first.
            auto force = [&](const Var2Thread<P, D>& th, int b, const double (&x)[NC], double (&an)[NC]) {
                const double* Xr = cbuf + b * L.cstride;
                if (th.role == 2) {
                    var2_force_second<P, D>(x, Xr, Xr + th.oa, Xr + th.ob, dm + th.pa * P, dm + th.pb * P, dg + th.pa * P, dg + th.pb * P, u, an);
                } else {
                    double S[D], SU[D];
#pragma unroll
                    for (int d = 0; d < D; d++) { S[d] = Xr[NC + d]; SU[d] = Xr[th.ou + NC + d]; }
                    var2_force_producer_planet<P, D>(th.role == 0, th.planet, Xr, Xr + th.ou, S, SU, dm + th.pa * P, u, an);
                }
            };

            ex.each([&](Var2Thread<P, D>& th) {
                if (th.role < 0) return;
                double x0[NC], v0[NC];
                var2_initial(th, md, el, x0, v0);
                th.acc = 0.0; th.mon_g = 0.0; th.mon_a = 0.0;
                const int nc = NCOF(th);
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    th.xn[c] = x0[c];
#pragma unroll
                    for (int k = 0; k < 7; k++) th.q[k][c] = 0.0;
                    if (c < nc) {
                        ST(th, K_X0, c) = x0[c]; ST(th, K_CSX, c) = 0.0; ST(th, K_CSV, c) = 0.0;
                        ST(th, K_X0C, c) = x0[c]; ST(th, K_V0, c) = v0[c]; ST(th, K_A0, c) = 0.0;
#pragma unroll
                        for (int k = 0; k < 7; k++) { ST(th, K_E + k, c) = 0.0; HS(th, k, c) = 0.0; HS(th, 7 + k, c) = 0.0; }
                    }
                }
            });
            publish_positions(0, false);
            ex.sync();

            VarClock w;
            w.t = 0.0; w.dt = md->dt0; w.dt_last_done = 0.0;

            // ---- one IAS15 step attempt of the whole group; bit0 accepted, bit1 encounter after the step ----
            auto attempt = [&]() -> int {
                n_attempt++;
                ex.each([&](Var2Thread<P, D>& th) {
                    if (th.role < 0) return;
                    const int nc = NCOF(th);
                    double x0[NC];
#pragma unroll
                    for (int cc = 0; cc < NC; cc++) x0[cc] = cc < nc ? ST(th, K_X0, cc) : 0.0;
                    double a0[NC];
                    force(th, 0, x0, a0);
#pragma unroll
                    for (int cc = 0; cc < NC; cc++) {
                        if (cc >= nc) break;
                        ST(th, K_A0, cc) = a0[cc];
                        ST(th, K_X0C, cc) = x0[cc] - ST(th, K_CSX, cc);
                        var_g_from_b<NC>(th.q, cc);
                    }
                });
                Ratio pc_err{1e300, 1.0}, pc_last{2.0, 1.0};
                int it = 0;
                const double dt = w.dt;
                while (true) {
                    if (ratio_lt(pc_err, 1e-16) || (it > 2 && ratio_le(pc_last, pc_err)) || it >= 12) break;
                    pc_last = pc_err;
                    it++;
#pragma unroll 1
                    for (int nn = 1; nn <= 7; nn++) {
                        // producer warp: predict, publish, signal, then its own force + corrector
                        ex.each([&](Var2Thread<P, D>& th) { if (th.role == 0 || th.role == 1) var2_predict_positions<D>(th, nn, dt); });
                        publish_positions(nn, true);
                        ex.signal(nn);
                        ex.producer_sync();
                        ex.each([&](Var2Thread<P, D>& th) {
                            if (th.role != 0 && th.role != 1) return;
                            double an[NC];
                            force(th, nn, th.xn, an);
                            var2_corrector<D>(th, nn, an);
                            if (nn == 7 && th.role == 0) {
#pragma unroll
                                for (int d = 0; d < D; d++) realv[th.planet * D + d] = an[d];
                            }
                        });
                        // second-order warps: predict in registers, wait for the producer's substep, force + corrector
                        ex.each([&](Var2Thread<P, D>& th) { if (th.role == 2) var2_predict_positions<NC>(th, nn, dt); });
                        ex.wait(nn);
                        ex.each([&](Var2Thread<P, D>& th) {
                            if (th.role != 2) return;
                            double an[NC];
                            force(th, nn, th.xn, an);
                            var2_corrector<NC>(th, nn, an);
                        });
                    }
                    ex.each([&](Var2Thread<P, D>& th) {
                        ex.stage_max(th, th.role >= 0 ? th.mon_g : 0.0, th.role >= 0 ? th.mon_a : 0.0);
                    });
                    ex.sync();
                    double maxdg, maxat;
                    ex.read_max(maxdg, maxat);
                    pc_err.num = maxdg; pc_err.den = maxat;
                    n_force += 7;
                }
                n_force += 1;
                // b from g; then step-size control over the real particles
                ex.each([&](Var2Thread<P, D>& th) {
                    double mb = 0.0, ma = 0.0;
                    if (th.role >= 0) {
                        const int nc = NCOF(th);
#pragma unroll
                        for (int cc = 0; cc < NC; cc++) {
                            if (cc >= nc) break;
                            var_b_from_g<NC>(th.q, cc);
                        }
                    }
                    if (th.role == 0) {
                        double v2 = 0.0, x2 = 0.0;
#pragma unroll
                        for (int d = 0; d < D; d++) { const double vd = ST(th, K_V0, d); v2 = fma(vd, vd, v2); x2 = fma(th.xn[d], th.xn[d], x2); }
                        const bool keep = !(fabs(v2 * dt * dt) < 1e-16 * x2);
#pragma unroll
                        for (int d = 0; d < D; d++) {
                            const double ak = fabs(realv[th.planet * D + d]), b6 = fabs(th.q[6][d]);
                            if (keep) norm_max(ak, ma);
                            if (keep) norm_max(b6, mb);
                        }
                    }
                    ex.stage_max(th, mb, ma);
                });
                ex.sync();
                double maxb6, maxak;
                ex.read_max(maxb6, maxak);
                const bool accepted = var_step_control(maxb6, maxak, epsilon, w, dt);
                if (!accepted) {
                    if (w.dt_last_done != 0.0) {
                        const double q = w.dt / w.dt_last_done;
                        ex.each([&](Var2Thread<P, D>& th) {
                            if (th.role < 0) return;
                            const int nc = NCOF(th);
                            auto e = [&](int k, int c) -> double& { return ST(th, K_E + k, c); };
                            auto h = [&](int k, int c) -> double& { return HS(th, k, c); };
#pragma unroll
                            for (int cc = 0; cc < NC; cc++) {
                                if (cc >= nc) break;
                                var_reject_coord<NC>(th.q, cc, q, e, h);
                            }
                        });
                    }
                } else {
                    const double dt2 = dt * dt, q = w.dt / dt;
                    ex.each([&](Var2Thread<P, D>& th) {
                        if (th.role < 0) return;
                        const int nc = NCOF(th);
                        auto e = [&](int k, int c) -> double& { return ST(th, K_E + k, c); };
                        auto h = [&](int k, int c) -> double& { return HS(th, k, c); };
#pragma unroll
                        for (int cc = 0; cc < NC; cc++) {
                            if (cc >= nc) break;
                            var_accept_coord<NC>(th.q, cc, ST(th, K_X0, cc), ST(th, K_CSX, cc), ST(th, K_V0, cc), ST(th, K_CSV, cc),
                                                 ST(th, K_A0, cc), dt, dt2, q, e, h);
                        }
                    });
                    w.t += dt;
                    w.dt_last_done = dt;
                }
                // publish x0 of the producer sets for the encounter test and the next attempt's a0
                publish_positions(0, false);
                ex.sync();
                int result = accepted ? 1 : 0;
                if (var_encounter<P, D>(cbuf, u)) result |= 2;
                return result;
            };

            final_status = var_leg_epochs(ex, a, md, item, w, attempt,
                [&]() { return var_encounter<P, D>(cbuf, u); },
                [&](int ie) {
                    // star vx of every set, chi2 / d / dd sums (state.py:264-271)
                    ex.each([&](Var2Thread<P, D>& th) {
                        if (th.role < 0) return;
                        if (th.role == 2) {
#pragma unroll
                            for (int p = 0; p < P; p++) vxs[th.set * P + p] = ST(th, K_V0, p * D);
                        } else {
                            vxs[th.set * P + th.planet] = ST(th, K_V0, 0);
                        }
                    });
                    ex.sync();
                    const double svx = var_star_vx<P>(vxs, dm, u, 0, 0, 0, 0, 0, 0);
                    if (!isfinite(svx)) return false;
                    const double res = svx - a.orv[ie], er = a.oerr[ie];
                    const double den = er * er * a.npoints;
                    ex.each([&](Var2Thread<P, D>& th) {
                        if (th.role < 0 || (th.role <= 1 && th.planet != 0)) return;
                        th.acc += var_epoch_term<P>(vxs, dm, u, th.role, th.set, 1 + th.pa, 1 + th.pb, th.pa, th.pb, res, den);
                    });
                    return true;
                });
        }
        const int fs = final_status;
        ex.each([&](Var2Thread<P, D>& th) {
            if (th.tid == 0) a.part_status[item] = fs;
            if (fs == ST_OK && th.role >= 0 && (th.role == 2 || th.planet == 0)) a.part[item * L.nsets + th.set] = th.acc;
        });
        ex.add_work(a.work_counters, n_force, n_attempt);
    }
}

}  // namespace rv
