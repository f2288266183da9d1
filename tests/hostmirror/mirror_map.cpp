// TEST-ONLY host build of the fit's per-walker arithmetic (rv_map.cuh): the Newton step and the line-search decision.
// A library of its own, compiled by tests/test_map_cpu.py into a temporary directory; NOT part of the product library.
#include <math.h>
#include <vector>
#include "../../rvel_mcmc_b200/csrc/rv_map.cuh"

extern "C" int mirror_map_step(int n, const double* th, const double* g, const double* H, double mu, int n_iter, int max_iter,
                               double tol, int n_trial, double* rows, double* dec) {
    std::vector<double> scr((size_t)2 * n * n, 0.0);
    return rv::map_step_one(n, th, g, H, mu, n_iter, max_iter, tol, n_trial, rows, dec, scr.data());
}

extern "C" int mirror_map_select(int n, int n_trial, const double* rows, const double* tlogp, const int* tstatus, double* th,
                                 double* mu, int* n_iter, int* code) {
    return rv::map_select_one(n, n_trial, rows, tlogp, tstatus, th, *mu, *n_iter, *code);
}
