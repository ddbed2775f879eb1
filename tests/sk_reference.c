/*
 * sk_reference.c — TEST INFRASTRUCTURE ONLY.  The density modes of one snapshot as a direct sum in double:
 *     rho_k = sum_j exp(i 2 pi t_j),  t_j = (n_x x_j + n_y y_j) / box  reduced to [-1/2, 1/2] by rint,
 * over the fp32 positions converted exactly to double.  OpenMP over the wave vectors; each vector's sum runs
 * in particle order, so the result does not depend on the thread count.  Compiled by tests/sk_reference.py.
 * The product never loads it.
 */
#include <math.h>
#include <stdint.h>

void skref_modes(int64_t N, const float* R, double box, int64_t K, const int32_t* nvec, double* rho) {
    const double two_pi = 6.283185307179586476925287;
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t k = 0; k < K; ++k) {
        const double nx = (double)nvec[2 * k], ny = (double)nvec[2 * k + 1];
        double re = 0.0, im = 0.0;
        for (int64_t j = 0; j < N; ++j) {
            double t = (nx * (double)R[2 * j] + ny * (double)R[2 * j + 1]) / box;
            t -= rint(t);
            re += cos(two_pi * t);
            im += sin(two_pi * t);
        }
        rho[2 * k] = re;
        rho[2 * k + 1] = im;
    }
}
