// Host build of the LeastSquares normal equations (sq_recovery_b200/csrc/sqloss.cu sq_least_squares_points_normal) -- TEST
// TOOL, never part of the product.
//
// lsq_point's GN mode point by point: each point's 18 sums and 78 J^T J sums in fp32, added across points in fp64, then
// finalize_kernel<FIN_LSQ_GN>'s arithmetic (energy, gradient with the prefactor's a term, a1 a2 a3 times the J^T J sums,
// clamped-out rows and columns zero).  libm instead of MUFU.  tests/test_lsq_normal.py checks it against the oracle.
#include "sq_core.cuh"

using namespace sq;

extern "C" {

// points: [sum m, 3] (x, y, z) with offsets[B+1]; energy [B]; grad [B, 12]; jtj [B, 12, 12]
int emu_lsq_normal(const double* pred, int B, const float* points, const long long* offsets, double* energy, double* grad,
                   double* jtj) {
    const Grid g = make_grid(2, 1.0, 0.0);
    for (int b = 0; b < B; ++b) {
        double p[12]; for (int i = 0; i < 12; ++i) p[i] = pred[12 * b + i];
        SampleFull S; prep_sample(p, true, g, S);
        JacConst jc; jac_const(S, jc);
        double accd[kAccN] = {0}, jd[kJtJN] = {0};
        for (long long j = offsets[b]; j < offsets[b + 1]; ++j) {
            Acc a; acc_zero(a);
            float jt[kJtJN] = {0};
            a.loss = lsq_point<true, true>(S, points[3 * j], points[3 * j + 1], points[3 * j + 2], a, &jc, jt);
            for (int i = 0; i < 3; ++i) accd[i] += a.gs[i];
            for (int i = 0; i < 9; ++i) accd[3 + i] += a.gm[i];
            for (int i = 0; i < 3; ++i) accd[12 + i] += a.wa[i];
            accd[15] += a.ge[0]; accd[16] += a.ge[1]; accd[17] += a.loss;
            for (int e = 0; e < kJtJN; ++e) jd[e] += jt[e];
        }
        const double vol = S.a[0] * S.a[1] * S.a[2];
        energy[b] = accd[17] * vol;
        double* gr = grad + 12 * b;
        finalize_sample(S, g, accd, 2.0 * vol, false, gr);
        for (int i = 0; i < 3; ++i) gr[i] += S.mask[i] * (vol * S.ia[i]) * accd[17];
        int e = 0;
        for (int k = 0; k < 12; ++k)
            for (int l = k; l < 12; ++l, ++e) {
                const bool live = (k >= 8 || S.mask[k] != 0.f) && (l >= 8 || S.mask[l] != 0.f);
                jtj[144 * b + 12 * k + l] = jtj[144 * b + 12 * l + k] = live ? vol * jd[e] : 0.0;
            }
    }
    return 0;
}

}  // extern "C"
