// Host build of the Jacobian mode of the implicit fwd+bwd kernel (sq_recovery_b200/csrc/sqloss.cu
// sq_depth_projection_jacobian) -- TEST TOOL, never part of the product.
//
// The group loop of emu_depth_vjp (emu_vjp.cpp) with the two things the Jacobian mode changes: the column weight is 1, and
// every column keeps its own sums, which finalize_sample maps to the column's row at the VJP's scale -k tau / n.  Same pool,
// fp64 refinement, corrected suffix weights and one-sample weight cut; each column's entries are added in entry order, as
// the kernel's lanes add them.  libm instead of MUFU.  tests/test_render_jacobian.py checks it against the oracle's
// forward-mode Jacobian, and checks that emu_depth_vjp with a one-hot upstream returns its rows bit for bit -- which pins
// this loop to that one.
#include "sq_core.cuh"

using namespace sq;

extern "C" {

// jac: [B, n, n, 12] fp32, image orientation: d depth[b, row, col] / d pred[b]
int emu_depth_jacobian(const double* pred, int B, int n, double step, double z0, float tau, float k, float* jac) {
    Grid g = make_grid(n, step, z0);
    ImplicitParams P{k * kLog2e, tau * kLog2e, implicit_cull_bound(k * kLog2e), implicit_active_bits(k * kLog2e, n, 1)};
    for (int b = 0; b < B; ++b) {
        double p[12]; for (int i = 0; i < 12; ++i) p[i] = pred[12 * b + i];
        SampleFull S; prep_sample(p, true, g, S);
        for (int g0 = 0; g0 < n * n; g0 += 32) {
            float qcf[kBwdPool], qpre[kBwdPool], qx[kBwdPool], qd[kBwdPool];
            BwdQueue q{qcf, qpre, qx, qd, (n <= kPoolMaxPlanes && S.cf0 < 1.0f) ? kBwdPool : 0, 0, 0u};
            int nr = 0, top = q.cap - 1;
            float bh[32][3], bl[32][3], U[32], dx[32], dy[32];
            int head[32], rowv[32], colv[32];
            Acc a[32];
            const int cols = n * n - g0 < 32 ? n * n - g0 : 32;
            for (int L = 0; L < cols; ++L) {
                const int ib = (g0 + L) / n, ia = (g0 + L) - ib * n;
                float cg[11];
                column_base(S, g, ia, ib, bh[L], bl[L]);
                int c_lo, c_hi;
                column_range(S, g, P.bound, bh[L], c_lo, c_hi);
                warp_range(n, c_lo, c_hi);
                U[L] = 0.f; head[L] = kNoLink; bool spilled = false;
                q.lane = L;
                const int own_lo = c_hi >= c_lo ? c_lo : n;
                implicit_column<true, true, true>(S, g, P, bh[L], bl[L], c_lo, c_hi, own_lo, cg, &q, &U[L], &nr, &top, &spilled, &head[L]);
                rowv[L] = n - 1 - ib; colv[L] = ia;
                acc_zero(a[L]);
                dx[L] = (float)(grid_coord(g, ia) - S.t[0]); dy[L] = (float)(grid_coord(g, ib) - S.t[1]);
                if (spilled) implicit_fold(a[L], cg, 1.0f, dx[L], dy[L]);
            }
            for (int e = 0; e < nr; ++e) {
                const int L = entry_lane(qcf[e]);
                queue_refine_entry(S, g.step, P.kl, q, e, (double)bh[L][0] + (double)bl[L][0], (double)bh[L][1] + (double)bl[L][1],
                                   (double)bh[L][2] + (double)bl[L][2], default_tabs());
            }
            const int np = q.cap - 1 - top;
            for (int j = 0; j < nr + np; ++j) {
                const int at = j < nr ? j : q.cap - 1 - (j - nr), L = entry_lane(qcf[at]);
                const float cf = entry_cf(S, qcf[at]);
                Bwd bq;
                queue_entry_backward<true>(S, bh[L], bl[L], cf, qx[at], queue_suffix_weight(q, at, head[L], U[L], tau), 1.0f, true, bq);
                acc_add_point(a[L], bq, cf, dx[L], dy[L]);
            }
            for (int L = 0; L < cols; ++L) {
                double accd[kAccN] = {0};
                for (int i = 0; i < 3; ++i) accd[i] = a[L].gs[i];
                for (int i = 0; i < 9; ++i) accd[3 + i] = a[L].gm[i];
                for (int i = 0; i < 3; ++i) accd[12 + i] = a[L].wa[i];
                accd[15] = a[L].ge[0]; accd[16] = a[L].ge[1];
                double gr[12];
                finalize_sample(S, g, accd, -(double)k * tau / (double)n, true, gr);
                float* out = jac + (((size_t)b * n + rowv[L]) * n + colv[L]) * 12;
                for (int i = 0; i < 12; ++i) out[i] = (float)gr[i];
            }
        }
    }
    return 0;
}

}  // extern "C"
