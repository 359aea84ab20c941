// Host build of the VJP mode of the implicit fwd+bwd kernel (sq_recovery_b200/csrc/sqloss.cu sq_depth_projection_vjp) --
// TEST TOOL, never part of the product.
//
// The loop of emu_implicit (emu.cpp) with the three things the VJP mode changes: the column weight is the upstream pixel
// dL/d depth[b, row, col] instead of sign(depth - target); the finalize scale is that of d depth / d theta alone, -k tau / n;
// the weight cut is the one-sample rule implicit_active_bits(kl, n, 1).  No loss.  Same pool, fp64 refinement and
// corrected suffix weights (sq_core.cuh), one group of 32 columns (raster order) at a time.  libm instead of MUFU.
// tests/test_depth_render_vjp.py checks it against the oracle's autograd VJP and, where every scaling is exact, against
// emu_implicit's gradient bit for bit -- which also pins this loop to emu_implicit's.
#include "sq_core.cuh"

using namespace sq;

extern "C" {

// upstream: [B, n, n] fp32, image orientation (row, col); grad: [B, 12]
int emu_depth_vjp(const double* pred, int B, int n, double step, double z0, const float* upstream, float tau, float k,
                  double* grad) {
    Grid g = make_grid(n, step, z0);
    ImplicitParams P{k * kLog2e, tau * kLog2e, implicit_cull_bound(k * kLog2e), implicit_active_bits(k * kLog2e, n, 1)};
    for (int b = 0; b < B; ++b) {
        double p[12]; for (int i = 0; i < 12; ++i) p[i] = pred[12 * b + i];
        SampleFull S; prep_sample(p, true, g, S);
        double accd[kAccN] = {0};
        for (int g0 = 0; g0 < n * n; g0 += 32) {
            float qcf[kBwdPool], qpre[kBwdPool], qx[kBwdPool], qd[kBwdPool];
            BwdQueue q{qcf, qpre, qx, qd, (n <= kPoolMaxPlanes && S.cf0 < 1.0f) ? kBwdPool : 0, 0, 0u};
            int nr = 0, top = q.cap - 1;
            float bh[32][3], bl[32][3], U[32], w[32], dx[32], dy[32];
            int head[32];
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
                const int row = n - 1 - ib, col = ia;
                acc_zero(a[L]);
                w[L] = upstream[(size_t)b * n * n + row * n + col];
                dx[L] = (float)(grid_coord(g, ia) - S.t[0]); dy[L] = (float)(grid_coord(g, ib) - S.t[1]);
                if (spilled) implicit_fold(a[L], cg, w[L], dx[L], dy[L]);
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
                queue_entry_backward<true>(S, bh[L], bl[L], cf, qx[at], queue_suffix_weight(q, at, head[L], U[L], tau), w[L], true, bq);
                acc_add_point(a[L], bq, cf, dx[L], dy[L]);
            }
            for (int L = 0; L < cols; ++L) {
                for (int i = 0; i < 3; ++i) accd[i] += a[L].gs[i];
                for (int i = 0; i < 9; ++i) accd[3 + i] += a[L].gm[i];
                for (int i = 0; i < 3; ++i) accd[12 + i] += a[L].wa[i];
                accd[15] += a[L].ge[0]; accd[16] += a[L].ge[1];
            }
        }
        finalize_sample(S, g, accd, -(double)k * tau / (double)n, true, grad + 12 * b);
    }
    return 0;
}

}  // extern "C"
