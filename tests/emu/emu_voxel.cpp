// Host build of the fused voxel loss (sq_recovery_b200/csrc/sqloss.cu sq_voxel_loss) -- TEST TOOL, never part of the
// product.
//
// The loop of emu_occupancy_vjp (emu_occ_vjp.cpp) with explicit_column's VOX mode: the target voxel v takes the place of
// the upstream and of o_t (d = v - o_p, sq += d^2), the walk and the cut are the VJP's, every voxel outside the walked
// range adds v^2 (voxel_sq_outside, also for a column whose range is empty), and the finalize scale is sq_explicit_loss's.
// libm instead of MUFU.  tests/test_voxel_loss.py checks it against the oracle's autograd.
#include "sq_core.cuh"

using namespace sq;

static float g_bits = 0.f;       // > 0: cut at this many bits instead of kExplicitVjpBits (measuring the cut)

extern "C" {

void emu_voxel_set_bits(float bits) { g_bits = bits; }

// voxels: [B, n, n, n] fp32, index order [x][y][z]; loss: [B] mult * mean_vox (v - o)^2; grad: [B, 12] d loss[b] / d params[b]
int emu_voxel_loss(const double* params, int B, int n, double step, double z0, const float* voxels, float k, float mult,
                   double* loss, double* grad) {
    Grid g = make_grid(n, step, z0);
    const float kl = k * kLog2e, kact = g_bits > 0.f ? g_bits : kExplicitVjpBits, bound = cull_bound_bits(kl, kact);
    const double n3 = (double)n * n * n;
    for (int b = 0; b < B; ++b) {
        double p[12]; for (int i = 0; i < 12; ++i) p[i] = params[12 * b + i];
        SampleFull Sp; prep_sample(p, true, g, Sp);
        double accd[kAccN] = {0};
        double sq = 0.0;
        for (int ib = 0; ib < n; ++ib) for (int ia = 0; ia < n; ++ia) {
            float bhp[3], blp[3];
            column_base(Sp, g, ia, ib, bhp, blp);
            Acc a; acc_zero(a);
            const float dx = (float)(grid_coord(g, ia) - Sp.t[0]), dy = (float)(grid_coord(g, ib) - Sp.t[1]);
            Range rp;
            column_range(Sp, g, bound, bhp, rp.lo, rp.hi); warp_range(n, rp.lo, rp.hi);
            const float* col = voxels + (((size_t)b * n + ia) * n + ib) * n;
            if (rp.hi < rp.lo) { sq += voxel_sq_outside(col, n, rp, 1.0f); continue; }
            sq += explicit_column<true, true, true>(Sp, Sp, g, kl, bhp, blp, bhp, blp, Range{0, -1}, rp, dx, dy, a, col, kact);
            for (int i = 0; i < 3; ++i) accd[i] += a.gs[i];
            for (int i = 0; i < 9; ++i) accd[3 + i] += a.gm[i];
            for (int i = 0; i < 3; ++i) accd[12 + i] += a.wa[i];
            accd[15] += a.ge[0]; accd[16] += a.ge[1];
        }
        loss[b] = sq * (double)mult / n3;
        finalize_sample(Sp, g, accd, 2.0 * (double)k * (double)mult / n3, true, grad + 12 * b, (double)plane_of_t(Sp, g));
    }
    return 0;
}

}  // extern "C"
