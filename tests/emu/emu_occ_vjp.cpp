// Host build of the occupancy field's VJP (sq_recovery_b200/csrc/sqloss.cu sq_occupancy_vjp) -- TEST TOOL, never part of
// the product.
//
// The loop of emu_explicit (emu.cpp) with the things the VJP changes: the predicted SQ alone, walked over its own culled
// z range; every point weighted by the upstream voxel dL/d o[b, x, y, z] instead of (o_t - o_p), cut at kExplicitVjpBits;
// the z moment about plane_of_t(); the finalize scale is that of d o / d F alone, -k.  No loss.  explicit_column's VJP mode itself, so the loads and the
// weight are the kernel's; libm instead of MUFU.  tests/test_occupancy_vjp.py checks it against the oracle's autograd VJP.
#include "sq_core.cuh"

using namespace sq;

static float g_bits = 0.f;       // > 0: cut at this many bits instead of kExplicitVjpBits (measuring the cut)

extern "C" {

void emu_occ_set_bits(float bits) { g_bits = bits; }

// upstream: [B, n, n, n] fp32, index order [x][y][z]; grad: [B, 12]
int emu_occupancy_vjp(const double* params, int B, int n, double step, double z0, const float* upstream, float k,
                      double* grad) {
    Grid g = make_grid(n, step, z0);
    const float kl = k * kLog2e, kact = g_bits > 0.f ? g_bits : kExplicitVjpBits, bound = cull_bound_bits(kl, kact);
    for (int b = 0; b < B; ++b) {
        double p[12]; for (int i = 0; i < 12; ++i) p[i] = params[12 * b + i];
        SampleFull Sp; prep_sample(p, true, g, Sp);
        double accd[kAccN] = {0};
        for (int ib = 0; ib < n; ++ib) for (int ia = 0; ia < n; ++ia) {
            float bhp[3], blp[3];
            column_base(Sp, g, ia, ib, bhp, blp);
            Acc a; acc_zero(a);
            const float dx = (float)(grid_coord(g, ia) - Sp.t[0]), dy = (float)(grid_coord(g, ib) - Sp.t[1]);
            Range rp;
            column_range(Sp, g, bound, bhp, rp.lo, rp.hi); warp_range(n, rp.lo, rp.hi);
            const float* col = upstream + (((size_t)b * n + ia) * n + ib) * n;
            explicit_column<true, true>(Sp, Sp, g, kl, bhp, blp, bhp, blp, Range{0, -1}, rp, dx, dy, a, col, kact);
            for (int i = 0; i < 3; ++i) accd[i] += a.gs[i];
            for (int i = 0; i < 9; ++i) accd[3 + i] += a.gm[i];
            for (int i = 0; i < 3; ++i) accd[12 + i] += a.wa[i];
            accd[15] += a.ge[0]; accd[16] += a.ge[1];
        }
        finalize_sample(Sp, g, accd, -(double)k, true, grad + 12 * b, (double)plane_of_t(Sp, g));
    }
    return 0;
}

}  // extern "C"
