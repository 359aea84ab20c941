// Per-point core of the superquadric inside-outside losses (B200 / sm_100a).
//
// What the reference computes per sample and grid point (torch/classes.py:142-184, 236-274, 398-424, 322-351;
// torch/quaternion.py:19-21, 46-67), restated for one thread walking one grid column along z:
//
//   M = mat(conj(q)),  s = (M (g - t)) / a                       (a,e,t clamped; q NOT normalised)
//   A = |sx|^(2/e2)  B = |sy|^(2/e2)  C = |sz|^(2/e1)            (s == 0 -> |s| := 1e-2, the "A1 += 1e-4" fix-up)
//   D = A + B   E = D^(e2/e1)   G = E + C   F = G^e1
//
// Numeric plan (DESIGN.md "precision"): the affine geometry is formed in fp64 once per column and carried
// along z as a two-float (hi, lo) pair, so s has only its own final fp32 rounding; every pow is
// ex2(p * lg2(x)) on the MUFU pipe; all derivative factors are written as ratios bounded by 1
// (C/G, A/D, ...) so nothing overflows for points that carry gradient.
//
// Everything here is SQ_HD (host + device) on purpose: tests/emu compiles this same header with g++ to check
// the forward/backward algebra against the oracle on the CPU.  The product never runs the host build.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define SQ_HD __host__ __device__ __forceinline__
#else
#define SQ_HD inline
#endif

#if !defined(__CUDACC__)
struct float2 { float x, y; };          // host build (tests/emu)
#endif

#ifndef SQ_COUNT_HOOK
#define SQ_COUNT_HOOK(i, n) do { } while (0)
#endif

namespace sq {

constexpr float kLog2e = 1.4426950408889634f;
constexpr double kLn2 = 0.6931471805599453;
constexpr float kAbsFix = 1e-2f;          // |s| used when s == 0  (s^2 := 1e-4, classes.py:171-173)
#ifndef SQ_KACTIVE
#define SQ_KACTIVE 24.0f
#endif
constexpr float kActive = SQ_KACTIVE;     // |log2 of the sigmoid odds| beyond which o(1-o) < 2^-kActive is dropped (ImplicitLoss at
                                          // the training setting; implicit_active_bits() widens it for soft sigmoids)
// ExplicitLoss (k = 5) walks a wide soft shell: thousands of points per sample sit at 2^-24 .. 2^-32, and their sum shows
// at 0.2x the gradient tolerance (measured) -- it keeps the wider cut
constexpr float kActiveExplicit = 32.0f;

// ---------------------------------------------------------------- MUFU primitives
SQ_HD float ex2(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return exp2f(x);
#endif
}
SQ_HD float lg2(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return log2f(x);
#endif
}
SQ_HD float sqrt_approx(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return sqrtf(x);
#endif
}
SQ_HD float rcp(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
#else
    return 1.0f / x;
#endif
}

// lg2|x| and 2^-|x| with the sign handling folded into the MUFU operand (MUFU.LG2 |R|, MUFU.EX2 -|R|).  Written
// with the non-.ftz abs/neg so ptxas can fold them; the arithmetic fabsf() under -ftz costs an FADD on the FMA
// pipe, which the MUFU ops contend with (profiles/peaks_r01.json).
SQ_HD float lg2_abs(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("{\n .reg .f32 t;\n abs.f32 t, %1;\n lg2.approx.ftz.f32 %0, t;\n}" : "=f"(y) : "f"(x)); return y;
#else
    return log2f(fabsf(x));
#endif
}
SQ_HD float ex2_neg_abs(float x) {
#if defined(__CUDA_ARCH__)
    float y; asm("{\n .reg .f32 t;\n abs.f32 t, %1;\n neg.f32 t, t;\n ex2.approx.ftz.f32 %0, t;\n}" : "=f"(y) : "f"(x)); return y;
#else
    return exp2f(-fabsf(x));
#endif
}

// ---------------------------------------------------------------- grid
// Every grid the reference builds is uniform: arange(0, 1+1/R, 1/R) (classes.py:122-123) or linspace(0,1,R)
// (:218, :389), i.e. coordinate(i) = i*step, with coordinate 0 replaced by 1e-4 for Explicit/Implicit (:126,:221).
struct Grid {
    int n;          // points per axis
    double step;    // spacing
    double z0;      // coordinate of index 0 (1e-4 with the zero fix-up, else 0)
    float inv_n;    // 1 / n
    float stepf, z0f;
};
SQ_HD Grid make_grid(int n, double step, double z0) {
    Grid g; g.n = n; g.step = step; g.z0 = z0; g.inv_n = 1.0f / (float)n; g.stepf = (float)step; g.z0f = (float)z0; return g;
}
SQ_HD double grid_coord(const Grid& g, int i) { return i == 0 ? g.z0 : (double)i * g.step; }
SQ_HD float grid_coord_f32(const Grid& g, int i) { return i == 0 ? g.z0f : (float)i * g.stepf; }

// double <-> float conversions without the denormal fix-up code that -ftz=true attaches to a plain cast (a DSETP and a
// predicated FMUL per conversion; the values converted here are never denormal)
SQ_HD float d2f(double v) {
#if defined(__CUDA_ARCH__)
    float y; asm("cvt.rn.f32.f64 %0, %1;" : "=f"(y) : "d"(v)); return y;
#else
    return (float)v;
#endif
}
SQ_HD double f2d(float v) {
#if defined(__CUDA_ARCH__)
    double y; asm("cvt.f64.f32 %0, %1;" : "=d"(y) : "f"(v)); return y;
#else
    return (double)v;
#endif
}

// ---------------------------------------------------------------- per-sample constants
// `Sample` is what the column kernels keep per warp in shared memory; `SampleFull` (what prep writes to HBM) appends
// the fields only finalize and the fp64 IoU tie-break read.
struct Sample {
    // fp64 geometry: rows of M pre-divided by a_i, so s = Ms (g - t)
    double Ms[9];
    double t[3];
    // fp32 copy of the affine map (gx, gy) -> s at plane index 0, for culling and cost estimates (column_base_f32)
    float mf[6];              // Ms[i][0], Ms[i][1]
    float of[3];              // -(Ms t)_i
    // fp32 constants of the point loop
    float dh[3], dl[3];       // Ms[i][2] * step, split hi/lo: s_i(c) = base_i + d_i * cf(c)
    float idh[3];             // 1 / dh (+-inf when the column runs parallel to a face of the SQ's box)
    float cf0;                // z0 / step: the (non-integer) "index" of plane 0
    float pxy, pz;            // 2/e2, 2/e1
    float e21, e1;            // e2/e1, e1
    // ellipsoid that contains every level set of F (column_range): w (sx^2 + sy^2) + sz^2 <= qB1 * F
    float wd[3];              // w_i * dh_i,  w = (qw, qw, 1)
    float qw, qa, qia, qB1;   // 2^(e2-1), sum w_i dh_i^2, its reciprocal, 2^(1-e1)
    // Exact zeros along z (zero_planes()): 10 bits per coordinate i, the plane (>= 1) where s_i is EXACTLY 0 in the reference's
    // fp64 arithmetic for every column, 0 = none.  Non-zero only for an axis-aligned rotation with t on a grid plane.
    int zpack;
    // fp64 exponents for the refinement of gradient-carrying points (refined_point): 2/e2, 2/e1, e2/e1, e1
    double pxy64, pz64, e21_64, e1_64;
};
struct SampleFull : Sample {
    double M[9];              // un-scaled rotation
    double a[3], e[2], q[4];
    double ia[3];             // 1 / a
    // fused network heads (heads_forward): sigmoid outputs before the clamp, 1 / |raw quaternion|; heads = 0: not used
    double hp[8], hrn;
    int heads, pad2_;
    float mask[8];            // clamp sub-gradient masks for a(3), e(2), t(3): 1 inside or on the boundary, else 0
};

SQ_HD void split2(double v, float& hi, float& lo) { hi = d2f(v); lo = d2f(v - f2d(hi)); }

// The network heads of torch/models.py (SizeHead :52, ShapeHead :75, PositionHead :98: sigmoid; RotationHead :28: L2
// normalisation) and the torch.cat of train.py:89, applied to one row of raw head outputs [3 | 2 | 3 | 4].  The
// reference runs them in fp32, so the sigmoid / normalised values are rounded to fp32 before the loss sees them.
SQ_HD void heads_forward(const double* raw, double* p, double* hp, double& hrn) {
    for (int i = 0; i < 8; ++i) { hp[i] = (double)(float)(1.0 / (1.0 + exp(-raw[i]))); p[i] = hp[i]; }
    const double n2 = raw[8] * raw[8] + raw[9] * raw[9] + raw[10] * raw[10] + raw[11] * raw[11];
    hrn = 1.0 / sqrt(n2);
    for (int i = 8; i < 12; ++i) p[i] = (double)(float)(raw[i] * hrn);
}
// d loss / d raw from d loss / d params (gr, in place): sigmoid'(x) = p (1 - p); d (r / |r|) = (I - q q^T) / |r|
SQ_HD void heads_backward(const double* hp, double hrn, const double* q, double* gr) {
    for (int i = 0; i < 8; ++i) gr[i] *= hp[i] * (1.0 - hp[i]);
    const double dot = q[0] * gr[8] + q[1] * gr[9] + q[2] * gr[10] + q[3] * gr[11];
    for (int i = 0; i < 4; ++i) gr[8 + i] = (gr[8 + i] - q[i] * dot) * hrn;
}

// p: 12 raw parameters [a1 a2 a3 e1 e2 t1 t2 t3 qx qy qz qw].  clamp per classes.py:129-136 (IoU: no clamp, :398).
// prep_sample() in independent parts, so that the plan kernel can spread them over the lanes of a warp (the serial fp64
// chain of one lane was 2.5 us of the call): part 0..2 = row i of the scaled rotation and everything derived from it,
// part 3 = exponents and the power-mean weights, then prep_finish() once parts 0..3 are visible.
SQ_HD double clamped_param(const double* p, bool clamp, int i, float* mask = nullptr) {
    const double lo = i < 3 ? 0.05 : (i < 5 ? 0.1 : 0.0);     // a in [0.05, 1], e in [0.1, 1], t in [0, 1]  (classes.py:129-136)
    double x = p[i];
    float m = 1.0f;
    if (clamp) {
        if (x < lo) { x = lo; m = 0.0f; }
        if (x > 1.0) { x = 1.0; m = 0.0f; }
    }
    if (mask) *mask = m;
    return x;
}
SQ_HD void prep_part(const double* p, bool clamp, const Grid& g, SampleFull& S, int part) {
    if (part < 3) {
        const int i = part;
        // M = mat(conj(q)) = mat(q)^T   (quaternion.py:19-21, 46-67), row i
        const double x = -p[8], y = -p[9], z = -p[10], w = p[11];
        const double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
        const double twx = tx * w, twy = ty * w, twz = tz * w;
        const double txx = tx * x, txy = ty * x, txz = tz * x;
        const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
        double m0, m1, m2;
        if (i == 0)      { m0 = 1.0 - (tyy + tzz); m1 = txy - twz;         m2 = txz + twy; }
        else if (i == 1) { m0 = txy + twz;         m1 = 1.0 - (txx + tzz); m2 = tyz - twx; }
        else             { m0 = txz - twy;         m1 = tyz + twx;         m2 = 1.0 - (txx + tyy); }
        S.M[3 * i] = m0; S.M[3 * i + 1] = m1; S.M[3 * i + 2] = m2;
        const double a = clamped_param(p, clamp, i);
        const double t0 = clamped_param(p, clamp, 5), t1 = clamped_param(p, clamp, 6), t2 = clamped_param(p, clamp, 7);
        const double ia = 1.0 / a;
        S.ia[i] = ia;
        const double s0 = m0 * ia, s1 = m1 * ia, s2 = m2 * ia;
        S.Ms[3 * i] = s0; S.Ms[3 * i + 1] = s1; S.Ms[3 * i + 2] = s2;
        split2(s2 * g.step, S.dh[i], S.dl[i]);
        S.idh[i] = 1.0f / S.dh[i];
        S.mf[2 * i] = (float)s0; S.mf[2 * i + 1] = (float)s1;
        S.of[i] = (float)-(s0 * t0 + s1 * t1 + s2 * t2);
    } else {
        const double e1 = clamped_param(p, clamp, 3), e2 = clamped_param(p, clamp, 4);
        // Power-mean inequality, for exponents 2/e >= 2:  F >= 2^(e1-1) (2^(e2-1) (sx^2 + sy^2) + sz^2); the factors
        // are 1 for e > 1 (unclamped IoU parameters).  Non-positive e: no bound (the reference yields inf/nan there).
        const double w1 = e2 > 0.0 ? (e2 < 1.0 ? exp2(e2 - 1.0) : 1.0) : 0.0;
        const double b1 = e1 > 0.0 ? (e1 < 1.0 ? exp2(1.0 - e1) : 1.0) : 1e30;
        S.qw = (float)w1; S.qB1 = (float)b1;
        S.pxy64 = 2.0 / e2; S.pz64 = 2.0 / e1; S.e21_64 = e2 / e1; S.e1_64 = e1;
        S.pxy = (float)S.pxy64; S.pz = (float)S.pz64; S.e21 = (float)S.e21_64; S.e1 = (float)e1;
        S.cf0 = (float)(g.z0 / g.step);
    }
}
// The reference replaces an EXACT zero of s_i^2 by 1e-4 (classes.py:171-173).  Along x and y such zeros come out of the
// fp64 column base by themselves; along z the kernels evaluate s_i(c) = base_i + d_i c, which in general is never exactly
// 0.  An exact zero on a whole plane happens in the reference when row i of M has exact zeros in its x and y entries (an
// axis-aligned rotation: q = (0,0,0,1), half turns) and t_z sits exactly on a grid coordinate -- e.g. a position
// clamped to 1 (classes.py:135), the last coordinate of every grid.  Then s_i = (M_i2 g_z - M_i2 t_z) / a_i for every column
// (the reference's einsum adds exact zeros), and it vanishes where the two fp64 products agree.  Found by the fuzz
// (tests/tools/parity_fuzz_other.py): a plane of |s| = 1e-2 instead of ~1e-17 moved an e1 gradient by 2x the tolerance.
// Returns 10 bits per coordinate i: the plane c >= 1 where s_i is exactly 0, else 0.  (Plane 0 sits at 1e-4, classes.py:126,
// which no clamp produces.  Rows with TWO non-zero entries -- quarter turns, whose matrix keeps a 1e-16 -- have zeros
// that depend on the summation order of the reference's matmul: rounding noise, not reproduced.)
SQ_HD int zero_planes(const SampleFull& S, const Grid& g) {
    int pack = 0;
    for (int i = 0; i < 3; ++i) {
        if (S.M[3 * i] != 0.0 || S.M[3 * i + 1] != 0.0 || S.M[3 * i + 2] == 0.0) continue;
        const double m = S.M[3 * i + 2], target = m * S.t[2];
        const int c0 = (int)(S.t[2] / g.step + 0.5);
        for (int c = c0 - 1; c <= c0 + 1; ++c) {
            if (c < 1 || c >= g.n || c > 1023) continue;
            if (m * grid_coord(g, c) == target) pack |= c << (10 * i);
        }
    }
    return pack;
}
// The kernels get these zeros for free: every one of them evaluates s_i = fma(cf, dh_i, bh_i) + fma(cf, dl_i, bl_i).  For
// a row with a zero plane c*, d_i is re-split into two pieces of 13 significant bits (relative error 2^-26, better than
// one float), so that c* dh_i and c* dl_i are exact in fp32, and column_base() hands out bh_i = -c* dh_i, bl_i = -c* dl_i
// (the row does not depend on x, y): both FMAs return exactly 0 on plane c*, and d_i (c - c*) elsewhere.
SQ_HD float round13(float v) {
    int b;
#if defined(__CUDA_ARCH__)
    b = __float_as_int(v);
#else
    memcpy(&b, &v, 4);
#endif
    b = (b + 0x400) & ~0x7ff;
#if defined(__CUDA_ARCH__)
    return __int_as_float(b);
#else
    float r; memcpy(&r, &b, 4); return r;
#endif
}
SQ_HD void resplit_zero_rows(SampleFull& S, const Grid& g) {
    for (int i = 0; i < 3; ++i) {
        if (!((S.zpack >> (10 * i)) & 1023)) continue;
        const double d = S.Ms[3 * i + 2] * g.step;
        S.dh[i] = round13(d2f(d));
        S.dl[i] = round13(d2f(d - f2d(S.dh[i])));
        S.idh[i] = 1.0f / S.dh[i];
    }
}

SQ_HD void prep_finish(const double* p, bool clamp, const Grid& g, SampleFull& S) {
    for (int i = 0; i < 8; ++i) {
        float m;
        const double v = clamped_param(p, clamp, i, &m);
        S.mask[i] = m;
        if (i < 3) S.a[i] = v; else if (i < 5) S.e[i - 3] = v; else S.t[i - 5] = v;
    }
    for (int i = 0; i < 4; ++i) S.q[i] = p[8 + i];
    S.zpack = zero_planes(S, g);
    if (S.zpack) resplit_zero_rows(S, g);
    S.heads = 0; S.pad2_ = 0; S.hrn = 1.0;
    for (int i = 0; i < 8; ++i) S.hp[i] = 0.0;
    double al = 0.0;                                           // ellipsoid of column_range(): needs rows and qw
    for (int i = 0; i < 3; ++i) {
        const double wi = i < 2 ? (double)S.qw : 1.0, d = S.Ms[3 * i + 2] * g.step;
        S.wd[i] = (float)(wi * d);
        al += wi * d * d;
    }
    S.qa = (float)al; S.qia = (float)(1.0 / al);
}
SQ_HD void prep_sample(const double* p, bool clamp, const Grid& g, SampleFull& S) {
    for (int part = 0; part < 4; ++part) prep_part(p, clamp, g, S, part);
    prep_finish(p, clamp, g, S);
}

// s at plane "index" 0 for the column through grid point (ia, ib): base_i = Ms_i . ((gx,gy,0) - t), as hi/lo floats
SQ_HD void column_base(const Sample& S, const Grid& g, int ia, int ib, float* bh, float* bl, float* dxy = nullptr) {
    const double dx = grid_coord(g, ia) - S.t[0], dy = grid_coord(g, ib) - S.t[1], dz = -S.t[2];
    for (int i = 0; i < 3; ++i)
        split2(S.Ms[3 * i] * dx + S.Ms[3 * i + 1] * dy + S.Ms[3 * i + 2] * dz, bh[i], bl[i]);
    if (S.zpack)                                              // rows with a plane of exact zeros (zero_planes())
        for (int i = 0; i < 3; ++i) {
            const int cz = (S.zpack >> (10 * i)) & 1023;
            if (cz) { bh[i] = -(float)cz * S.dh[i]; bl[i] = -(float)cz * S.dl[i]; }
        }
    if (dxy) { dxy[0] = d2f(dx); dxy[1] = d2f(dy); }          // column position relative to t (for the M gradient)
}

// The same in plain fp32 (absolute error ~2e-6 for |s| <= 30): good enough to decide which planes can hold occupancy
// (column_range has 1e-3 of slack in the bound and a plane of slack per side), and 6 FMAs instead of 40 instructions
// of fp64 -- more than half of all warp column groups turn out empty and never need the exact base.
SQ_HD void column_base_f32(const Sample& S, const Grid& g, int ia, int ib, float* b) {
    const float gx = grid_coord_f32(g, ia), gy = grid_coord_f32(g, ib);
    for (int i = 0; i < 3; ++i) b[i] = fmaf(S.mf[2 * i], gx, fmaf(S.mf[2 * i + 1], gy, S.of[i]));
}

// ---------------------------------------------------------------- forward at one point
// The pow chain is evaluated in the log2 domain with the two sums done as log-sum-exp:
//   lA = (2/e2) lg2|sx|   lB = (2/e2) lg2|sy|   lC = (2/e1) lg2|sz|
//   lD = lg2(A + B) = max(lA, lB) + lg2(1 + 2^-|lA - lB|)
//   lE = (e2/e1) lD
//   lG = lg2(E + C) = max(lE, lC) + lg2(1 + 2^-|lE - lC|)
//   F  = 2^(e1 lG)
// Nothing under- or overflows before the last step (A = |s|^(2/e2) leaves fp32 range for |s| < 0.01 at e2 = 0.1,
// and such points DO carry gradient through E = D^(e2/e1) when e2/e1 is small), the ratios A/D, E/G needed by the
// backward come out of the same two exponentials, and it is 8 MUFU ops per F instead of the 10 of five pows.
struct Fwd {
    float sx, sy, sz;
    float d1, t1, h1;         // lA - lB, 2^-|d1|, lg2(1 + t1)
    float d2, t2, h2;         // lE - lC, 2^-|d2|, lg2(1 + t2)
    float lG, F;
};

template <bool FIX>
SQ_HD void point_forward(const Sample& S, float sx, float sy, float sz, Fwd& f) {
    f.sx = sx; f.sy = sy; f.sz = sz;
    float mx = sx, my = sy, mz = sz;
    if (FIX) {      // s == 0 exactly -> |s| := 1e-2 (the reference's "s^2 == 0 -> 1e-4")
        mx = (sx == 0.0f) ? kAbsFix : mx; my = (sy == 0.0f) ? kAbsFix : my; mz = (sz == 0.0f) ? kAbsFix : mz;
    }
    const float lA = S.pxy * lg2_abs(mx);
    const float lB = S.pxy * lg2_abs(my);
    const float lC = S.pz * lg2_abs(mz);
    f.d1 = lA - lB;
    f.t1 = ex2_neg_abs(f.d1);
    f.h1 = lg2(1.0f + f.t1);
    const float lE = S.e21 * (fmaxf(lA, lB) + f.h1);
    f.d2 = lE - lC;
    f.t2 = ex2_neg_abs(f.d2);
    f.h2 = lg2(1.0f + f.t2);
    f.lG = fmaxf(lE, lC) + f.h2;
    f.F = ex2(S.e1 * f.lG);
}

// occupancy o = sigmoid(k (1 - F)) = 1 / (1 + 2^(kl (F - 1))),  kl = k log2(e).   classes.py:187, :274
SQ_HD float occupancy(float F, float kl, float& odds_log2, float& eo) {
    odds_log2 = fmaf(F, kl, -kl);
    eo = ex2(odds_log2);
    return rcp(1.0f + eo);
}

// ---------------------------------------------------------------- backward at one point
// Derivative of F (times a caller weight W) with respect to the scaled coordinates s, the sizes and the shapes.
// With cG = C/G, eG = E/G, aD = A/D, bD = B/D (each pair sums to 1; the larger one is 1/(1+t), the smaller t/(1+t)):
//   dF/dsz = 2 F cG / sz        dF/dsx = 2 F eG aD / sx        dF/dsy = 2 F eG bD / sy
//   dF/da3 = -2 F cG / a3       dF/da1 = -2 F eG aD / a1       dF/da2 = -2 F eG bD / a2
//   dF/de1 = F ln2 (lG - cG lC - eG lE)    = F ln2 H2         H2 = h2 + min(cG, eG) |d2|   (no cancellation)
//   dF/de2 = F ln2 eG (lD - aD lA - bD lB) = F ln2 eG H1      H1 = h1 + min(aD, bD) |d1|
// The factors 2, ln2, 1/a_i are per-sample constants applied in finalize_sample().
struct Bwd {
    float gs[3];      // W F {eG aD/sx, eG bD/sy, cG/sz}
    float wa[3];      // W F {eG aD, eG bD, cG}
    float ge[2];      // W F H2,  W F eG H1
};

// Option SQ_MERGED_RCP: the five reciprocals (1 + t1, 1 + t2, sx, sy, sz) from ONE MUFU.RCP of their product plus 12 multiplications:
// on B200 a MUFU warp instruction costs ~6 issue cycles and an FMUL ~0.9 (profiles/peaks_r01.json), and the kernels are
// bound by instruction dispatch.  The product cannot leave fp32 range: 1 + t is in [1, 2], and of the three
// coordinates of a gradient-carrying point (F ~ 1) at most two are small, each at least ~1e-15 when not exactly 0.
// Measured: no gain for the implicit kernel, 2.5 % slower for the explicit one (longer dependent chain) -> off.
template <bool FIX = true>
SQ_HD void point_backward(const Fwd& f, float W, Bwd& b) {
    const float WF = W * f.F;
    float sx = f.sx, sy = f.sy, sz = f.sz;
    bool zx = false, zy = false, zz = false;
    if (FIX) {          // exact zeros: the fix-up replaces s^2 by a constant, so no gradient reaches s or a through that term
        zx = (sx == 0.0f); zy = (sy == 0.0f); zz = (sz == 0.0f);
        sx = zx ? 1.0f : sx; sy = zy ? 1.0f : sy; sz = zz ? 1.0f : sz;
    }
#ifdef SQ_MERGED_RCP
    const float p1 = 1.0f + f.t1, p2 = 1.0f + f.t2;
    const float pa = p1 * p2, pb = sx * sy, pc = pb * sz;
    const float inv = rcp(pa * pc);
    const float ia = inv * pc, ic = inv * pa;              // 1 / (p1 p2), 1 / (sx sy sz)
    const float r1 = ia * p2, r2 = ia * p1;
    const float ib = ic * sz;                              // 1 / (sx sy)
    const float isx = ib * sy, isy = ib * sx, isz = ic * pb;
#else
    const float r1 = rcp(1.0f + f.t1), r2 = rcp(1.0f + f.t2);
    const float isx = rcp(sx), isy = rcp(sy), isz = rcp(sz);
#endif
    const float s1 = f.t1 * r1, s2 = f.t2 * r2;
    const bool a_big = f.d1 >= 0.0f, e_big = f.d2 >= 0.0f;
    const float aD = a_big ? r1 : s1, bD = a_big ? s1 : r1;
    const float eG = e_big ? r2 : s2, cG = e_big ? s2 : r2;
    const float wz = WF * cG, wxy = WF * eG;
    const float wx = wxy * aD, wy = wxy * bD;
    b.ge[0] = WF * fmaf(s2, fabsf(f.d2), f.h2);
    b.ge[1] = wxy * fmaf(s1, fabsf(f.d1), f.h1);
    if (FIX) {
        b.wa[0] = zx ? 0.0f : wx;
        b.wa[1] = zy ? 0.0f : wy;
        b.wa[2] = zz ? 0.0f : wz;
        b.gs[0] = zx ? 0.0f : wx * isx;
        b.gs[1] = zy ? 0.0f : wy * isy;
        b.gs[2] = zz ? 0.0f : wz * isz;
    } else {            // the caller knows no coordinate of this column can be exactly 0 (column_zero_possible)
        b.wa[0] = wx; b.wa[1] = wy; b.wa[2] = wz;
        b.gs[0] = wx * isx;
        b.gs[1] = wy * isy;
        b.gs[2] = wz * isz;
    }
}

// a harmless point for lanes that carry no gradient but run the backward with their warp (weight 0)
SQ_HD void fwd_neutral(Fwd& f) {
    f.sx = f.sy = f.sz = 1.f;
    f.d1 = f.d2 = 0.f; f.t1 = f.t2 = 1.f; f.h1 = f.h2 = 1.f; f.lG = 0.f; f.F = 1.f;
}

// ---------------------------------------------------------------- fp64 refinement of gradient-carrying points
// At sigmoid sharpness k the gradient weight of a point is o (1 - o) with o = sigmoid(-x ln2), x = k log2(e) (F - 1): an
// error dF in F becomes 375 dF in x at k = 260 (torch/train.py:64, classes.py:274).  The fp32 chain above carries
// ~4e-7 (MUFU lg2 alone: 2e-7 absolute on each of up to three logarithms), i.e. dx ~ 1e-4, which is the whole gradient
// tolerance (rtol 1e-4).  So for the few points that carry the gradient -- |x| < kRefine, about a quarter of the points
// the compacted backward handles, ~0.4 % of the grid -- F - 1 is re-evaluated in fp64: geometry from the fp64 column
// base, log2 / exp2 from two small constant tables plus a short polynomial (1e-13 relative), F - 1 as expm1.  No MUFU
// approximation enters x; what the backward needs besides x (ratios bounded by 1, not amplified by k) is rounded to
// fp32 from the same chain.  B200 issues DFMA at half the FP32 rate on a pipe of its own (profiles/peaks_r01.json:
// 64 / clk / SM, co-issues with MUFU), so this costs ~150 instructions per refined point.
// Host and device run the same arithmetic (tests/emu), tables included.
#include "sq_tables.inc"
#if defined(__CUDACC__)
static __device__ const double kExp2TabDev[128] = {SQ_EXP2_TAB_VALUES};
static __device__ __align__(16) const double kLog2TabDev[256] = {SQ_LOG2_TAB_VALUES};
#endif
#if !defined(__CUDA_ARCH__)
static const double kExp2TabHost[128] = {SQ_EXP2_TAB_VALUES};
static const double kLog2TabHost[256] = {SQ_LOG2_TAB_VALUES};
#endif

SQ_HD int dbl_hi(double v) {
#if defined(__CUDA_ARCH__)
    return __double2hiint(v);
#else
    long long b; memcpy(&b, &v, 8); return (int)(b >> 32);
#endif
}
SQ_HD int dbl_lo(double v) {
#if defined(__CUDA_ARCH__)
    return __double2loint(v);
#else
    long long b; memcpy(&b, &v, 8); return (int)(b & 0xffffffffll);
#endif
}
SQ_HD double dbl_make(int hi, int lo) {
#if defined(__CUDA_ARCH__)
    return __hiloint2double(hi, lo);
#else
    const long long b = ((long long)hi << 32) | (long long)(unsigned int)lo; double v; memcpy(&v, &b, 8); return v;
#endif
}
// small int -> double without a conversion instruction (those share the MUFU pipe): 2^52 + 2^31 + k, minus the constant
SQ_HD double int_to_dbl(int k) { return dbl_make(0x43300000, k ^ (int)0x80000000) - 4503601774854144.0; }

// where the tables are read from: the constant arrays (host build; device: through L1), or a copy in shared memory
struct RefTabs { const double* e2; const double* l2; };
SQ_HD RefTabs default_tabs() {
#if defined(__CUDA_ARCH__)
    return RefTabs{kExp2TabDev, kLog2TabDev};
#else
    return RefTabs{kExp2TabHost, kLog2TabHost};
#endif
}

// 2^y for |y| <= 1000, relative error ~1e-15: y = q/128 + f, 2^y = 2^floor(q/128) * T[q mod 128] * exp(f ln2)
SQ_HD double exp2_acc(double y, const RefTabs& tb) {
    const double kMagic = 6755399441055744.0;                // 1.5 * 2^52: adding it leaves round(v) in the low word
    const double t = fma(y, 128.0, kMagic);
    const int q = dbl_lo(t);
    const double f = fma(t - kMagic, -0.0078125, y);         // y - q/128, |f| <= 1/256
    const int j = q & 127, k = q >> 7;
    const double z = f * kLn2, z2 = z * z;                  // exp(z) = (1 + z) + z^2 (1/2 + z/6) + z^4/24, shallow (latency)
    const double p = fma(z2 * z2, 1.0 / 24.0, fma(z2, fma(z, 1.0 / 6.0, 0.5), 1.0 + z));
    const double r = tb.e2[j] * p;
    return dbl_make(dbl_hi(r) + (k << 20), dbl_lo(r));       // times 2^k (the result stays a normal number)
}

// log2(m) for a positive normal m, absolute error ~1e-15 + 1e-16 |result|: m = 2^k f, f in [1,2) split at the midpoints
// c_j of 128 mantissa intervals: log2 m = k + log2 c_j + log1p(f / c_j - 1) / ln2
SQ_HD double log2_acc(double m, const RefTabs& tb) {
    const int hi = dbl_hi(m), lo = dbl_lo(m);
    const int k = ((hi >> 20) & 0x7ff) - 1023;
    const int j = (hi >> 13) & 127;
    const double f = dbl_make((hi & 0x000fffff) | 0x3ff00000, lo);
#if defined(__CUDA_ARCH__)
    const double2 tab = reinterpret_cast<const double2*>(tb.l2)[j];
    const double ic = tab.x, lc = tab.y;
#else
    const double ic = tb.l2[2 * j], lc = tb.l2[2 * j + 1];
#endif
    const double r = fma(f, ic, -1.0);                       // |r| < 1/250
    const double r2 = r * r;                                 // log1p(r) = r + r^2 (-1/2 + r/3) + r^4 (-1/4 + r/5), shallow
    const double p = fma(r2 * r2, fma(r, 0.2, -0.25), fma(r2, fma(r, 1.0 / 3.0, -0.5), r));
    return fma(p, 1.4426950408889634, lc + int_to_dbl(k));
}

#ifndef SQ_KREFINE
#define SQ_KREFINE 8.0f
#endif
constexpr float kRefine = SQ_KREFINE;     // |x| below which a gradient-carrying point is re-evaluated in fp64

// One point in fp64: s = base + cf d (d_i = Ms[i][2] step), the forward chain of point_forward() and x = kl (F - 1).
#ifdef SQ_REFINE_NOINLINE
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
#else
SQ_HD
#endif
float refined_x(const Sample& S, double step, float kl, double b0, double b1, double b2, float cf, const RefTabs& tb) {
    const double c = f2d(cf);
    double s0 = fma(c, S.Ms[2] * step, b0), s1 = fma(c, S.Ms[5] * step, b1), s2 = fma(c, S.Ms[8] * step, b2);
    if (S.zpack) {                                            // planes of exact zeros (zero_planes()): cf is an exact integer there
        const int pc = cf < 1.0f ? -1 : (int)cf;          // plane 0 (cf = cf0 < 1) never is one
        if ((S.zpack & 1023) == pc) s0 = 0.0;
        if (((S.zpack >> 10) & 1023) == pc) s1 = 0.0;
        if (((S.zpack >> 20) & 1023) == pc) s2 = 0.0;
    }
    const double a0 = s0 == 0.0 ? 1e-2 : fabs(s0), a1 = s1 == 0.0 ? 1e-2 : fabs(s1), a2 = s2 == 0.0 ? 1e-2 : fabs(s2);
    const double lA = S.pxy64 * log2_acc(a0, tb), lB = S.pxy64 * log2_acc(a1, tb), lC = S.pz64 * log2_acc(a2, tb);
    const double t1 = exp2_acc(-fmin(fabs(lA - lB), 64.0), tb);
    const double lE = S.e21_64 * (fmax(lA, lB) + log2_acc(1.0 + t1, tb));
    const double t2 = exp2_acc(-fmin(fabs(lE - lC), 64.0), tb);
    const double y = S.e1_64 * (fmax(lE, lC) + log2_acc(1.0 + t2, tb));
    double Fm1;                                               // F - 1 = 2^y - 1
    if (fabs(y) < 0.0625) {
        const double z = y * kLn2;                            // |z| < 0.044: the series is exact to 1e-16 after z^7
        const double z2 = z * z, z4 = z2 * z2;
        const double hi = fma(z2, 1.0 / 5040.0, fma(z, 1.0 / 720.0, 1.0 / 120.0));          // z^4 .. z^6 terms
        const double lo = fma(z2, fma(z, 1.0 / 24.0, 1.0 / 6.0), fma(z, 0.5, 1.0));          // 1 .. z^3 terms
        Fm1 = z * fma(z4, hi, lo);
    } else {
        Fm1 = exp2_acc(fmin(fmax(y, -1000.0), 1000.0), tb) - 1.0;
    }
    return d2f(f2d(kl) * Fm1);
}

// ---------------------------------------------------------------- per-thread accumulators
// Sums over the points a thread visits (all columns of one sample), in the units finalize_sample() expects.
struct Acc {
    float gs[3];      // sum gs_i
    float gm[9];      // sum gs_i * (g_j - t_j)  for j = x, y;  sum gs_i * cf for j = z   (row-major i, j)
    float wa[3];
    float ge[2];
    float loss;
};
constexpr int kAccN = 18;
SQ_HD void acc_zero(Acc& a) {
    for (int i = 0; i < 3; ++i) { a.gs[i] = 0.f; a.wa[i] = 0.f; }
    for (int i = 0; i < 9; ++i) a.gm[i] = 0.f;
    a.ge[0] = a.ge[1] = 0.f; a.loss = 0.f;
}

// ---------------------------------------------------------------- finalize: partial sums -> d loss / d params
// acc: the 18 sums over all points of one sample (fp64).  scale = d loss / d (weighted sum of F) constant, i.e.
// the product of every per-sample constant factor the point loop left out except 2, ln2, 1/a, step.
//   grad wrt t_j  = -sum_i Ms_ij gs_i
//   grad wrt M_ij = (1/a_i) sum gs_i (g_j - t_j)
//   grad wrt q    = sum_ij dM_ij/dq * grad M_ij,  M = mat(conj(q))
// z_is_index: the z moment gm[i][2] holds sum gs_i * cf (grid index units, column kernels) instead of
// sum gs_i * (z - t_z) (point-list kernel).
// z_centre (z_is_index only): the z moment holds sum gs_i * (cf - z_centre) instead (explicit_column's VJP mode: plane_of_t()).
SQ_HD void finalize_sample(const SampleFull& S, const Grid& g, const double* acc, double scale, bool z_is_index,
                           double* grad12, double z_centre = 0.0) {
    const double tz = z_centre != 0.0 ? S.t[2] - g.step * z_centre : S.t[2];
    const double* gs = acc; const double* gm = acc + 3; const double* wa = acc + 12; const double* ge = acc + 15;
    double gM[9];
    for (int i = 0; i < 3; ++i) {
        const double ia = S.ia[i];
        gM[3 * i + 0] = 2.0 * ia * gm[3 * i + 0];
        gM[3 * i + 1] = 2.0 * ia * gm[3 * i + 1];
        gM[3 * i + 2] = 2.0 * ia * (z_is_index ? g.step * gm[3 * i + 2] - tz * gs[i] : gm[3 * i + 2]);
    }
    for (int i = 0; i < 3; ++i) grad12[i] = -2.0 * wa[i] * S.ia[i] * S.mask[i] * scale;
    grad12[3] = kLn2 * ge[0] * S.mask[3] * scale;
    grad12[4] = kLn2 * ge[1] * S.mask[4] * scale;
    for (int j = 0; j < 3; ++j) {
        double s = 0.0;
        for (int i = 0; i < 3; ++i) s += S.Ms[3 * i + j] * gs[i];
        grad12[5 + j] = -2.0 * s * S.mask[5 + j] * scale;
    }
    // M = mat(conj(q)):  M00=1-2(y2+z2) M01=2xy+2zw M02=2xz-2yw / M10=2xy-2zw M11=1-2(x2+z2) M12=2yz+2xw /
    //                    M20=2xz+2yw M21=2yz-2xw M22=1-2(x2+y2)
    const double x = S.q[0], y = S.q[1], z = S.q[2], w = S.q[3];
    const double g00 = gM[0], g01 = gM[1], g02 = gM[2], g10 = gM[3], g11 = gM[4], g12 = gM[5],
                 g20 = gM[6], g21 = gM[7], g22 = gM[8];
    grad12[8]  = scale * 2.0 * (y * (g01 + g10) + z * (g02 + g20) + w * (g12 - g21) - 2.0 * x * (g11 + g22));
    grad12[9]  = scale * 2.0 * (x * (g01 + g10) + z * (g12 + g21) + w * (g20 - g02) - 2.0 * y * (g00 + g22));
    grad12[10] = scale * 2.0 * (x * (g02 + g20) + y * (g12 + g21) + w * (g01 - g10) - 2.0 * z * (g00 + g11));
    grad12[11] = scale * 2.0 * (z * (g01 - g10) + y * (g20 - g02) + x * (g12 - g21));
}

// ---------------------------------------------------------------- culling
// F >= max(sx^2, sy^2, sz^2) for every shape (G >= C and G >= E >= A^(e2/e1), ...), so a point with
// max |s_i| >= bound(bits) has kl (F - 1) >= bits, i.e. occupancy o = 1/(1 + 2^(kl (F-1))) < 2^-bits.  A column only
// has to be walked over the z range where it can be inside the box |s_i| < bound; the rest is accounted for in closed
// form with o = 0.
//   bits = 128: 2^that overflows and o is 0 EXACTLY in this kernel's own fp32 arithmetic -- culling changes nothing.
//   bits = 32 (ImplicitLoss, kImplicitCullBits; 40 until round 2): the dropped occupancies sum to < n 2^-32 = 1.5e-8 per
//   column, below the fp32 resolution of cs wherever cs matters (cs > 1e-7 is needed for a depth above 1e-16); their
//   gradient weight o (1 - o) < 2^-32 is below the 2^-kact cut the backward applies anyway.  The box edge shrinks from
//   1.159 (bits = 128) to 1.042 at k = 260: a quarter fewer points to evaluate.
SQ_HD float cull_bound(float kl) { return sqrtf((1.0f + 128.0f / kl) * 1.002f); }
#ifndef SQ_IMPLICIT_CULL_BITS
#define SQ_IMPLICIT_CULL_BITS 32.0f
#endif
constexpr float kImplicitCullBits = SQ_IMPLICIT_CULL_BITS;

// ExplicitLoss has sharpness 5, for which the exact bound is |s| >= 4.3 and culls nothing.  Its terms are differences
// (o_t - o_p)^2 of numbers in [0,1] accumulated in fp32, so an occupancy below 2^-24 is below the resolution of the
// difference whenever the other one matters, and contributes < 2^-48 when both are that small.  Outside
// |s_i| < bound24 the occupancy is < 2^-24 and is taken as 0 (DESIGN.md "culling").
SQ_HD float cull_bound_bits(float kl, float bits) { return sqrtf((1.0f + bits / kl) * 1.002f); }
SQ_HD float implicit_cull_bound(float kl) { return cull_bound_bits(kl, kImplicitCullBits); }

// The VJP of the occupancy field (sq_occupancy_vjp) drops every point whose weight o (1 - o) is below 2^-bits: it culls the
// walk at that level and cuts the backward there too.  Unlike the loss, whose upstream (o_p - o_t) vanishes where both
// occupancies are tiny, an upstream can be large and of one sign over the whole soft shell (d sum(o) / d theta: the soft
// volume), so what is dropped adds up coherently.  Per unit of grid volume that is
//   sum_{x > bits} k 2^-x |dF/dtheta| dV  ~  2^-bits |dF/dtheta| dV/dF   (one octave of o (1 - o) spans ln2 / k in F)
// at F_cut = 1 + bits ln2 / k, against the per-sample tolerance 5e-9 n^3 max|upstream|, i.e. 5e-9 per unit volume: the
// grid size drops out and bits depends on k alone.  Measured at k = 5 on the host build (tests/emu/emu_occ_vjp.cpp, the
// random goldens at R = 8..64, edge, pred24, zero planes), worst entry in units of the tolerance for the upstream +1 on
// the shell o (1 - o) in [2^-34, 2^-20] -- one sign, all of it below the loss path's 2^-24:
//   cut at 24 bits: 26..63    28: 1.5..5.6    32: 0.07..0.15    34 and beyond: < 1e-3 (the whole shell kept)
// i.e. the dropped sum shrinks ~16x per 4 bits; at 36 bits what lies beyond the cut is ~1/100 of the tolerance for any
// upstream.  (The constant upstream is not limited by the cut: from 28 bits on its error is the fp32 floor of the sums.)
// A sharper sigmoid needs fewer bits (F_cut closer to 1), so 36 is conservative for k >= 5.
constexpr float kExplicitVjpBits = 36.0f;

// The box is loose for round shapes (for an ellipsoid it has twice the volume of the level set).  Second bound, from
// the power-mean inequality (exponents 2/e >= 2):
//   F >= 2^(e1-1) (2^(e2-1) (sx^2 + sy^2) + sz^2)
// so F < bound^2 also confines the point to the ellipsoid  w (sx^2 + sy^2) + sz^2 < bound^2 2^(1-e1), whose
// intersection with the column is the root interval of a quadratic in the plane index.  Box and ellipsoid together
// leave 15 % fewer planes to walk on BASELINE config 2 (exact level-set ranges would leave 29 % fewer).
#ifndef SQ_NO_QUADRIC
#define SQ_QUADRIC 1
#endif

// inclusive z-index range [c_lo, c_hi] outside which F >= bound^2; empty when c_hi < c_lo
SQ_HD void column_range(const Sample& S, const Grid& g, float bound, const float* bh, int& c_lo, int& c_hi) {
    float lo = -1e30f, hi = 1e30f;
    for (int i = 0; i < 3; ++i) {
        const float u = (bound - bh[i]) * S.idh[i], v = (-bound - bh[i]) * S.idh[i];
        lo = fmaxf(lo, fminf(u, v));       // fminf/fmaxf drop the NaN of 0 * inf
        hi = fminf(hi, fmaxf(u, v));
    }
#ifdef SQ_QUADRIC
    {
        // alpha c^2 + 2 beta c + gamma < 0 with s(c) = bh + c dh; 0.4 % of slack on the radius^2 on top of the 0.2 % in
        // `bound` covers the fp32 evaluation (|bh| <= ~30: relative 1e-6 on the discriminant)
        const float qB = bound * bound * 1.004f * S.qB1;
        const float beta = fmaf(S.wd[0], bh[0], fmaf(S.wd[1], bh[1], S.wd[2] * bh[2]));
        const float gamma = fmaf(S.qw, fmaf(bh[0], bh[0], bh[1] * bh[1]), fmaf(bh[2], bh[2], -qB));
        const float disc = fmaf(beta, beta, -S.qa * gamma);
        const float sq = sqrt_approx(fmaxf(disc, 0.0f));
        const float u = (-beta - sq) * S.qia, v = (sq - beta) * S.qia;
        lo = fmaxf(lo, u);
        hi = fminf(hi, disc > 0.0f ? v : -1e30f);           // no real roots: the column misses the ellipsoid
    }
#endif
    // one plane of slack per side: rounding of the bounds, the lo parts of s, and plane 0 sitting at z0 not 0
    const float nf = (float)g.n;
    lo = fminf(fmaxf(lo - 1.0f, 0.0f), nf);
    hi = fmaxf(fminf(hi + 1.0f, nf - 1.0f), -1.0f);
    c_lo = (int)ceilf(lo);
    c_hi = (int)floorf(hi);
}

// Upper bound on the z planes ANY column of a rectangular footprint (centre (cx, cy), half extents (hx, hy), in grid
// steps) can need: the bounds of column_range() evaluated once at the centre, widened by how far s can move across the
// footprint (so a thin object that slips between probe columns is never taken for empty).  0 is a PROOF that every
// column of the footprint has an empty range -- the plan kernel relies on it to drop work items for good
// (tests/test_emu_math.py checks the claim against the fp64 F).
SQ_HD int footprint_planes(const Sample& S, const Grid& g, float bound, float cx, float cy, float hx, float hy, int* range_lo = nullptr) {
    const float gx = cx * g.stepf, gy = cy * g.stepf;
    float lo = -1e30f, hi = 1e30f, he2 = 0.f, bc[3];
    for (int i = 0; i < 3; ++i) {
        bc[i] = fmaf(S.mf[2 * i], gx, fmaf(S.mf[2 * i + 1], gy, S.of[i]));
        // + the 0 -> z0 substitution of grid index 0, + 1 % and 1e-4 for the fp32 evaluation here and in the kernels
        const float hw = ((fabsf(S.mf[2 * i]) * hx + fabsf(S.mf[2 * i + 1]) * hy) * g.stepf
                          + (fabsf(S.mf[2 * i]) + fabsf(S.mf[2 * i + 1])) * fabsf(g.z0f)) * 1.01f + 1e-4f;
        const float bi = bound + hw;
        const float u = (bi - bc[i]) * S.idh[i], v = (-bi - bc[i]) * S.idh[i];
        lo = fmaxf(lo, fminf(u, v));
        hi = fminf(hi, fmaxf(u, v));
        he2 = fmaf(i < 2 ? S.qw : 1.0f, hw * hw, he2);
    }
    {
        const float r = sqrtf(bound * bound * 1.004f * S.qB1) + sqrtf(he2);
        const float beta = fmaf(S.wd[0], bc[0], fmaf(S.wd[1], bc[1], S.wd[2] * bc[2]));
        const float gamma = fmaf(S.qw, fmaf(bc[0], bc[0], bc[1] * bc[1]), fmaf(bc[2], bc[2], -r * r));
        const float disc = fmaf(beta, beta, -S.qa * gamma);
        const float sq = sqrtf(fmaxf(disc, 0.0f));
        lo = fmaxf(lo, (-beta - sq) * S.qia);
        hi = fminf(hi, disc > 0.0f ? (sq - beta) * S.qia : -1e30f);
    }
    const float nf = (float)g.n;
    lo = fminf(fmaxf(lo - 1.0f, 0.0f), nf);
    hi = fmaxf(fminf(hi + 1.0f, nf - 1.0f), -1.0f);
    const int c_lo = (int)ceilf(lo), c_hi = (int)floorf(hi);
    if (range_lo) *range_lo = c_lo;
    return c_hi >= c_lo ? c_hi - c_lo + 1 : 0;
}

// How many of those planes an ImplicitLoss walk really visits.  The walk comes from high z and a lane is finished once its
// transmittance is below 2^-32, i.e. `die` = 32 / (tau log2 e) planes of full occupancy after it entered the object; the
// warp stops when its last lane has.  The unit ball |s|_2 <= 1 lies inside every superquadric with exponents 2/e >= 2
// (|.|_p <= |.|_2), so a column whose chord through the ball |s|^2 <= 0.97 (occupancy > 0.99 at any sharpness >= 200; an
// estimate, like everything here) is at least `die` planes long is finished `die` planes behind the chord's near end.
// Chord length and near end are concave over the footprint (a convex body), so the four corner columns decide: if all
// of them go opaque, every column between them does, and the walk ends at the lowest of their stopping planes; a group
// on the silhouette keeps walking to the end of its range.  Objects that fill the grid (bench.py's `dense` workload) have
// the same plane count in nearly every group, but real walks from 15 planes (interior) to all of them (silhouette): by plane
// count alone the order was random there and the end-game 30 % of the launch (profiles/item_costs_r02.txt).
SQ_HD int footprint_walk(const Sample& S, const Grid& g, float bound, float die, float cx, float cy, float hx, float hy) {
    int c_lo = 0;
    const int planes = footprint_planes(S, g, bound, cx, cy, hx, hy, &c_lo);
    if (planes <= 0 || !(die > 0.f)) return planes;
    const float a = fmaf(S.dh[0], S.dh[0], fmaf(S.dh[1], S.dh[1], S.dh[2] * S.dh[2])), ia = 1.0f / a, nf = (float)(g.n - 1);
    float stop = 1e30f;
    for (int k = 0; k < 4; ++k) {
        const float gx = (cx + ((k & 1) ? hx : -hx)) * g.stepf, gy = (cy + ((k & 2) ? hy : -hy)) * g.stepf;
        float b[3];
        for (int i = 0; i < 3; ++i) b[i] = fmaf(S.mf[2 * i], gx, fmaf(S.mf[2 * i + 1], gy, S.of[i]));
        const float beta = fmaf(S.dh[0], b[0], fmaf(S.dh[1], b[1], S.dh[2] * b[2]));
        const float gamma = fmaf(b[0], b[0], fmaf(b[1], b[1], fmaf(b[2], b[2], -0.97f)));
        const float disc = fmaf(beta, beta, -a * gamma);
        float s = (float)c_lo;                                        // not opaque: walks to the end of the range
        if (disc > 0.f) {
            const float sq = sqrtf(disc);
            const float far_ = fmaxf((-beta - sq) * ia, 0.f), near_ = fminf((sq - beta) * ia, nf);
            if (near_ - far_ >= die) s = fmaxf(near_ - die - 1.0f, (float)c_lo);
        }
        stop = fminf(stop, s);
    }
    const int cut = (int)(stop - (float)c_lo);
    return cut > 0 ? (planes - cut > 1 ? planes - cut : 1) : planes;
}

// Footprint (centre and half extents, in grid steps) of the 32-slot column group `group` in the x-fastest layout used
// when n is not a multiple of 8: slots [32 group, 32 group + 31] of the n*n columns, slot = ib * n + ia.  For n < 32 a
// group spans up to ceil(32 / n) + 1 rows, so the row span is computed, not assumed.
SQ_HD void xfast_group_footprint(int n, int group, float& cx, float& cy, float& hx, float& hy) {
    const int first = group * 32;
    int last = first + 31;
    if (last > n * n - 1) last = n * n - 1;
    const int ib0 = first / n, ia0 = first - ib0 * n, ib1 = last / n, ia1 = last - ib1 * n;
    if (ib1 == ib0) { cx = 0.5f * (float)(ia0 + ia1); hx = 0.5f * (float)(ia1 - ia0); cy = (float)ib0; hy = 0.f; }
    else { cx = 0.5f * (float)(n - 1); hx = cx; cy = 0.5f * (float)(ib0 + ib1); hy = 0.5f * (float)(ib1 - ib0); }
}

#if defined(__CUDA_ARCH__)
#define SQ_ANY(p) __any_sync(0xffffffffu, (p))
#define SQ_BALLOT(p) __ballot_sync(0xffffffffu, (p))
#define SQ_WARP_MAX(v) __reduce_max_sync(0xffffffffu, (v))
#define SQ_WARP_MIN(v) __reduce_min_sync(0xffffffffu, (v))
#else
#define SQ_ANY(p) (p)
#define SQ_BALLOT(p) ((p) ? 1u : 0u)          // host build: a "warp" of one lane
#define SQ_WARP_MAX(v) (v)
#define SQ_WARP_MIN(v) (v)
#endif
// bits of the lanes below this one (host build: none)
SQ_HD unsigned lanes_below() {
#if defined(__CUDA_ARCH__)
    unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m;
#else
    return 0u;
#endif
}
SQ_HD int popcount(unsigned m) {
#if defined(__CUDA_ARCH__)
    return __popc(m);
#else
    return __builtin_popcount(m);
#endif
}

// union over the warp of the lanes' ranges; (0, -1) when every lane's range is empty
SQ_HD void warp_range(int n, int& c_lo, int& c_hi) {
    const bool empty = c_hi < c_lo;
    c_hi = SQ_WARP_MAX(empty ? -1 : c_hi);
    c_lo = SQ_WARP_MIN(empty ? n : c_lo);
    if (c_hi < c_lo) { c_lo = 0; c_hi = -1; }
}

// Can a scaled coordinate of this column be EXACTLY 0 on some plane?  s_i(c) = (bh_i + c dh_i) + (bl_i + c dl_i)
// vanishes only where the hi part does to within the (2^-24 relative) lo part, i.e. at a plane index within ~1e-5 of
// c* = -bh_i / dh_i.  Conservative (NaN/inf from dh_i = 0 count as "possible"); true for ~1e-3 of random columns.
// Columns for which this is false skip the three "s == 0 -> |s| := 1e-2" selects per plane and the six in the backward.
SQ_HD bool column_zero_possible(const Sample& S, const float* bh) {
    bool m = false;
    for (int i = 0; i < 3; ++i) {
        const float cs = -bh[i] * S.idh[i];
        const float r = cs - rintf(cs);
        m = m || !(fabsf(r) > 1e-4f) || !(fabsf(cs - S.cf0) > 1e-4f);
    }
    return m;
}

// ---------------------------------------------------------------- ImplicitLoss: one column
// classes.py:274-279.  Walk from the camera side (z index n-1) down to 0:
//   o_c = sigmoid(k (1 - F_c)),  cs_c = running sum of o,  T_c = exp(-tau cs_c),  depth = 1 - sum_c T_c / n.
// d depth / d o_c = (tau/n) S_c with the suffix sum S_c = sum_{c' at or behind c} T_c'.  S_c is only known at the
// end of the walk, so gradient terms are accumulated twice -- sum x and sum P_c x with P_c the sum of T in front
// of c -- and combined as U sum x - sum P x when the column ends.  P and U start at the first point that carries
// gradient, which keeps the subtraction well conditioned.
struct ImplicitParams { float kl; float tl; float bound; float kact; };   // k log2(e), tau log2(e), implicit_cull_bound(kl),
                                                                          // implicit_active_bits(kl, n, batch)
// The backward drops points whose weight o (1 - o) is below 2^-kact.  Two things decide how small that has to be:
//  * what is dropped adds up over the band of points between the cut and the culling bound, and the band is as thick as the
//    sigmoid is soft: (32 - kact) / kl in F, i.e. at most a point per column at k = 260 but tens at k = 20, more on finer
//    grids -- found by the fuzz: k = 20 on a 96^3 grid was 1.1x the tolerance off with a fixed 24, 0.1x with 28.3;
//  * one dropped point moves the gradient of the MEAN loss by up to 2^-kact kl |dF/dtheta| / (n^2 batch), which has to stay well
//    below the ABSOLUTE tolerance 1e-6: on a 12^3 grid with three samples a 2^-24 point is 3e-7 (fuzz: 0.94x at k = 500).
// kact = 24 at the reference's training setting (k = 260, 64 planes, batches of 8 and more: the dropped sum is 0.03x the
// tolerance), more where either rule asks for it, up to the culling bound's 32.
SQ_HD float implicit_active_bits(float kl, int n, int batch) {
    const float band = (260.0f * kLog2e / kl) * ((float)n / 64.0f);
    float bits = kActive + (band > 1.0f ? log2f(band) : 0.0f);
    const float point = log2f(kl * 1e9f / ((float)n * (float)n * (float)(batch > 0 ? batch : 1)));     // 2^-bits kl 10 / (n^2 B) <= 1e-8
    if (point > bits) bits = point;
    return bits < kImplicitCullBits ? bits : kImplicitCullBits;
}

#ifndef SQ_KDEEP
#define SQ_KDEEP 32.0f
#endif
constexpr float kDeep = SQ_KDEEP;       // points behind 2^-kDeep of transmittance carry no gradient (S_c < n 2^-kDeep)

struct ColGrad {       // two-moment accumulators of one column
    float gs0[3], gs1[3], gz0[3], gz1[3], ge0[2], ge1[2];
};

// Returns the rendered depth.  1 - sum T / n cannot resolve depths below ~1e-7 in fp32, but the sign of
// (depth - target) on silhouette pixels (target exactly 0, depth 1e-16..1e-7 in the fp64 reference) decides whether
// the column's gradient counts, and those columns carry k-amplified gradient.  So the first-order sum
// (tau/n) sum_c cs_c is carried along and used when the depth is tiny (relative error < 0.4% there).
// [c_lo, c_hi]: the (warp-uniform) z range to walk, from column_range() / warp_range().
// running state of one column walk
// The warp's pool of gradient-carrying points (SQ_BWD_COMPACT), structure of arrays, `cap` slots shared by the warp's 32
// columns.  During the walk the lanes whose point carries gradient append to it together (two ballots per plane that has
// any): points near the surface (|x| < kRefine, re-evaluated in fp64 later) fill the pool from the FRONT, the others from the
// BACK, so after the walk the two lists are already compact -- entries [0, nr) and (top, cap - 1] -- and are dealt out to the
// lanes by index: no per-lane counts, no scan, no index list.  A column that grazes the surface for dozens of planes simply
// takes more of the pool (it was a 15-deep queue per lane until round 2's last third; columns with more gradient points than
// that fell back to the unrefined on-the-spot path -- the one parity outlier of the fuzz).  Only when a whole plane's new
// points do not fit any more (more than `cap` gradient points in one 32-column group, or more than 255 of them near the
// surface) do those points take the on-the-spot path.
//
// An entry's plane index is a small integer in a float (or cf0 < 1 for plane 0): its low 13 mantissa bits are free and carry
// the lane of the entry's column (5 bits) and, for front entries, the previous front entry of the same column (8 bits,
// kNoLink = none) -- the chain queue_suffix_weight() follows.  Grids beyond 1024 planes, or whose plane 0 sits a whole step or
// more from the origin (cf0 >= 1: not a grid the reference's classes build), get no pool (cap = 0).
struct BwdQueue {
    float* cf;       // plane "index" of the point | tag (entry_cf / entry_lane / entry_link)
    float* pre;      // sum of T in front of it since its column's first gradient-carrying point
    float* x;        // the weight o (1 - o) = eo o^2 of the point; for front entries the log2 odds x = k log2(e) (F - 1)
                     // the scan used, replaced by the weight at the fp64-refined x in queue_refine_entry()
    float* d;        // front entries: occupancy correction o(x refined) - o(x scan)
    int cap;         // slots (kernels: kBwdPool; host build: settable, to exercise the overflow path)
    int lane;        // this thread's lane (host build: the column's slot in its group of 32)
    unsigned where;  // kernels: shared-memory address of cf[0] (32-byte aligned; pre, x, d follow at kBwdPool floats each) | lane
};
constexpr int kNoLink = 255;
constexpr unsigned kTagMask = 0x1fffu;
constexpr int kPoolMaxPlanes = 1024;

SQ_HD unsigned f32_bits(float v) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(v);
#else
    unsigned u; memcpy(&u, &v, 4); return u;
#endif
}
SQ_HD float bits_f32(unsigned u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float v; memcpy(&v, &u, 4); return v;
#endif
}
SQ_HD float entry_cf(const Sample& S, float tagged) {
    const float cf = bits_f32(f32_bits(tagged) & ~kTagMask);
    return cf < 1.0f ? S.cf0 : cf;                       // plane 0: cf0 is not an integer, its low bits were not free
}
SQ_HD int entry_lane(float tagged) { return (int)(f32_bits(tagged) & 31u); }
SQ_HD int entry_link(float tagged) { return (int)((f32_bits(tagged) >> 5) & 255u); }

struct ColState {
    float csl, cssum, tsum, psh, seen, T;
    // SQ_BWD_COMPACT: the warp's pool, front entries so far and the next free back slot (both warp-uniform), this column's
    // latest front entry, whether a point of this column had to be handled on the spot because the pool was full
    BwdQueue q;
    int nr, top, head;
    bool spilled;
};

// SQ_BWD_COMPACT.  The backward block runs for the whole warp as soon as ONE lane carries gradient, and the surface
// crosses the 32 columns of a patch on different planes: 5.7 of 32 lanes do on average (tools/timeline.py).  So during
// the walk a gradient-carrying lane only notes (plane, prefix of T) in the warp's shared-memory pool; after the walk --
// when the column's suffix weight U and the sign of (depth - target) are known -- the pooled points of all 32 columns
// are dealt out evenly to the lanes, which redo the forward for their point and run the backward once, weighted,
// straight into the item's sums.  Points that find the pool full fall back to the on-the-spot two-moment path.
#if !defined(SQ_NO_BWD_COMPACT) && !defined(SQ_BWD_COMPACT)
#define SQ_BWD_COMPACT 1
#endif
#ifndef SQ_BWD_DEPTH
#define SQ_BWD_DEPTH 15       // pool slots per lane; 15 (not 16): five blocks' pools fit one SM's shared memory (sqloss.cu SQ_IMPB_MINB)
#endif
constexpr int kBwdDepth = SQ_BWD_DEPTH;
constexpr int kBwdPool = kBwdDepth * 32;      // slots of a warp's pool


// geometry + forward chain + occupancy of one plane (independent of the scan state: two planes can be in flight)
struct Plane { Fwd f; float x, eo, o, cf; };

template <bool FIX>
SQ_HD void plane_forward(const Sample& S, const ImplicitParams& P, const float* bh, const float* bl, float cf, Plane& p) {
    p.cf = cf;
    float sx = fmaf(cf, S.dh[0], bh[0]) + fmaf(cf, S.dl[0], bl[0]);
    float sy = fmaf(cf, S.dh[1], bh[1]) + fmaf(cf, S.dl[1], bl[1]);
    float sz = fmaf(cf, S.dh[2], bh[2]) + fmaf(cf, S.dl[2], bl[2]);
    point_forward<FIX>(S, sx, sy, sz, p.f);
    p.o = occupancy(p.f.F, P.kl, p.x, p.eo);
}

// SQ_F32X2: 0 = off, 1 = forward-only kernels (default), 2 = also the fwd+bwd kernel.  Measured (profiles/tune_r01.txt):
// forward-only kernel -3.7 %; fwd+bwd kernel no gain (the register pairing costs as many moves as the packing saves).
#ifndef SQ_F32X2
#define SQ_F32X2 1
#endif
#if defined(__CUDA_ARCH__) && SQ_F32X2
// Packed fp32 (Blackwell fma/add/sub/mul.f32x2: two operations per issue slot).  The two planes in flight execute the same
// sequence on different data, and the kernel is bound by issue slots, so their non-MUFU arithmetic is done pairwise.
struct F2 { float x, y; };
__device__ __forceinline__ F2 f2(float a, float b) { F2 r; r.x = a; r.y = b; return r; }
#define SQ_F2_OP3(name, op) \
    __device__ __forceinline__ F2 name(F2 a, F2 b, F2 c) { F2 r; \
        asm("{\n .reg .b64 ra, rb, rc, rd;\n mov.b64 ra, {%2, %3};\n mov.b64 rb, {%4, %5};\n mov.b64 rc, {%6, %7};\n " op " rd, ra, rb, rc;\n mov.b64 {%0, %1}, rd;\n}" \
            : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y)); return r; }
#define SQ_F2_OP2(name, op) \
    __device__ __forceinline__ F2 name(F2 a, F2 b) { F2 r; \
        asm("{\n .reg .b64 ra, rb, rd;\n mov.b64 ra, {%2, %3};\n mov.b64 rb, {%4, %5};\n " op " rd, ra, rb;\n mov.b64 {%0, %1}, rd;\n}" \
            : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y)); return r; }
SQ_F2_OP3(fma2, "fma.rn.ftz.f32x2")
SQ_F2_OP2(add2, "add.rn.ftz.f32x2")
SQ_F2_OP2(sub2, "sub.rn.ftz.f32x2")
SQ_F2_OP2(mul2, "mul.rn.ftz.f32x2")

// plane_forward() for two planes at once
template <bool FIX>
__device__ __forceinline__ void plane_forward2(const Sample& S, const ImplicitParams& P, const float* bh, const float* bl,
                                               float cfa, float cfb, Plane& pa, Plane& pb) {
    pa.cf = cfa; pb.cf = cfb;
    const F2 cf = f2(cfa, cfb);
    F2 s[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
        s[i] = add2(fma2(cf, f2(S.dh[i], S.dh[i]), f2(bh[i], bh[i])), fma2(cf, f2(S.dl[i], S.dl[i]), f2(bl[i], bl[i])));
    pa.f.sx = s[0].x; pa.f.sy = s[1].x; pa.f.sz = s[2].x;
    pb.f.sx = s[0].y; pb.f.sy = s[1].y; pb.f.sz = s[2].y;
    F2 m[3] = {s[0], s[1], s[2]};
    if (FIX) {
#pragma unroll
        for (int i = 0; i < 3; ++i) { m[i].x = (m[i].x == 0.0f) ? kAbsFix : m[i].x; m[i].y = (m[i].y == 0.0f) ? kAbsFix : m[i].y; }
    }
    const F2 pxy = f2(S.pxy, S.pxy), one = f2(1.0f, 1.0f);
    const F2 lA = mul2(pxy, f2(lg2_abs(m[0].x), lg2_abs(m[0].y)));
    const F2 lB = mul2(pxy, f2(lg2_abs(m[1].x), lg2_abs(m[1].y)));
    const F2 lC = mul2(f2(S.pz, S.pz), f2(lg2_abs(m[2].x), lg2_abs(m[2].y)));
    const F2 d1 = sub2(lA, lB);
    const F2 t1 = f2(ex2_neg_abs(d1.x), ex2_neg_abs(d1.y));
    const F2 u1 = add2(t1, one);
    const F2 h1 = f2(lg2(u1.x), lg2(u1.y));
    const F2 lE = mul2(f2(S.e21, S.e21), add2(f2(fmaxf(lA.x, lB.x), fmaxf(lA.y, lB.y)), h1));
    const F2 d2 = sub2(lE, lC);
    const F2 t2 = f2(ex2_neg_abs(d2.x), ex2_neg_abs(d2.y));
    const F2 u2 = add2(t2, one);
    const F2 h2 = f2(lg2(u2.x), lg2(u2.y));
    const F2 lG = add2(f2(fmaxf(lE.x, lC.x), fmaxf(lE.y, lC.y)), h2);
    const F2 yy = mul2(f2(S.e1, S.e1), lG);
    const F2 F = f2(ex2(yy.x), ex2(yy.y));
    const F2 xx = fma2(F, f2(P.kl, P.kl), f2(-P.kl, -P.kl));
    const F2 eo = f2(ex2(xx.x), ex2(xx.y));
    const F2 v = add2(eo, one);
    pa.f.d1 = d1.x; pa.f.t1 = t1.x; pa.f.h1 = h1.x; pa.f.d2 = d2.x; pa.f.t2 = t2.x; pa.f.h2 = h2.x; pa.f.lG = lG.x; pa.f.F = F.x;
    pb.f.d1 = d1.y; pb.f.t1 = t1.y; pb.f.h1 = h1.y; pb.f.d2 = d2.y; pb.f.t2 = t2.y; pb.f.h2 = h2.y; pb.f.lG = lG.y; pb.f.F = F.y;
    pa.x = xx.x; pa.eo = eo.x; pa.o = rcp(v.x);
    pb.x = xx.y; pb.eo = eo.y; pb.o = rcp(v.y);
}
#endif

// scan step of one plane: transmittance, suffix-sum bookkeeping and (for gradient-carrying warps) the backward
template <bool BWD, bool FIX, bool QUEUE>      // QUEUE: gradient-carrying points go to the lane's BwdQueue (SQ_BWD_COMPACT)
SQ_HD void plane_scan(const ImplicitParams& P, const Plane& p, ColState& st, ColGrad& cg) {
#if defined(__CUDA_ARCH__)
    SQ_COUNT_HOOK(0, 1);
#endif
    st.csl = fmaf(p.o, -P.tl, st.csl);
    st.cssum += st.csl;
    st.T = ex2(st.csl);
    if (BWD) {
        const bool active = (fabsf(p.x) < P.kact) && (st.csl > -kDeep);
        const unsigned ma = SQ_BALLOT(active);
        if (ma) {
#if defined(SQ_BWD_HOOK) && defined(__CUDA_ARCH__)
            SQ_BWD_HOOK(active);                // debug builds: statistics of how many lanes carry gradient
#endif
            bool now = active;                  // lanes whose point is handled on the spot
            bool any_now = true;                // warp-uniform: does any lane have one
#if defined(SQ_BWD_COMPACT)
            if (QUEUE) {
                // all active lanes of this plane append together, in lane order: front slots for the points near the
                // surface, back slots for the others
                const bool shell = active && fabsf(p.x) < kRefine;
                const unsigned ms = SQ_BALLOT(shell), mp = ma ^ ms;
                // (POPC runs on the MUFU pipe at the MUFU rate -- csrc/peaks.cu EX2_POPC -- but taking the two counts from one
                // REDUX of packed flags instead, which does not, measured no faster: profiles/tune_r02.txt run q)
                const int cnt_r = popcount(ms), cnt_p = popcount(mp);
                const int nr1 = st.nr + cnt_r, top1 = st.top - cnt_p;
                if (nr1 <= top1 + 1 && nr1 < kNoLink) {        // warp-uniform: they all fit
                    if (active) {
#if defined(__CUDA_ARCH__)
                        // `where` = the pool's shared-memory address | this lane: one register, opaque to the compiler --
                        // left to itself it rebuilds address, lane and lane mask from special registers at every append
                        // (three S2R and six more instructions, measured 3 k cycles per warp)
                        const unsigned lane_ = st.q.where & 31u;
                        const int rank = popcount((shell ? ms : mp) & ((1u << lane_) - 1u));
                        const int at = shell ? st.nr + rank : st.top - rank;
                        const unsigned tag = lane_ | ((unsigned)(shell ? st.head : kNoLink) << 5);
                        const unsigned addr = (st.q.where & ~31u) + 4u * (unsigned)at;
                        asm volatile("st.shared.b32 [%0], %1;\n\tst.shared.f32 [%0 + %4], %2;\n\tst.shared.f32 [%0 + %5], %3;"
                                     :: "r"(addr), "r"((f32_bits(p.cf) & ~kTagMask) | tag), "f"(st.psh),
                                        "f"(shell ? p.x : p.eo * p.o * p.o), "n"(4 * kBwdPool), "n"(8 * kBwdPool) : "memory");
#else
                        const int rank = popcount((shell ? ms : mp) & lanes_below());
                        const int at = shell ? st.nr + rank : st.top - rank;
                        const unsigned tag = (unsigned)st.q.lane | ((unsigned)(shell ? st.head : kNoLink) << 5);
                        st.q.cf[at] = bits_f32((f32_bits(p.cf) & ~kTagMask) | tag);    // plane | lane | previous front entry of the column
                        st.q.pre[at] = st.psh;                            // T in front of it since the first active point
                        st.q.x[at] = shell ? p.x : p.eo * p.o * p.o;      // refined later: x; else the weight o (1 - o) itself
#endif
                        st.head = shell ? at : st.head;
                        st.seen = 1.0f;
                    }
                    st.nr = nr1; st.top = top1;
                    now = false; any_now = false;
                } else {
                    st.spilled = st.spilled || active;
                }
            }
            if (any_now)
#endif
            {
#if defined(__CUDA_ARCH__)
                SQ_COUNT_HOOK(1, 1);
#endif
                // do/dF = -k o (1-o) = -k eo o^2 ; the -k is applied in finalize
                const float W = now ? p.eo * p.o * p.o : 0.0f;
                Fwd fa = p.f;
                if (!now) fwd_neutral(fa);          // keep the other lanes finite
                Bwd b;
                point_backward<FIX>(fa, W, b);
                st.seen = now ? 1.0f : st.seen;
                const float pp = st.psh;       // T in front of this point (since the first active one)
                for (int i = 0; i < 3; ++i) {
                    cg.gs0[i] += b.gs[i];            cg.gs1[i] = fmaf(pp, b.gs[i], cg.gs1[i]);
                    const float gz = b.gs[i] * p.cf;
                    cg.gz0[i] += gz;                 cg.gz1[i] = fmaf(pp, gz, cg.gz1[i]);
                }
                for (int i = 0; i < 2; ++i) { cg.ge0[i] += b.ge[i]; cg.ge1[i] = fmaf(pp, b.ge[i], cg.ge1[i]); }
            }
        }
        st.psh = fmaf(st.seen, st.T, st.psh);
    }
    st.tsum += st.T;
}

// ---- the queued points after the walk (SQ_BWD_COMPACT), three steps; `at` = index of the entry in the queue arrays
// 1. refined entries: x from the fp64 chain, and the first-order change of the point's occupancy that goes with it
SQ_HD void queue_store_refined(const BwdQueue& q, int at, float x0, float x1) {
    const float eo = ex2(x1), o = rcp(1.0f + eo), w = eo * o * o;
    q.x[at] = w;
    q.d[at] = -(float)kLn2 * w * (x1 - x0);               // d o / d x = -ln2 o (1 - o)
}
SQ_HD void queue_refine_entry(const Sample& S, double step, float kl, const BwdQueue& q, int at,
                              double b0, double b1, double b2, const RefTabs& tb) {
    const float x0 = q.x[at];
    queue_store_refined(q, at, x0, refined_x(S, step, kl, b0, b1, b2, entry_cf(S, q.cf[at]), tb));
}
// 2. suffix weight of entry e of a column, S_e = U - prefix_e, corrected to first order for the occupancy changes of the
// column's refined entries.  T_c = exp(-tau cs_c) and cs_c sums the occupancies at or in front of c, so with
// o_p -> o_p + d_p:  T_c -> T_c (1 - tau sum_{p <= c} d_p)  and
//   S_e -> S_e - tau ( S_e sum_{p <= e} d_p  +  sum_{p > e} d_p S_p ).
// The occupancy the scan saw carries the fp32 chain's error in x (~1e-4 at k = 260), and through tau cs it reaches the
// weight of EVERY point behind; measured (tests/emu, profiles/parity_sweep_r02.json) this is the larger part of the
// fp32 gradient error.  Evaluated per dealt entry by a loop over the front entries of the entry's column (one to three,
// typically: the planes where the column crosses the surface), which are chained through `meta` from the column's latest
// one (`head`) back; the walk goes down the planes, so "at or before e" is "plane index not below e's".
SQ_HD float queue_suffix_weight(const BwdQueue& q, int at, int head, float U, float tau) {
    // (plane order is read off the tagged values: the tag sits below the plane's bits, and two entries of one column are on
    // different planes unless they are the same entry)
    const float Se = U - q.pre[at];
    const unsigned cfe = f32_bits(q.cf[at]) | kTagMask;
    float a = 0.f, b = 0.f;                                  // sum of d over front entries at or before e; sum of d S behind e
    for (int r = head; r != kNoLink; ) {
        const float tagged = q.cf[r], d = q.d[r], Sr = U - q.pre[r];
        if ((f32_bits(tagged) | kTagMask) >= cfe) a += d; else b = fmaf(d, Sr, b);
        r = entry_link(tagged);
    }
    return Se - tau * fmaf(a, Se, b);
}
// The same occupancy changes move the rendered depth of the column: depth = 1 - sum_c T_c / n, so
//   depth -> depth + (tau / n) sum_{refined p} d_p S_p.
// At 1e-7 it is invisible in one pixel, but it has the sign of the MUFU lg2 bias on every surface pixel, and for an object
// that fills the image and a prediction close to the target (loss ~ 3e-3) it is 2e-5 of the loss (measured); the loss
// tolerance is rtol 1e-5.  Returns sum d_p S_p for one column (its owner adds sign * tau / n * this to the loss).
SQ_HD float queue_depth_shift(const BwdQueue& q, int head, float U) {
    float acc = 0.f;
    for (int r = head; r != kNoLink; r = entry_link(q.cf[r])) acc = fmaf(q.d[r], U - q.pre[r], acc);
    return acc;
}
// (The points a full pool sends to the on-the-spot path get neither the refinement nor this correction; with 480 slots per
// 32-column group that takes more gradient points than any workload of the parity fuzz has.)
// 3. every entry: forward redone in fp32 for the ratios the backward needs (not amplified by k); weight o (1 - o) and
// suffix weight from the queue.  sign = sign(depth - target) of the column.
template <bool FIX>
SQ_HD void queue_entry_backward(const Sample& S, const float* bh, const float* bl, float cf,
                                float w, float Sw, float sign, bool has, Bwd& b) {
    Fwd f;
    float sx = fmaf(cf, S.dh[0], bh[0]) + fmaf(cf, S.dl[0], bl[0]), sy = fmaf(cf, S.dh[1], bh[1]) + fmaf(cf, S.dl[1], bl[1]),
          sz = fmaf(cf, S.dh[2], bh[2]) + fmaf(cf, S.dl[2], bl[2]);
    point_forward<FIX>(S, sx, sy, sz, f);
    float W = w * Sw * sign;
    if (!has) { fwd_neutral(f); W = 0.f; }
    point_backward<FIX>(f, W, b);
}

// ILP: number of z planes whose (independent) forward chains are in flight per thread.  A column walk is a serial
// chain of ~8 dependent MUFU ops per plane; two planes in flight halve the latency of the longest work item, which
// is what bounds the kernel at small batch.
#ifndef SQ_IMP_ILP
#define SQ_IMP_ILP 2
#endif

template <bool BWD, bool FIX = true, bool QUEUE = false>
// QUEUE (SQ_BWD_COMPACT): bwd_q / U_out / nr_io / top_io / spilled_out / head_out are used (see ColState; nr_io, top_io: the
// pool's front count and next free back slot, in and out -- the kernels start every column group at 0 and cap - 1, the host
// build carries them from column to column of a group); colgrad11 then holds only what was handled on the spot.
SQ_HD float implicit_column(const Sample& S, const Grid& g, const ImplicitParams& P,
                            const float* bh, const float* bl, int c_lo, int c_hi, int lane_lo, float* colgrad11,
                            const BwdQueue* bwd_q = nullptr, float* U_out = nullptr, int* nr_io = nullptr, int* top_io = nullptr,
                            bool* spilled_out = nullptr, int* head_out = nullptr) {
    // planes in front of the range: o = 0, cs = 0, T = 1 each
    ColState st;
    if (QUEUE) { st.q = *bwd_q; st.nr = *nr_io; st.top = *top_io; }
    else { st.q.cf = st.q.pre = st.q.x = st.q.d = nullptr; st.q.cap = 0; st.q.lane = 0; st.q.where = 0u; st.nr = 0; st.top = -1; }
    st.spilled = false; st.head = kNoLink;
    st.csl = 0.f;                                     // -tau log2(e) cs
    st.T = 1.0f;                                      // 2^csl
    st.tsum = (float)(g.n - 1 - c_hi);
    st.cssum = 0.f;                                   // sum_c csl_c
    st.psh = 0.f; st.seen = 0.f;
    ColGrad cg;
    if (BWD) {
        for (int i = 0; i < 3; ++i) cg.gs0[i] = cg.gs1[i] = cg.gz0[i] = cg.gz1[i] = 0.f;
        cg.ge0[0] = cg.ge0[1] = cg.ge1[0] = cg.ge1[1] = 0.f;
    }
    int c = c_hi;
    float cfi = (float)c_hi;                          // plane "index": exact small integers, z0/step for plane 0
    // The walk ends early once no lane of the warp needs the planes that are left: a lane is finished when its
    // transmittance has fallen below 2^-kDeep (what lies behind adds < n 2^-kDeep to the depth and carries no gradient, see
    // kDeep) or when the walk has left the lane's OWN culled range [lane_lo, ..] (the warp walks the union).  The planes
    // not walked are accounted for in closed form below, like the planes behind the range.
    bool stop = false;
#if SQ_IMP_ILP >= 2
    for (; !stop && c - (SQ_IMP_ILP - 1) >= c_lo; c -= SQ_IMP_ILP, cfi -= (float)SQ_IMP_ILP) {
        Plane p[SQ_IMP_ILP];
#if defined(__CUDA_ARCH__) && SQ_F32X2 && SQ_IMP_ILP == 2
        if (SQ_F32X2 >= 2 || !BWD) {
            plane_forward2<FIX>(S, P, bh, bl, cfi, (c - 1 == 0) ? S.cf0 : cfi - 1.0f, p[0], p[1]);
        } else
#endif
        {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int j = 0; j < SQ_IMP_ILP; ++j)
                plane_forward<FIX>(S, P, bh, bl, (j > 0 && c - j == 0) ? S.cf0 : cfi - (float)j, p[j]);
        }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int j = 0; j < SQ_IMP_ILP; ++j) plane_scan<BWD, FIX, QUEUE>(P, p[j], st, cg);
#ifndef SQ_NO_EARLY_EXIT
        stop = !SQ_ANY(st.csl > -kDeep && c - SQ_IMP_ILP >= lane_lo);
#endif
    }
#endif
    for (; !stop && c >= c_lo; --c, cfi -= 1.0f) {
        Plane p0;
        plane_forward<FIX>(S, P, bh, bl, (c == 0) ? S.cf0 : cfi, p0);
        plane_scan<BWD, FIX, QUEUE>(P, p0, st, cg);
#ifndef SQ_NO_EARLY_EXIT
        stop = !SQ_ANY(st.csl > -kDeep && c - 1 >= lane_lo);
#endif
    }
    // planes behind the range (and planes left out by the early exit): o = 0, cs and T stay what they are
    const float nb = (float)(c + 1);
    st.tsum = fmaf(nb, st.T, st.tsum);
    st.cssum = fmaf(nb, st.csl, st.cssum);
    if (BWD) {
        const float U = fmaf(nb * st.seen, st.T, st.psh);
        if (QUEUE) { *U_out = U; *nr_io = st.nr; *top_io = st.top; *spilled_out = st.spilled; *head_out = st.head; }
        for (int i = 0; i < 3; ++i) {
            colgrad11[i]     = fmaf(U, cg.gs0[i], -cg.gs1[i]);
            colgrad11[3 + i] = fmaf(U, cg.gz0[i], -cg.gz1[i]);
            // the size gradient needs sum gs_i s_i, and s_i = base_i + d_i cf is affine along the column: no accumulator
            colgrad11[6 + i] = fmaf(bh[i], colgrad11[i], fmaf(S.dh[i], colgrad11[3 + i],
                               fmaf(bl[i], colgrad11[i], S.dl[i] * colgrad11[3 + i])));
        }
        colgrad11[9]  = fmaf(U, cg.ge0[0], -cg.ge1[0]);
        colgrad11[10] = fmaf(U, cg.ge0[1], -cg.ge1[1]);
    }
    const float depth = fmaf(-st.tsum, g.inv_n, 1.0f);
    return depth < 1e-4f ? -(float)kLn2 * st.cssum * g.inv_n : depth;     // tau sum cs = -ln2 sum csl
}

// fold one finished column (weight w = sign(depth - target), coordinates relative to t) into the thread totals
SQ_HD void implicit_fold(Acc& acc, const float* colgrad11, float w, float dx, float dy) {
    for (int i = 0; i < 3; ++i) {
        const float gsi = w * colgrad11[i];
        acc.gs[i] += gsi;
        acc.gm[3 * i + 0] = fmaf(gsi, dx, acc.gm[3 * i + 0]);
        acc.gm[3 * i + 1] = fmaf(gsi, dy, acc.gm[3 * i + 1]);
        acc.gm[3 * i + 2] = fmaf(w, colgrad11[3 + i], acc.gm[3 * i + 2]);
        acc.wa[i] = fmaf(w, colgrad11[6 + i], acc.wa[i]);
    }
    acc.ge[0] = fmaf(w, colgrad11[9], acc.ge[0]);
    acc.ge[1] = fmaf(w, colgrad11[10], acc.ge[1]);
}

// one queued point's backward terms into the item's sums (dx, dy: its column's position relative to t)
SQ_HD void acc_add_point(Acc& acc, const Bwd& b, float cf, float dx, float dy) {
    for (int i = 0; i < 3; ++i) {
        acc.gs[i] += b.gs[i];
        acc.gm[3 * i + 0] = fmaf(b.gs[i], dx, acc.gm[3 * i + 0]);
        acc.gm[3 * i + 1] = fmaf(b.gs[i], dy, acc.gm[3 * i + 1]);
        acc.gm[3 * i + 2] = fmaf(b.gs[i], cf, acc.gm[3 * i + 2]);
        acc.wa[i] += b.wa[i];
    }
    acc.ge[0] += b.ge[0]; acc.ge[1] += b.ge[1];
}

// ---------------------------------------------------------------- ExplicitLoss: one column
// classes.py:187-198: o = sigmoid(5 (1 - F)) for the true and the predicted SQ, loss = 100 mean (o_t - o_p)^2.
// Returns sum_c (o_t - o_p)^2 over the column and accumulates d/d(pred) terms weighted by (o_t - o_p).
// rt / rp: warp-uniform z ranges {lo, hi} of the true / predicted SQ (column_range + warp_range); outside its
// range an SQ's occupancy is exactly 0 and its chain is not evaluated.
struct Range { int lo, hi; };

// SQ_EXP_PAIR: where both superquadrics are in range, their two forward chains -- the same instruction sequence on
// different data and different per-sample constants -- run as packed fp32 pairs (true SQ in .x, predicted in .y).
#ifndef SQ_EXP_PAIR
#define SQ_EXP_PAIR 0
#endif
#if defined(__CUDA_ARCH__) && SQ_F32X2 && SQ_EXP_PAIR
template <bool FIX>
__device__ __forceinline__ void forward_pair(const Sample& Sa, const Sample& Sb, float kl, float cf,
                                             const float* bha, const float* bla, const float* bhb, const float* blb,
                                             Fwd& fa, Fwd& fb, float& oa, float& ob, float& xb, float& eb) {
    const F2 c = f2(cf, cf);
    F2 s[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
        s[i] = add2(fma2(c, f2(Sa.dh[i], Sb.dh[i]), f2(bha[i], bhb[i])), fma2(c, f2(Sa.dl[i], Sb.dl[i]), f2(bla[i], blb[i])));
    fa.sx = s[0].x; fa.sy = s[1].x; fa.sz = s[2].x;
    fb.sx = s[0].y; fb.sy = s[1].y; fb.sz = s[2].y;
    F2 m[3] = {s[0], s[1], s[2]};
    if (FIX) {
#pragma unroll
        for (int i = 0; i < 3; ++i) { m[i].x = (m[i].x == 0.0f) ? kAbsFix : m[i].x; m[i].y = (m[i].y == 0.0f) ? kAbsFix : m[i].y; }
    }
    const F2 pxy = f2(Sa.pxy, Sb.pxy), one = f2(1.0f, 1.0f);
    const F2 lA = mul2(pxy, f2(lg2_abs(m[0].x), lg2_abs(m[0].y)));
    const F2 lB = mul2(pxy, f2(lg2_abs(m[1].x), lg2_abs(m[1].y)));
    const F2 lC = mul2(f2(Sa.pz, Sb.pz), f2(lg2_abs(m[2].x), lg2_abs(m[2].y)));
    const F2 d1 = sub2(lA, lB);
    const F2 t1 = f2(ex2_neg_abs(d1.x), ex2_neg_abs(d1.y));
    const F2 u1 = add2(t1, one);
    const F2 h1 = f2(lg2(u1.x), lg2(u1.y));
    const F2 lE = mul2(f2(Sa.e21, Sb.e21), add2(f2(fmaxf(lA.x, lB.x), fmaxf(lA.y, lB.y)), h1));
    const F2 d2 = sub2(lE, lC);
    const F2 t2 = f2(ex2_neg_abs(d2.x), ex2_neg_abs(d2.y));
    const F2 u2 = add2(t2, one);
    const F2 h2 = f2(lg2(u2.x), lg2(u2.y));
    const F2 lG = add2(f2(fmaxf(lE.x, lC.x), fmaxf(lE.y, lC.y)), h2);
    const F2 yy = mul2(f2(Sa.e1, Sb.e1), lG);
    const F2 F = f2(ex2(yy.x), ex2(yy.y));
    const F2 xx = fma2(F, f2(kl, kl), f2(-kl, -kl));
    const F2 eo = f2(ex2(xx.x), ex2(xx.y));
    const F2 v = add2(eo, one);
    fa.d1 = d1.x; fa.t1 = t1.x; fa.h1 = h1.x; fa.d2 = d2.x; fa.t2 = t2.x; fa.h2 = h2.x; fa.lG = lG.x; fa.F = F.x;
    fb.d1 = d1.y; fb.t1 = t1.y; fb.h1 = h1.y; fb.d2 = d2.y; fb.t2 = t2.y; fb.h2 = h2.y; fb.lG = lG.y; fb.F = F.y;
    oa = rcp(v.x); ob = rcp(v.y); xb = xx.y; eb = eo.y;
}
#endif

// one z plane of explicit_column; HAS_T / HAS_P: whether the true / predicted SQ can be occupied on this plane.
// VJP (sq_occupancy_vjp): no true SQ, no squared difference; the point's weight is the upstream voxel `up` (dL/d o) and the
// weight cut is `kact` bits (kExplicitVjpBits) instead of kActiveExplicit, and the z moment is taken about plane `zc`.
// VOX (with VJP; sq_voxel_loss): `up` is the target voxel v and takes the place of o_t: d = v - o_p, sq += d^2, weight d as in
// the loss, with the VJP's cut and z centre.  BWD = false is the forward-only walk of the same points.
template <bool BWD, bool HAS_T, bool HAS_P, bool VJP = false, bool VOX = false>
SQ_HD void explicit_step(const Sample& St, const Sample& Sp, float kl, float cf,
                         const float* bht, const float* blt, const float* bhp, const float* blp,
                         float& sq, float* gs, float* gz, Acc& acc, float up = 0.f, float kact = kActiveExplicit, float zc = 0.f) {
    static_assert(!VJP || ((BWD || VOX) && !HAS_T && HAS_P), "the VJP mode walks the predicted SQ alone");
    static_assert(!VOX || VJP, "the voxel loss is a variant of the VJP walk");
    float ot = 0.f, op = 0.f, xp = 1e30f, ep = 0.f;
    Fwd ft, fp;
#if defined(__CUDA_ARCH__) && SQ_F32X2 && SQ_EXP_PAIR
    if (HAS_T && HAS_P) {
        forward_pair<true>(St, Sp, kl, cf, bht, blt, bhp, blp, ft, fp, ot, op, xp, ep);
    } else
#endif
    {
    if (HAS_T) {
        float sx = fmaf(cf, St.dh[0], bht[0]) + fmaf(cf, St.dl[0], blt[0]), sy = fmaf(cf, St.dh[1], bht[1]) + fmaf(cf, St.dl[1], blt[1]),
              sz = fmaf(cf, St.dh[2], bht[2]) + fmaf(cf, St.dl[2], blt[2]);
        point_forward<true>(St, sx, sy, sz, ft);
    }
    if (HAS_P) {
        float sx = fmaf(cf, Sp.dh[0], bhp[0]) + fmaf(cf, Sp.dl[0], blp[0]), sy = fmaf(cf, Sp.dh[1], bhp[1]) + fmaf(cf, Sp.dl[1], blp[1]),
              sz = fmaf(cf, Sp.dh[2], bhp[2]) + fmaf(cf, Sp.dl[2], blp[2]);
        point_forward<true>(Sp, sx, sy, sz, fp);
    }
    if (HAS_T) { float xt, et; ot = occupancy(ft.F, kl, xt, et); }
    if (HAS_P) op = occupancy(fp.F, kl, xp, ep);
    }
    const float d = (VOX ? up : ot) - op;
    if (!VJP || VOX) sq = fmaf(d, d, sq);
    if (BWD && HAS_P) {
        // VJP: points under a zero upstream voxel carry nothing (sparse upstreams skip the backward)
        const bool active = VJP ? (fabsf(xp) < kact && (VOX || up != 0.0f)) : fabsf(xp) < kActiveExplicit;
        if (SQ_ANY(active)) {
            // d/dF_p of (o_t - o_p)^2 = 2 d * k o_p (1 - o_p); constants 2, k applied in finalize
            // (VJP: d o_p / dF_p = -k o_p (1 - o_p) times the upstream; -k applied in finalize)
            const float W = active ? (VJP && !VOX ? up : d) * ep * op * op : 0.0f;
            Fwd fa = fp;
            if (!active) fwd_neutral(fa);
            Bwd b;
            point_backward(fa, W, b);
            for (int i = 0; i < 3; ++i) {
                gs[i] += b.gs[i];
                gz[i] = fmaf(b.gs[i], VJP ? cf - zc : cf, gz[i]);
            }
            acc.ge[0] += b.ge[0];
            acc.ge[1] += b.ge[1];
        }
    }
}

// The plane "index" of t_z, cf(t) = t_z / step, rounded to fp32 the same way in the column kernel and in finalize.  The
// VJP's z moment is taken about it: sum gs (cf - cf(t)) instead of sum gs cf.  The gradient sums of a VJP can be large and of
// one sign on each side of the object and cancel only between far-apart columns (the soft volume's rotation and translation
// entries; measured: 1e-5 of the size entries), so their fp32 roundings have to be small against the centred moment, not
// against z (t_z = 1: |z| up to 1, |z - t_z| at most ~0.35 over the object's shell).
SQ_HD float plane_of_t(const Sample& S, const Grid& g) { return d2f(S.t[2] / g.step); }

// read-only load of an upstream value (device: through the non-coherent path, cached in L1)
SQ_HD float load_ro(const float* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
SQ_HD float load_ro(const unsigned char* p) {
#if defined(__CUDA_ARCH__)
    return (float)__ldg(p);
#else
    return (float)*p;
#endif
}

// sum of v^2, v = vscale * vox[c], over the planes of one column of n voxels outside the walked range rp (all of them when
// rp is empty): the voxel loss's terms where the predicted occupancy is below the cut and taken as 0.  NULL: a masked lane.
// No MUFU work: the loop is bound by the loads, which are independent of each other.
template <typename V>
SQ_HD float voxel_sq_outside(const V* vox, int n, Range rp, float vscale) {
    float sq = 0.f;
    if (!vox) return sq;
    const int hi = rp.hi < rp.lo ? -1 : rp.hi, lo = rp.hi < rp.lo ? 0 : rp.lo;
#pragma unroll 4
    for (int c = hi + 1; c < n; ++c) { const float v = vscale * load_ro(vox + c); sq = fmaf(v, v, sq); }
#pragma unroll 4
    for (int c = 0; c < lo; ++c) { const float v = vscale * load_ro(vox + c); sq = fmaf(v, v, sq); }
    return sq;
}

// VJP (sq_occupancy_vjp): the predicted SQ alone over rp (rt is ignored), every point weighted by the upstream voxel
// up[c] of the column (NULL: a masked lane, weight 0), weight cut at `kact` bits, the z moment acc.gm[i][2] taken about
// plane_of_t() (finalize_sample's z_centre); returns 0.
// VOX (with VJP; sq_voxel_loss): up[c] (V = float or uint8_t, times vscale) is the target voxel v; returns the column's
// whole sum of squares: (v - o_p)^2 over the walked planes, then v^2 over the others (voxel_sq_outside).  With BWD = false
// the same planes are walked for the loss alone, so the loss does not depend on whether a gradient is asked for.
// A lane reads its own column, consecutive floats along z, 32 different rows per warp and plane: each 32-byte sector
// comes from DRAM once per walk and serves the next planes from L1.  The loads are issued two planes ahead of the plane
// that uses them, so the one plane in eight that misses L1 waits behind two forward chains instead of stalling one.
template <bool BWD, bool VJP = false, bool VOX = false, typename V = float>
SQ_HD float explicit_column(const Sample& St, const Sample& Sp, const Grid& g, float kl,
                            const float* bht, const float* blt, const float* bhp, const float* blp,
                            Range rt, Range rp, float dx, float dy, Acc& acc,
                            const V* up = nullptr, float kact = kActiveExplicit, float vscale = 1.f) {
    float sq = 0.f;
    float gs[3] = {0.f, 0.f, 0.f}, gz[3] = {0.f, 0.f, 0.f};
    float zc = 0.f;
    if constexpr (VJP) {
        zc = plane_of_t(Sp, g);
        const int c_hi = rp.hi, c_lo = rp.lo;
        auto ld = [&](int c) { return VOX ? vscale * load_ro(up + c) : load_ro(up + c); };
        float u0 = (up && c_hi >= c_lo) ? ld(c_hi) : 0.f;
        float u1 = (up && c_hi - 1 >= c_lo) ? ld(c_hi - 1) : 0.f;
        float cfi = (float)c_hi;
        for (int c = c_hi; c >= c_lo; --c, cfi -= 1.0f) {
            const float u2 = (up && c - 2 >= c_lo) ? ld(c - 2) : 0.f;
            const float cf = (c == 0) ? Sp.cf0 : cfi;
            explicit_step<BWD, false, true, true, VOX>(Sp, Sp, kl, cf, bhp, blp, bhp, blp, sq, gs, gz, acc, u0, kact, zc);
            u0 = u1; u1 = u2;
        }
        if constexpr (VOX) sq += voxel_sq_outside(up, g.n, rp, vscale);
    } else {
        const bool et = rt.hi < rt.lo, ep = rp.hi < rp.lo;
        const int c_hi = rt.hi > rp.hi ? rt.hi : rp.hi;
        const int c_lo = et ? rp.lo : ep ? rt.lo : (rt.lo < rp.lo ? rt.lo : rp.lo);
        float cfi = (float)c_hi;
        for (int c = c_hi; c >= c_lo; --c, cfi -= 1.0f) {
            const float cf = (c == 0) ? Sp.cf0 : cfi;
            const bool in_t = (c >= rt.lo && c <= rt.hi), in_p = (c >= rp.lo && c <= rp.hi);    // warp-uniform
            if (in_t && in_p) explicit_step<BWD, true, true>(St, Sp, kl, cf, bht, blt, bhp, blp, sq, gs, gz, acc);
            else if (in_p)    explicit_step<BWD, false, true>(St, Sp, kl, cf, bht, blt, bhp, blp, sq, gs, gz, acc);
            else if (in_t)    explicit_step<BWD, true, false>(St, Sp, kl, cf, bht, blt, bhp, blp, sq, gs, gz, acc);
        }
    }
    if (BWD) {
        for (int i = 0; i < 3; ++i) {
            acc.gs[i] += gs[i];
            acc.gm[3 * i + 0] = fmaf(gs[i], dx, acc.gm[3 * i + 0]);
            acc.gm[3 * i + 1] = fmaf(gs[i], dy, acc.gm[3 * i + 1]);
            acc.gm[3 * i + 2] += gz[i];
            // sum gs_i s_i with s_i = base_i + d_i cf (see implicit_column; VJP: s_i = (base_i + d_i zc) + d_i (cf - zc))
            if (VJP) acc.wa[i] += fmaf(fmaf(Sp.dh[i], zc, bhp[i]), gs[i], fmaf(Sp.dh[i], gz[i], fmaf(fmaf(Sp.dl[i], zc, blp[i]), gs[i], Sp.dl[i] * gz[i])));
            else acc.wa[i] += fmaf(bhp[i], gs[i], fmaf(Sp.dh[i], gz[i], fmaf(blp[i], gs[i], Sp.dl[i] * gz[i])));
        }
    }
    return sq;
}

// ---------------------------------------------------------------- IoU: one column
// classes.py:398-438: no clamp, no fix-up; inside <=> F <= 1 <=> e1 * lg2(G) <= 0.  Points whose decision is
// within `margin` of the boundary are re-evaluated in fp64 with the reference's own operation order so the
// voxel counts match the fp64 reference exactly (DESIGN.md "IoU exactness").
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
bool inside_exact(const SampleFull& S, const Grid& g, int ia, int ib, int ic) {
    const double gx = grid_coord(g, ia), gy = grid_coord(g, ib), gz = grid_coord(g, ic);
    double s[3];
    for (int i = 0; i < 3; ++i) {
        const double r = S.M[3 * i] * gx + S.M[3 * i + 1] * gy + S.M[3 * i + 2] * gz;
        const double tr = S.M[3 * i] * S.t[0] + S.M[3 * i + 1] * S.t[1] + S.M[3 * i + 2] * S.t[2];
        s[i] = (r - tr) / S.a[i];
    }
    const double A = pow(s[0] * s[0], 1.0 / S.e[1]), B = pow(s[1] * s[1], 1.0 / S.e[1]), C = pow(s[2] * s[2], 1.0 / S.e[0]);
    const double F = pow(pow(A + B, S.e[1] / S.e[0]) + C, S.e[0]);
    return F <= 1.0;
}

SQ_HD float log2F(const Sample& S, float sx, float sy, float sz) {
    Fwd f;
    point_forward<false>(S, sx, sy, sz, f);
    return S.e1 * f.lG;
}

constexpr float kIoUMargin = 2e-4f;     // |log2 F| below which the fp32 decision is not trusted

// The z ranges come from column_range() with kIoUBound: a point with max|s_i| >= kIoUBound has F >= 1.002, far
// beyond the margin, so it is outside without evaluating anything.
constexpr float kIoUBound = 1.001f;

// Ft / Fp: the full records (in HBM), read only for the fp64 tie-break
SQ_HD float log2F_plane(const Sample& S, const float* bh, const float* bl, float cf) {
    return log2F(S, fmaf(cf, S.dh[0], bh[0]) + fmaf(cf, S.dl[0], bl[0]),
                    fmaf(cf, S.dh[1], bh[1]) + fmaf(cf, S.dl[1], bl[1]),
                    fmaf(cf, S.dh[2], bh[2]) + fmaf(cf, S.dl[2], bl[2]));
}

// Two planes per iteration: up to four independent MUFU chains (two SQs x two planes) in flight per thread -- the
// one-plane version spent most of its time waiting on the chain's own latency (ncu: XU pipe 37 % busy).
SQ_HD void iou_column(const Sample& St, const Sample& Sp, const SampleFull* Ft, const SampleFull* Fp, const Grid& g,
                      int ia, int ib, const float* bht, const float* blt, const float* bhp, const float* blp,
                      Range rt, Range rp, unsigned& inter, unsigned& uni) {
    const int c_hi = rt.hi > rp.hi ? rt.hi : rp.hi;
    const int c_lo = (rt.hi < rt.lo) ? rp.lo : (rp.hi < rp.lo) ? rt.lo : (rt.lo < rp.lo ? rt.lo : rp.lo);
    float cfi = (float)c_hi;
    for (int c = c_hi; c >= c_lo; c -= 2, cfi -= 2.0f) {
        const int c1 = c - 1;
        const bool has1 = c1 >= c_lo;
        const float cf0 = (c == 0) ? Sp.cf0 : cfi, cf1 = (c1 == 0) ? Sp.cf0 : cfi - 1.0f;
        const bool t0 = c >= rt.lo && c <= rt.hi, t1 = has1 && c1 >= rt.lo && c1 <= rt.hi;       // warp-uniform
        const bool p0 = c >= rp.lo && c <= rp.hi, p1 = has1 && c1 >= rp.lo && c1 <= rp.hi;
        float yt0 = 1.f, yt1 = 1.f, yp0 = 1.f, yp1 = 1.f;                                       // log2 F > 0: outside
        if (t0 || t1) { yt0 = log2F_plane(St, bht, blt, cf0); yt1 = log2F_plane(St, bht, blt, cf1); }
        if (p0 || p1) { yp0 = log2F_plane(Sp, bhp, blp, cf0); yp1 = log2F_plane(Sp, bhp, blp, cf1); }
        bool it0 = t0 && yt0 <= 0.f, it1 = t1 && yt1 <= 0.f, ip0 = p0 && yp0 <= 0.f, ip1 = p1 && yp1 <= 0.f;
        // decisions too close to call in fp32 (also NaN) are re-taken in fp64, in the reference's operation order
        const bool n_t0 = t0 && !(fabsf(yt0) > kIoUMargin), n_t1 = t1 && !(fabsf(yt1) > kIoUMargin);
        const bool n_p0 = p0 && !(fabsf(yp0) > kIoUMargin), n_p1 = p1 && !(fabsf(yp1) > kIoUMargin);
        if (n_t0 || n_t1 || n_p0 || n_p1) {
            if (n_t0) it0 = inside_exact(*Ft, g, ia, ib, c);
            if (n_t1) it1 = inside_exact(*Ft, g, ia, ib, c1);
            if (n_p0) ip0 = inside_exact(*Fp, g, ia, ib, c);
            if (n_p1) ip1 = inside_exact(*Fp, g, ia, ib, c1);
        }
        inter += ((it0 && ip0) ? 1u : 0u) + ((it1 && ip1) ? 1u : 0u);
        uni += ((it0 || ip0) ? 1u : 0u) + ((it1 || ip1) ? 1u : 0u);
    }
}

// ---------------------------------------------------------------- LeastSquares: one point
// classes.py:322-355: (sqrt(a1 a2 a3) (F - 1))^2 at a back-projected depth pixel (x, y, z).  Returns the squared
// term without the a1 a2 a3 factor; accumulates d/dF-weighted terms.  The a-gradient of the prefactor is added in
// finalize from the returned sum.
template <bool BWD>
SQ_HD float lsq_point(const Sample& S, float px, float py, float pz, Acc& acc) {
    const double dx = (double)px - S.t[0], dy = (double)py - S.t[1], dz = (double)pz - S.t[2];
    float s[3];
    for (int i = 0; i < 3; ++i) s[i] = (float)(S.Ms[3 * i] * dx + S.Ms[3 * i + 1] * dy + S.Ms[3 * i + 2] * dz);
    Fwd f;
    point_forward<true>(S, s[0], s[1], s[2], f);
    const float r = f.F - 1.0f;
    if (BWD) {
        // d/dF of (F-1)^2 = 2 (F-1); the 2 and a1 a2 a3 are applied in finalize
        Fwd fa = f;
        const bool ok = f.F < 1e18f;
        if (!ok) fwd_neutral(fa);
        Bwd b;
        point_backward(fa, ok ? r : 0.f, b);
        const float fdx = (float)dx, fdy = (float)dy, fdz = (float)dz;
        for (int i = 0; i < 3; ++i) {
            acc.gs[i] += b.gs[i];
            acc.gm[3 * i + 0] = fmaf(b.gs[i], fdx, acc.gm[3 * i + 0]);
            acc.gm[3 * i + 1] = fmaf(b.gs[i], fdy, acc.gm[3 * i + 1]);
            acc.gm[3 * i + 2] = fmaf(b.gs[i], fdz, acc.gm[3 * i + 2]);
            acc.wa[i] += b.wa[i];
        }
        acc.ge[0] += b.ge[0];
        acc.ge[1] += b.ge[1];
    }
    return r * r;
}

}  // namespace sq
