// ast_math.h -- SPH kernel shapes and normalisations.
//   W(r,h) = norm(h) * f(q),  q = r/h,  support q < 2  (hard mask of the reference, _pixel_calculations.pyx:31)
// Reference kernel: tools/projections/_kernels.pyx:15-19 (M4 cubic spline, 1/(pi h^3)).
#pragma once
#if defined(__CUDACC__)
#include <cuda_runtime.h>
#else
struct float2 { float x, y; };
#endif
#include "ast_geom.h"

namespace ast {

constexpr double kPi = 3.14159265358979323846;

enum : int { SHAPE_CUBIC = 0, SHAPE_WENDLAND = 1, SHAPE_TABLE = 2 };

// tabulated shape f(q) on q in [0,2]: n intervals, entry j = {f(q_j), f(q_j+1) - f(q_j)}, q_j = 2j/n (device pointer)
struct ShapeTab {
    const float2 *tab;
    float scale;      // n / 2
    int n;
};

AST_HD bool kernel_valid(int kid) { return kid >= 0 && kid <= 4; }     // 4 = AST_KERNEL_TABLE (deposition only)
AST_HD int kernel_shape(int kid) { return kid == 4 ? SHAPE_TABLE : ((kid == 1 || kid == 2) ? SHAPE_WENDLAND : SHAPE_CUBIC); }

// norm(h) for the shape functions below
AST_HD double kernel_norm(int kid, double h)
{
    switch (kid) {
    case 0: return 1.0 / (kPi * h * h * h);                 // cubic spline, 3-D normalisation (reference)
    case 1: return 7.0 / (4.0 * kPi * h * h);               // Wendland C2, 7/(pi (2h)^2)
    case 2: return 21.0 / (16.0 * kPi * h * h * h);         // Wendland C2, 21/(2 pi (2h)^3)
    default: return 10.0 / (7.0 * kPi * h * h);             // cubic spline, 2-D normalisation
    }
}

// float64 evaluation, same expression tree as the reference for the cubic spline (pow(q,2) -> q*q etc.)
AST_HD double kernel_f64(int kid, double r, double h)
{
    double q = r / h;
    if (kernel_shape(kid) == SHAPE_CUBIC) {
        double n = kernel_norm(kid, h);
        if (q < 1.0) return (1.0 - 1.5 * (q * q) + 0.75 * (q * q * q)) * n;
        if (q < 2.0) { double t = 2.0 - q; return 0.25 * (t * t * t) * n; }
        return 0.0;
    }
    double u = 0.5 * q;
    if (!(u < 1.0)) return 0.0;
    double t = 1.0 - u;
    t = t * t;
    t = t * t;
    return kernel_norm(kid, h) * t * (1.0 + 4.0 * u);
}

#if defined(__CUDACC__)
// float32 shape functions for the deposition kernels.  Branch-free: the clamps are the .SAT modifier of the
// producing FADD/FFMA, so q >= 2 gives exactly 0 and the piecewise cubic needs no select.
//   cubic:    f(q) = 0.25 [ (2-q)+^3 - 4 (1-q)+^3 ] = 2 a^3 - b^3,  a = sat(1 - q/2), b = sat(1 - q)
//   wendland: f(q) = (1-u)^4 (1+4u), u = q/2        = a^4 (1 + 2q)
__device__ __forceinline__ float shape_cubic(float q)
{
    float a = __saturatef(fmaf(q, -0.5f, 1.0f));
    float b = __saturatef(1.0f - q);
    float a3 = a * a * a;
    float b3 = b * b * b;
    return fmaf(2.0f, a3, -b3);
}
__device__ __forceinline__ float shape_wendland(float q)
{
    float a = __saturatef(fmaf(q, -0.5f, 1.0f));
    float a2 = a * a;
    return (a2 * a2) * fmaf(q, 2.0f, 1.0f);
}
// linear interpolation in the table; exactly 0 for q >= 2 (the reference's hard mask)
__device__ __forceinline__ float shape_table(float q, const ShapeTab &t)
{
    const float x = q * t.scale;
    const int j = min((int)x, t.n - 1);
    const float2 e = __ldg(t.tab + j);
    return q < 2.0f ? fmaf(x - (float)j, e.y, e.x) : 0.0f;
}
template <int SHAPE>
__device__ __forceinline__ float shape_eval(float q, const ShapeTab &t)
{
    return SHAPE == SHAPE_CUBIC ? shape_cubic(q) : (SHAPE == SHAPE_WENDLAND ? shape_wendland(q) : shape_table(q, t));
}
__device__ __forceinline__ float fast_sqrt(float x)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// Deposition-loop forms taking s = q^2 and returning f/2 for the cubic spline (the factor 2 is folded into the weights at
// staging time) and f for the other shapes:
//   cubic: f/2 = min(1/2 + s (3q/8 - 3/4), sat(1 - q/2)^3).  The first argument is the inner branch 1 - 3/2 q^2 + 3/4 q^3 of
//   _kernels.pyx:17 (halved), the second the outer branch 1/4 (2-q)^3 of :19 (halved); inner - outer = -(1-q)^3 / 2 changes
//   sign exactly at q = 1, so the minimum selects the right branch, and it is exactly 0 beyond q = 2.
template <int SHAPE>
__device__ __forceinline__ float shape_half_full(float s, const ShapeTab &tab)
{
    const float q = fast_sqrt(s);
    if (SHAPE == SHAPE_CUBIC) {
        const float p = fmaf(s, fmaf(0.375f, q, -0.75f), 0.5f);
        const float a1 = __saturatef(fmaf(q, -0.5f, 1.0f));
        return fminf(p, a1 * a1 * a1);
    }
    return shape_eval<SHAPE>(q, tab);
}
// cubic spline, inner region only (every q < 1): f/2 = 1/2 + s (3q/8 - 3/4)   (_kernels.pyx:17, halved)
__device__ __forceinline__ float shape_half_inner(float s)
{
    return fmaf(s, fmaf(0.375f, fast_sqrt(s), -0.75f), 0.5f);
}
// cubic spline, outer annulus only (every q >= 1): f/2 = sat(1 - q/2)^3
__device__ __forceinline__ float shape_half_outer(float s)
{
    const float a1 = __saturatef(fmaf(fast_sqrt(s), -0.5f, 1.0f));
    return a1 * a1 * a1;
}

// The same three forms on a PAIR of pixels, for the packed float32 pipes of sm_100 (FFMA2 / FMUL2 / FADD2 through
// __ffma2_rn / __fmul2_rn / __fadd2_rn).  Each component of a packed rn operation rounds exactly like its scalar twin and the
// expression trees are those of the scalar forms, so every value is bit-identical to them.  There is no packed square root
// and no packed saturate or minimum: MUFU.SQRT, FFMA.SAT and FMNMX stay scalar.  Shapes other than the cubic spline go
// through the scalar form component by component.
__device__ __forceinline__ float2 f2(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 fast_sqrt2(float2 s) { return make_float2(fast_sqrt(s.x), fast_sqrt(s.y)); }
__device__ __forceinline__ float2 half_outer_of_q2(float2 q)          // sat(1 - q/2)^3
{
    const float2 a1 = make_float2(__saturatef(fmaf(q.x, -0.5f, 1.0f)), __saturatef(fmaf(q.y, -0.5f, 1.0f)));
    return __fmul2_rn(__fmul2_rn(a1, a1), a1);
}
template <int SHAPE>
__device__ __forceinline__ float2 shape_half_full2(float2 s, const ShapeTab &tab)
{
    if (SHAPE == SHAPE_CUBIC) {
        const float2 q = fast_sqrt2(s);
        const float2 p = __ffma2_rn(s, __ffma2_rn(f2(0.375f), q, f2(-0.75f)), f2(0.5f));
        const float2 o = half_outer_of_q2(q);
        return make_float2(fminf(p.x, o.x), fminf(p.y, o.y));
    }
    return make_float2(shape_half_full<SHAPE>(s.x, tab), shape_half_full<SHAPE>(s.y, tab));
}
__device__ __forceinline__ float2 shape_half_inner2(float2 s)
{
    return __ffma2_rn(s, __ffma2_rn(f2(0.375f), fast_sqrt2(s), f2(-0.75f)), f2(0.5f));
}
__device__ __forceinline__ float2 shape_half_outer2(float2 s)
{
    return half_outer_of_q2(fast_sqrt2(s));
}
#endif

}  // namespace ast
