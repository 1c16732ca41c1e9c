// hop_dynamics.cuh -- device twins of the reference's dynamics closures F(x, u) (systems.py).
//
// A Python closure cannot be called from a kernel, so each benchmark system is a device function
// selected by a compile-time id (include/hop_b200.h HOP_SYS_*) and fed a parameter vector.
// Products and sums are written with the unfused helpers below so that the rounding matches the
// scalar Python arithmetic of the reference (nvcc would otherwise contract a*b+c into an FMA);
// sin/cos/tan are CUDA's (<= 2 ulp), the only source of last-bit differences in F.
#pragma once
#include <math.h>

#include "hop_select_body.cuh"   // wrap_pi, HOP_DEVICE

namespace hop {

#if defined(__CUDA_ARCH__)
HOP_DEVICE double mul(double a, double b) { return __dmul_rn(a, b); }
HOP_DEVICE double add(double a, double b) { return __dadd_rn(a, b); }
HOP_DEVICE double sub(double a, double b) { return __dsub_rn(a, b); }
#else
HOP_DEVICE double mul(double a, double b) { volatile double r = a * b; return r; }
HOP_DEVICE double add(double a, double b) { volatile double r = a + b; return r; }
HOP_DEVICE double sub(double a, double b) { volatile double r = a - b; return r; }
#endif

template <int SYS> struct SysDims;
template <> struct SysDims<0> { static constexpr int n = 2, m = 1; };
template <> struct SysDims<1> { static constexpr int n = 4, m = 1; };
template <> struct SysDims<2> { static constexpr int n = 12, m = 4; };
template <> struct SysDims<3> { static constexpr int n = 4, m = 1; };

template <int SYS>
HOP_DEVICE void dynamics(const double* p, const double* x, const double* u, double* xn);

// systems.py:30-33
template <>
HOP_DEVICE void dynamics<0>(const double* p, const double* x, const double* u, double* xn) {
    const double dt = p[0];
    const double a = add(x[0], mul(dt, x[1])), b = add(x[1], mul(dt, u[0]));
    xn[0] = a; xn[1] = b;
}
// systems.py:72-95
template <>
HOP_DEVICE void dynamics<1>(const double* p, const double* x, const double* u, double* xn) {
    const double dt = p[0], g = p[1], m_pole = p[2], length = p[3], total = p[4], pml = p[5];
    const double pos = x[0], vel = x[1], th = x[2], om = x[3], force = u[0];
    const double a = sub(th, 3.141592653589793);
    double sa, ca;
    sincos(a, &sa, &ca);
    const double tmp = add(force, mul(mul(mul(pml, om), om), sa)) / total;
    const double den = mul(length, sub(4.0 / 3.0, mul(mul(m_pole, ca), ca) / total));
    const double th_acc = sub(mul(g, sa), mul(ca, tmp)) / den;
    const double x_acc = sub(tmp, mul(mul(pml, th_acc), ca) / total);
    const double n0 = add(pos, mul(dt, vel)), n1 = add(vel, mul(dt, x_acc));
    const double n2 = wrap_pi(add(th, mul(dt, om))), n3 = add(om, mul(dt, th_acc));
    xn[0] = n0; xn[1] = n1; xn[2] = n2; xn[3] = n3;
}
// systems.py:321-333
template <>
HOP_DEVICE void dynamics<3>(const double* p, const double* x, const double* u, double* xn) {
    const double dt = p[0], a_tau = p[1], a_th = p[2], b_tau = p[3], b_th = p[4];
    const double pos = x[0], vel = x[1], th = x[2], om = x[3], tau = u[0];
    const double acc = add(mul(a_tau, tau), mul(a_th, th));
    const double alp = add(mul(b_tau, tau), mul(b_th, th));
    const double n0 = add(pos, mul(dt, vel)), n1 = add(vel, mul(dt, acc));
    const double n2 = wrap_pi(add(th, mul(dt, om))), n3 = add(om, mul(dt, alp));
    xn[0] = n0; xn[1] = n1; xn[2] = n2; xn[3] = n3;
}
// systems.py:170-210 (rotm :145-156, Tmat :158-163, guards :175-191), split so that the finite-difference
// kernel can share the trigonometry of the unperturbed angles between the 16 perturbed evaluations of a (problem, step);
// dynamics<2> below and k_linearize_quad_row evaluate exactly the same operation sequence.
struct QuadTrig { double sph, cph, sth, cth, tth, sps, cps; };

// the guards that do not need trigonometry (systems.py:175-183,188-191)
HOP_DEVICE bool quad_guard(const double* p, const double* x, const double* u) {
    const double wmax = p[12], nmax = p[13];
    bool bad = false;
    double ss = 0.0;
#pragma unroll
    for (int i = 0; i < 12; ++i) { bad = bad || !isfinite(x[i]); ss = add(ss, mul(x[i], x[i])); }
#pragma unroll
    for (int i = 0; i < 4; ++i) bad = bad || !isfinite(u[i]);
    bad = bad || (sqrt(ss) > nmax);
    return bad || (fabs(x[9]) > wmax) || (fabs(x[10]) > wmax) || (fabs(x[11]) > wmax);
}

HOP_DEVICE void quad_core(const double* p, const double* x, const double* u, const QuadTrig& T, double* xn) {
    const double dt = p[0], mass = p[1], g = p[2], Ix = p[3], Iy = p[4], Iz = p[5];
    const double iIx = p[6], iIy = p[7], iIz = p[8], kv = p[9], kw = p[10];
    const double wp = x[9], wq = x[10], wr = x[11];
    const double sph = T.sph, cph = T.cph, sth = T.sth, cth = T.cth, sps = T.sps, cps = T.cps;
    const double tth = T.tth, sec = 1.0 / cth, thrust = u[0];
    const double r02 = add(mul(-sps, -sph), mul(mul(cps, sth), cph));
    const double r12 = add(mul(cps, -sph), mul(mul(sps, sth), cph));
    const double r22 = mul(cth, cph);
    double xd[12];
    xd[0] = x[3]; xd[1] = x[4]; xd[2] = x[5];
    xd[3] = sub(sub(mul(r02, thrust) / mass, 0.0), mul(kv, x[3]));
    xd[4] = sub(sub(mul(r12, thrust) / mass, 0.0), mul(kv, x[4]));
    xd[5] = sub(sub(mul(r22, thrust) / mass, g), mul(kv, x[5]));
    xd[6] = add(add(wp, mul(mul(sph, tth), wq)), mul(mul(cph, tth), wr));
    xd[7] = add(mul(cph, wq), mul(-sph, wr));
    xd[8] = add(mul(mul(sph, sec), wq), mul(mul(cph, sec), wr));
    const double h0 = mul(Ix, wp), h1 = mul(Iy, wq), h2 = mul(Iz, wr);
    xd[9] = sub(mul(iIx, sub(u[1], sub(mul(wq, h2), mul(wr, h1)))), mul(kw, wp));
    xd[10] = sub(mul(iIy, sub(u[2], sub(mul(wr, h0), mul(wp, h2)))), mul(kw, wq));
    xd[11] = sub(mul(iIz, sub(u[3], sub(mul(wp, h1), mul(wq, h0)))), mul(kw, wr));
#pragma unroll
    for (int i = 0; i < 12; ++i) xn[i] = add(x[i], mul(dt, xd[i]));
}

template <>
HOP_DEVICE void dynamics<2>(const double* p, const double* x, const double* u, double* xn) {
    bool bad = quad_guard(p, x, u);
    QuadTrig T;
    sincos(x[7], &T.sth, &T.cth);
    bad = bad || (fabs(T.cth) < p[11]);
    if (bad) {
#pragma unroll
        for (int i = 0; i < 12; ++i) xn[i] = nan("");
        return;
    }
    sincos(x[6], &T.sph, &T.cph);
    sincos(x[8], &T.sps, &T.cps);
    T.tth = tan(x[7]);
    quad_core(p, x, u, T, xn);
}

}  // namespace hop
