// Pair arithmetic shared by every kernel of the path.
//
// Reference: samples/nbody.cc:56-74 (the pair term), :9-20 (constants); hw5.cu:200-213 (the
// sqrt(r2^3) form).  Two variants:
//   STRICT  IEEE-only, explicitly rounded intrinsics (never contracted to FMA):
//           r2 = ((dx*dx + dy*dy) + dz*dz) + eps*eps; dist3 = sqrt((r2*r2)*r2);
//           a += ((G*mj)*d) / dist3         -> bit-identical to the CPU oracle's SQRT3 mode
//   FAST    16 FP64-pipe instructions per pair, no IEEE div/sqrt:
//           r2 by an FMA chain, y0 = rsqrt.approx.ftz.f64(r2) (MUFU.RSQ64H, ~2^-20),
//           e = 1 - r2*y0^2, r2^-3/2 = y0^3 * (1 + 1.5e + 1.875e^2) (truncation ~ |e|^3*2.2 < 2^-55),
//           a = fma(c, d, a).
#pragma once
#include <cuda_runtime.h>

namespace nb {

constexpr double DT = 60.0;
constexpr double EPS = 1e-3;
constexpr double EPS2 = EPS * EPS;  // param::eps * param::eps, folded exactly as the host compiler does
constexpr double G = 6.674e-11;
constexpr double PLANET_RADIUS = 1e7;
constexpr double PLANET_RADIUS2 = PLANET_RADIUS * PLANET_RADIUS;
constexpr double MISSILE_SPEED = 1e6;
constexpr double MISSILE_STEP = MISSILE_SPEED * DT;  // hw5.cu:273 (param::missile_speed * param::dt)

constexpr int MATH_FAST = 0;
constexpr int MATH_STRICT = 1;

__device__ __forceinline__ double rsqrt_seed(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}

// G * m_eff of a body at a step: nbody.cc:14-16 with t = step*dt folded into fst = |sin(step*dt/6000)|
// (host glibc table), then the first product of `G * mj * dx / dist3` (nbody.cc:70) hoisted.
__device__ __forceinline__ double gm_eff(double m0, bool is_device, double fst) {
    double mj = m0;
    if (is_device) mj = __dadd_rn(m0, __dmul_rn(__dmul_rn(0.5, m0), fst));
    return __dmul_rn(G, mj);
}

// d^2 between two bodies, evaluated exactly like nbody.cc:131-134 / hw5.cu:255-259 (no FMA), so
// that the discrete observers do not depend on the math mode.
__device__ __forceinline__ double dist2_rn(double ax, double ay, double az, double bx, double by, double bz) {
    double dx = __dsub_rn(ax, bx), dy = __dsub_rn(ay, by), dz = __dsub_rn(az, bz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

template <int MATH>
__device__ __forceinline__ void pair(double xi, double yi, double zi, double xj, double yj, double zj, double gmj,
                                     double& ax, double& ay, double& az) {
    if (MATH == MATH_STRICT) {
        double dx = __dsub_rn(xj, xi), dy = __dsub_rn(yj, yi), dz = __dsub_rn(zj, zi);
        double r2 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)), EPS2);
        double dist3 = __dsqrt_rn(__dmul_rn(__dmul_rn(r2, r2), r2));
        ax = __dadd_rn(ax, __ddiv_rn(__dmul_rn(gmj, dx), dist3));
        ay = __dadd_rn(ay, __ddiv_rn(__dmul_rn(gmj, dy), dist3));
        az = __dadd_rn(az, __ddiv_rn(__dmul_rn(gmj, dz), dist3));
    } else {
        double dx = xj - xi, dy = yj - yi, dz = zj - zi;
        double r2 = fma(dx, dx, fma(dy, dy, fma(dz, dz, EPS2)));
        double y0 = rsqrt_seed(r2);
        double y2 = y0 * y0;
        double e = fma(-r2, y2, 1.0);
        double p = fma(e, fma(e, 1.875, 1.5), 1.0);
        double c = (gmj * y0) * (y2 * p);
        // The three accumulates share the multiplicand c.  A DFMA that reads three distinct register
        // pairs costs 3 pipe cycles instead of 2 on B200 (measured: nb_fp64_peak_variant 1 = 24.8 of
        // 37.1 TFLOP/s); when ptxas keeps the triple adjacent it marks c ".reuse" for the 2nd and 3rd.
        ax = fma(c, dx, ax);
        ay = fma(c, dy, ay);
        az = fma(c, dz, az);
    }
}

// FAST pair term split in two, so that a kernel can first compute the coefficients of several pairs and then
// issue all their accumulate DFMAs back to back (three per pair, sharing the multiplicand c: see pair<>).
__device__ __forceinline__ void pair_coeff_fast(double xi, double yi, double zi, double xj, double yj, double zj,
                                                double gmj, double& c, double& dx, double& dy, double& dz) {
    dx = xj - xi, dy = yj - yi, dz = zj - zi;
    const double r2 = fma(dx, dx, fma(dy, dy, fma(dz, dz, EPS2)));
    const double y0 = rsqrt_seed(r2);
    const double y2 = y0 * y0;
    const double e = fma(-r2, y2, 1.0);
    const double p = fma(e, fma(e, 1.875, 1.5), 1.0);
    c = (gmj * y0) * (y2 * p);
}
__device__ __forceinline__ void pair_accum_fast(double c, double dx, double dy, double dz, double& ax, double& ay,
                                                double& az) {
    ax = fma(c, dx, ax);
    ay = fma(c, dy, ay);
    az = fma(c, dz, az);
}

// FAST, one UNORDERED pair: s = |d|^-3 as in pair<> (rsqrt seed + cubic correction), both accelerations (nb_sym.cu,
// traj_sym_kernel)
__device__ __forceinline__ void pair_sym(double xi, double yi, double zi, double gmi, double xj, double yj, double zj,
                                         double gmj, double& aix, double& aiy, double& aiz, double& ajx, double& ajy,
                                         double& ajz) {
    const double dx = xj - xi, dy = yj - yi, dz = zj - zi;
    const double r2 = fma(dx, dx, fma(dy, dy, fma(dz, dz, EPS2)));
    const double y0 = rsqrt_seed(r2);
    const double y2 = y0 * y0;
    const double e = fma(-r2, y2, 1.0);
    const double p = fma(e, fma(e, 1.875, 1.5), 1.0);
    const double s = y0 * (y2 * p);
    const double ci = gmj * s, cj = gmi * s;
    aix = fma(ci, dx, aix);
    aiy = fma(ci, dy, aiy);
    aiz = fma(ci, dz, aiz);
    ajx = fma(-cj, dx, ajx);
    ajy = fma(-cj, dy, ajy);
    ajz = fma(-cj, dz, ajz);
}

// v += a*dt; q += v*dt (nbody.cc:77-88, hw5.cu:235-236).  O(n) per step, so both math modes keep
// the reference's four separate roundings (no FMA): the state update is then exactly run_step's.
__device__ __forceinline__ void kick_drift(double a, double& v, double& q) {
    v = __dadd_rn(v, __dmul_rn(a, DT));
    q = __dadd_rn(q, __dmul_rn(v, DT));
}

}  // namespace nb
