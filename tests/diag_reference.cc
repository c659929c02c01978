// Long-double reference of the diagnostics (include/nbody_b200.h nb_diag) — TEST INFRASTRUCTURE ONLY.
//
// diag_reference(n, q, v, m, is_device, step, nthreads, out[9]) = {mass, kinetic, potential, P[3], L[3]} of one state with
// the effective masses of `step` (m0 + 0.5*m0*|sin(step*dt/6000)| for gravity devices, |sin| the library's host glibc
// expression).  Every term in long double, every sum compensated (Neumaier).  The pair sum is split into rows i (OpenMP
// when built with it); the row sums are added in ascending i, so the result does not depend on nthreads.
// Built by tests/diag_reference.py: g++ -O2 -std=c++17 -ffp-contract=off [-fopenmp] -shared -fPIC.
#include <cmath>
#include <vector>

namespace {

// nbody.cc:9-20
const double dt = 60;
const double eps = 1e-3;
const double G = 6.674e-11;

struct NeumaierSum {
    long double s = 0, c = 0;
    void add(long double x) {
        const long double t = s + x;
        c += fabsl(s) >= fabsl(x) ? (s - t) + x : (x - t) + s;
        s = t;
    }
    long double value() const { return s + c; }
};

}  // namespace

extern "C" int diag_reference(int n, const double* q, const double* v, const double* m, const unsigned char* is_device,
                              int step, int nthreads, long double* out) {
    if (n <= 0 || !q || !v || !m || !is_device || !out || step < 0) return -1;
    const long double fst = fabs(sin((step * dt) / 6000));  // the library's |sin| expression (nb_host.cu fst_at)
    std::vector<long double> me(n), row(n);
    for (int i = 0; i < n; i++) me[i] = is_device[i] ? (long double)m[i] + 0.5L * m[i] * fst : (long double)m[i];
    const double* x = q;
    const double* y = q + n;
    const double* z = q + 2 * n;
    const long double eps2 = (long double)eps * eps;
    (void)nthreads;
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads) if (nthreads > 1)
    for (int i = 0; i < n; i++) {
        NeumaierSum r;
        for (int j = i + 1; j < n; j++) {
            const long double dx = (long double)x[j] - x[i], dy = (long double)y[j] - y[i], dz = (long double)z[j] - z[i];
            r.add(me[j] / sqrtl(dx * dx + dy * dy + dz * dz + eps2));
        }
        row[i] = me[i] * r.value();
    }
    NeumaierSum mass, kin, pot, p[3], l[3];
    for (int i = 0; i < n; i++) {
        const long double vx = v[i], vy = v[i + n], vz = v[i + 2 * n], xi = x[i], yi = y[i], zi = z[i], w = me[i];
        mass.add(w);
        kin.add(w * (vx * vx + vy * vy + vz * vz));
        pot.add(row[i]);
        p[0].add(w * vx), p[1].add(w * vy), p[2].add(w * vz);
        // each cross-product component as its two products, so that the compensation sees every term
        l[0].add(w * yi * vz), l[0].add(-(w * zi * vy));
        l[1].add(w * zi * vx), l[1].add(-(w * xi * vz));
        l[2].add(w * xi * vy), l[2].add(-(w * yi * vx));
    }
    out[0] = mass.value();
    out[1] = 0.5L * kin.value();
    out[2] = -(long double)G * pot.value();
    for (int c = 0; c < 3; c++) out[3 + c] = p[c].value(), out[6 + c] = l[c].value();
    return 0;
}
