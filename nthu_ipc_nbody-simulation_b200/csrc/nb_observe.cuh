// The in-kernel observers of one trajectory, shared by traj_kernel, traj_sym_kernel (nb_traj.cu), the observer warp of
// grid_traj_kernel (nb_grid.cu) and large_observe_kernel (nb_large.cu, n > 1024): minimum distance, missile reach, hit test and the Q3 destroy (hw5.cu:241-309), and the
// gravity devices' mass rule.  Every comparison is the reference's un-contracted arithmetic (dist2_rn), so the discrete
// outputs do not depend on the math mode.
#pragma once
#include "nb_internal.h"
#include "nb_math.cuh"

namespace nb {

// The scalar events of a trajectory while a kernel runs; device reach steps are kept by the threads that own the devices.
struct Observed {
    double min_d2;
    int argmin_step;
    int hit_step;
    int destroyed_step;
    double cost;

    __device__ __forceinline__ void load(const nb_events* ev) {
        min_d2 = ev->min_d2;
        argmin_step = ev->argmin_step;
        hit_step = ev->hit_step;
        destroyed_step = ev->destroyed_step;
        cost = ev->cost;
    }
    // one thread per trajectory: the events, the last step observed, and the destroyed device's mass (hw5.cu:306)
    __device__ __forceinline__ void store(const TrajDesc& d, int steps_done) const {
        d.ev->min_d2 = min_d2;
        d.ev->argmin_step = argmin_step;
        d.ev->hit_step = hit_step;
        d.ev->destroyed_step = destroyed_step;
        d.ev->cost = cost;
        d.ev->steps_done = steps_done;
        d.ev->n_reach = d.n_dev;
        if (d.kind == NB_KIND_Q3 && destroyed_step != -2) d.m[d.destroy_device] = 0.0;
    }
};

constexpr int OBS_HIT = 1, OBS_DESTROYED = 2;  // observe_step's result

// Q3: the destroy test runs only for a device that exists and still has mass (hw5.cu:299).
__device__ __forceinline__ bool q3_armed(int kind, int DD, int n, const double* m) {
    return (kind == NB_KIND_Q3) && DD >= 0 && DD < n && m[DD] != 0.0;
}

// G*m_eff of gravity device `dev` at `step` (nbody.cc:14-16, 61-64): 0 once it is the destroyed Q3 device.  It reads the
// table entry and the destroyed step itself, where the rule uses them: passed in as values, they move instructions of
// the traj kernels (measured in their SASS).
__device__ __forceinline__ double device_gm(int kind, int dev, int DD, const Observed& ob, double m0, const double* fst, int step) {
    const bool gone = (kind == NB_KIND_Q3) && dev == DD && ob.destroyed_step != -2;
    return gm_eff(gone ? 0.0 : m0, true, fst[step]);
}

// The missile, fired at step 0, has reached body (dx, dy, dz) from the planet at step st (hw5.cu:265-287).
__device__ __forceinline__ bool missile_reaches(double px, double py, double pz, double dx, double dy, double dz, int st) {
    const double md = __dmul_rn(MISSILE_STEP, (double)st);
    return dist2_rn(px, py, pz, dx, dy, dz) < __dmul_rn(md, md);
}

// The observers of step st, in the reference's order: minimum distance, the Q2 reach of the ND devices this thread looks
// after (my_dev[h] < 0: none), then the hit test, else the Q3 destroy.  rec(i, x, y, z) reads body i's position at st.
// Returns OBS_HIT, OBS_DESTROYED (this step) or 0.
template <int ND, class Rec>
__device__ __forceinline__ int observe_step(Observed& ob, int st, int kind, int P, int A, bool armed, int DD,
                                            const int* my_dev, int* my_reach, Rec rec) {
    double px, py, pz, ax, ay, az;
    rec(P, px, py, pz);
    rec(A, ax, ay, az);
    const double d2 = dist2_rn(px, py, pz, ax, ay, az);
    if (d2 < ob.min_d2) {  // hw5.cu:245-247
        ob.min_d2 = d2;
        ob.argmin_step = st;
    }
#pragma unroll
    for (int h = 0; h < ND; h++)
        if (kind == NB_KIND_Q2 && my_dev[h] >= 0 && my_reach[h] == -2) {  // before the hit test (hw5.cu:396-397)
            double dx, dy, dz;
            rec(my_dev[h], dx, dy, dz);
            if (missile_reaches(px, py, pz, dx, dy, dz, st)) my_reach[h] = st;
        }
    if (kind >= NB_KIND_Q2) {
        if (d2 < PLANET_RADIUS2) {  // nbody.cc:134, hw5.cu:295-298
            ob.hit_step = st;
            return OBS_HIT;
        } else if (armed && ob.destroyed_step == -2) {  // hw5.cu:299-307
            double dx, dy, dz;
            rec(DD, dx, dy, dz);
            if (missile_reaches(px, py, pz, dx, dy, dz, st)) {
                ob.destroyed_step = st;
                ob.cost = __dadd_rn(1e5, __dmul_rn(1e3, __dmul_rn((double)(st + 1), DT)));
                return OBS_DESTROYED;
            }
        }
    }
    return 0;
}

}  // namespace nb
