// Internal declarations shared by the translation units of libnbody_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <string>

#include "../../include/nbody_b200.h"

namespace nb {

// One trajectory (one system) as the persistent kernels see it.  All pointers are device pointers.
struct TrajDesc {
    int n, planet, asteroid, kind;
    int destroy_device, step_begin, step_end, n_dev;
    double* q;                       // [3n] planar, in/out
    double* v;                       // [3n] planar, in/out
    double* m;                       // [n] base masses, in/out (a destroyed device is zeroed)
    const unsigned char* is_device;  // [n]
    const int* dev_index;            // [n_dev] body indexes of the devices, ascending
    nb_events* ev;                   // in/out
};

// error plumbing -------------------------------------------------------------------------------
void set_error_detail(const std::string& s);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
#define NB_CUDA(call)                                                        \
    do {                                                                     \
        cudaError_t _e = (call);                                             \
        if (_e != cudaSuccess) return nb::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)

void count_launch(int n = 1);
// nb_profile_enable / nb_profile_read (nb_large.cu): event pairs around the acceleration kernel, calling thread only
bool profile_on();
void profile_push(cudaEvent_t e0, cudaEvent_t e1);
// nb_large.cu: stream-ordered wait until counters[0 .. count) all reach target; a wait that times out writes code to *status
int launch_counter_wait(const unsigned long long* counters, int count, unsigned long long target, int* status, int code,
                        cudaStream_t stream);
// nb_large.cu: the observers of step `step` of trajectory d on the pos4 records [n][4] the step's integrate kernel wrote
int launch_large_observe(const TrajDesc& d, double* pos4_dev, int step, cudaStream_t stream);
// nb_sym.cu: forget the steps of a one-rank handle, so that its next step may be any step (positions repacked by the caller)
int sym_restart(nb_sym* h);

// per-GPU |sin(step*dt/6000)| table (host glibc sin: nbody.cc:14-16 with t = step*dt, nbody.cc:63),
// entries 0..len-1, built lazily and grown on demand.  Returns a device pointer valid for the
// life of the process.
int fst_table(int gpu, int min_len, const double** table_dev);
double fst_value(int step);

// nb_traj.cu: n_traj single-block persistent trajectories of the same n in one launch
int launch_traj_batch(int math, int n, int n_traj, const TrajDesc* descs_dev, const double* fst_dev,
                      cudaStream_t stream);
int traj_js_for(int math, int n);

// nb_grid.cu: one trajectory batch spread over the whole GPU (cooperative persistent kernel)
int launch_grid_traj(int math, int n, int n_traj, const TrajDesc* descs_dev, const double* fst_dev, int gpu,
                     void* workspace_dev, size_t workspace_bytes, cudaStream_t stream);
size_t grid_traj_workspace_bytes(int n);
const int* grid_traj_status(const void* workspace_dev, int n);  // sticky status word, read it once the stream is idle
bool grid_traj_supported(int gpu, int n);
void grid_traj_warm();  // loads the kernels' module on the current device (lazy loading would do it at the first launch)

}  // namespace nb
