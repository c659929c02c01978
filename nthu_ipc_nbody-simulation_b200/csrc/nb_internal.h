// Internal declarations shared by the translation units of libnbody_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <memory>
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

// Owners of CUDA resources: move-only, and an empty owner frees nothing.  g_leak_on_exit is set by nb_hw5_main: the
// process leaves through _exit right after the output file is written, so device buffers, pinned mailboxes and streams
// are not torn down one by one (cudaFree / cudaFreeHost cost up to 0.7 s there); while it is set the deleters free nothing.
extern std::atomic<bool> g_leak_on_exit;
template <auto Free>
struct Deleter {
    template <class P>
    void operator()(P p) const {
        if (!g_leak_on_exit.load()) Free(p);
    }
};
template <class T> using DeviceMem = std::unique_ptr<T, Deleter<cudaFree>>;
template <class T> using PinnedMem = std::unique_ptr<T, Deleter<cudaFreeHost>>;
using Stream = std::unique_ptr<CUstream_st, Deleter<cudaStreamDestroy>>;
using Event = std::unique_ptr<CUevent_st, Deleter<cudaEventDestroy>>;
using SymHandle = std::unique_ptr<nb_sym, Deleter<nb_sym_destroy>>;

// Fill an owner; on failure it is left empty.  Call them through NB_CUDA.
template <class T>
cudaError_t alloc(DeviceMem<T>& p, size_t bytes) {
    void* raw = nullptr;
    const cudaError_t e = cudaMalloc(&raw, bytes);
    p.reset(e == cudaSuccess ? (T*)raw : nullptr);
    return e;
}
template <class T>
cudaError_t alloc(PinnedMem<T>& p, size_t bytes) {
    void* raw = nullptr;
    const cudaError_t e = cudaHostAlloc(&raw, bytes, cudaHostAllocDefault);
    p.reset(e == cudaSuccess ? (T*)raw : nullptr);
    return e;
}
inline cudaError_t create(Stream& s) {  // non-blocking: no implicit ordering with the legacy default stream
    cudaStream_t raw = nullptr;
    const cudaError_t e = cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking);
    s.reset(e == cudaSuccess ? raw : nullptr);
    return e;
}
inline cudaError_t create(Event& ev, unsigned flags = cudaEventDefault) {
    cudaEvent_t raw = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&raw, flags);
    ev.reset(e == cudaSuccess ? raw : nullptr);
    return e;
}

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

// nb_diag.cu: the diagnostics of S systems of n bodies (device arrays laid out as nb_diagnostics' host arrays) with the
// masses of the step whose |sin| is fst; out = [S][9] doubles {mass, kinetic, potential, P[3], L[3]}.  Tile edge DIAG_T.
constexpr int DIAG_T = 256;
size_t diag_scratch_bytes(int S, int n);
int diag_launch(int S, int n, const double* q, const double* v, const double* m, const unsigned char* is_device, double fst,
                void* scratch, double* out, cudaStream_t stream);
// |sin(step*dt/6000)| of any step >= 0, the expression the table is built with
double fst_at(int step);

// nb_ens.cu: ensembles of n > NB_MAX_SMALL_N bodies, G systems stepped by one launch per kernel.  A system's records are
// pos4 + (parity * G + g) * n_pad (parity = step & 1), its partial accelerations slots + g * n_slots * 3 * n_pad.
struct EnsGroup {
    const TrajDesc* descs;  // [G] device
    double4* pos4;          // [2][G][n_pad] {x, y, z, G*m_eff}; bodies n .. n_pad-1 zero
    double* slots;          // [G][n_slots][3][n_pad]
    int n, n_pad, n_slots, G;
};
int ens_pad(int n);              // bodies per system record buffer: whole tiles
int ens_slots(int math, int n);  // partial-acceleration slots per body
// step `step` (reads the records of step - 1, writes those of step): the pair kernel and the integrate kernel
int ens_step(int math, const EnsGroup& e, int step, cudaStream_t stream);
// the observers of step `step` on its records, one warp per system
int ens_observe(const EnsGroup& e, int step, cudaStream_t stream);

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
