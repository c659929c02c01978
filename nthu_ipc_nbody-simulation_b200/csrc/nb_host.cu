// C ABI of libnbody_b200.so: device plumbing, trajectory handles, ensembles, the three-query
// driver and its ensemble scheduler.  Host code is C++ in the .cu translation unit, as the
// reference's is (hw5.cu:311-616); the kernels live in nb_traj.cu / nb_grid.cu / nb_large.cu.
#include <atomic>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "nb_internal.h"

namespace nb {

// ---- errors / counters ---------------------------------------------------------------------------
static thread_local std::string g_detail;
void set_error_detail(const std::string& s) { g_detail = s; }
int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s:%d)", cudaGetErrorString(e), what, file, line);
    g_detail = buf;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice) return NB_ERR_NO_GPU;
    return NB_ERR_CUDA;
}
static std::atomic<long long> g_launches{0};
// set by nb_hw5_main: the process leaves through _exit right after the output file is written, so device buffers,
// pinned mailboxes and streams are not torn down one by one (cudaFree / cudaFreeHost cost up to 0.7 s there)
std::atomic<bool> g_leak_on_exit{false};
static std::atomic<long long> g_torn_records{0};
void count_launch(int n) { g_launches += n; }

// ---- |sin(step*dt/6000)| table ----------------------------------------------------------------------
// nbody.cc:14-16 with t = step*dt (nbody.cc:63): fabs(sin((step*60.0)/6000)), host glibc sin, so the
// modulation is the oracle's to the bit whatever the device sin() does.  (The reference's own table,
// hw5.cu:143-148,555, is one entry short and built with the device sin.)
static std::mutex g_fst_mu;
static std::vector<double> g_fst_host;
struct FstDev {
    double* ptr = nullptr;
    int len = 0;
};
static FstDev g_fst_dev[64];

// grows the host table to at least min_len entries; call with g_fst_mu held
static void fst_grow_locked(int min_len) {
    if ((int)g_fst_host.size() < min_len) {
        int len = min_len < NB_N_STEPS + 2 ? NB_N_STEPS + 2 : min_len;
        std::vector<double> t(len);
        for (int s = 0; s < len; s++) t[s] = fabs(sin((s * NB_DT) / 6000));
        g_fst_host.swap(t);
    }
}

// one entry, by value: safe against a concurrent growth of the table by another host thread
double fst_value(int step) {
    std::lock_guard<std::mutex> lk(g_fst_mu);
    fst_grow_locked(step + 1);
    return g_fst_host[step];
}

int fst_table(int gpu, int min_len, const double** out) {
    if (gpu < 0 || gpu >= 64) return NB_ERR_ARG;
    std::lock_guard<std::mutex> lk(g_fst_mu);
    fst_grow_locked(min_len);
    FstDev& d = g_fst_dev[gpu];
    if (d.len < min_len) {
        const int len = (int)g_fst_host.size();
        double* p = nullptr;
        NB_CUDA(cudaSetDevice(gpu));
        NB_CUDA(cudaMalloc(&p, (size_t)len * sizeof(double)));
        NB_CUDA(cudaMemcpy(p, g_fst_host.data(), (size_t)len * sizeof(double), cudaMemcpyHostToDevice));
        // the old table (if any) is leaked on purpose: a running kernel may still read it
        d.ptr = p;
        d.len = len;
    }
    *out = d.ptr;
    return NB_OK;
}

static int check_gpu(int gpu) {
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) {
        (void)cudaGetLastError();
        set_error_detail(std::string("no CUDA device: ") + cudaGetErrorString(e));
        return NB_ERR_NO_GPU;
    }
    if (gpu < 0 || gpu >= cnt) {
        set_error_detail("GPU ordinal out of range");
        return NB_ERR_NO_GPU;
    }
    return NB_OK;
}

// Busy-wait for the stream (or for event e) instead of a blocking synchronize: the blocking wait costs tens of milliseconds
// of wake-up latency now and then (measured on the B200 boxes), and the chain plan of nb_solve waits every few thousand
// steps.  (round 2: spin for the first 200 us only, then poll every 20 us - a launch lasts milliseconds to seconds, and a
// host core at 100 % for all of it bought nothing)
static int spin_wait(cudaStream_t stream, cudaEvent_t e = nullptr) {
    const auto w0 = std::chrono::steady_clock::now();
    for (;;) {
        cudaError_t qe = e ? cudaEventQuery(e) : cudaStreamQuery(stream);
        if (qe == cudaSuccess) return NB_OK;
        if (qe != cudaErrorNotReady) return cuda_fail(qe, e ? "cudaEventQuery" : "cudaStreamQuery", __FILE__, __LINE__);
        if (std::chrono::steady_clock::now() - w0 > std::chrono::microseconds(200))
            std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
}

// ---- the large-N steppers, one system at a time ----------------------------------------------------------
// n > NB_MAX_SMALL_N on one GPU, all bodies local.  FAST takes the symmetric stepper (nb_sym.cu: every unordered pair once),
// STRICT the row kernel (nb_large.cu: one j split, the reference's ascending-j sum).  The stepper owns the two pos4 buffers
// [n][4], and the symmetric stepper's handle and PJ buffer or the row kernel's j-split scratch; the caller's q stays
// planar [3][n] and its v is stepped in place.  Used by nb_run_steps and by the query path (DeviceBatch::run).
struct LargeStepper {
    int n = 0, math = 0, cur = 0;  // pos[cur] holds the current step
    nb_sym* h = nullptr;
    double* pos[2] = {nullptr, nullptr};
    void* work = nullptr;

    // on the current device; the PJ zero-fill is enqueued on st
    int init(int n_, int math_, cudaStream_t st) {
        n = n_, math = math_;
        if (math == NB_MATH_FAST) {
            const int rc = nb_sym_create(n, 1, 0, &h);
            if (rc) return rc;
        }
        NB_CUDA(cudaMalloc(&pos[0], 4 * (size_t)n * sizeof(double)));
        NB_CUDA(cudaMalloc(&pos[1], 4 * (size_t)n * sizeof(double)));
        const size_t bytes = (size_t)(h ? nb_sym_pj_bytes(h) : nb_large_scratch_bytes(n, n));
        NB_CUDA(cudaMalloc(&work, bytes));
        if (h) NB_CUDA(cudaMemsetAsync(work, 0, bytes, st));  // PJ rows nobody writes are summed as zeros
        return NB_OK;
    }
    // planar positions of step step_next - 1 with the masses of step_next: the next step() is step_next, any step
    int pack(const double* q, const double* m, const unsigned char* is_device, int step_next, cudaStream_t st) {
        cur = 0;
        if (h) {
            const int rc = sym_restart(h);
            if (rc) return rc;
        }
        return nb_large_pack(math, n, q, m, is_device, step_next, pos[0], st);
    }
    int step(int s, double* v, const double* m, const unsigned char* is_device, cudaStream_t st) {
        double *next = pos[cur ^ 1], *pj = (double*)work;
        const int rc = h ? nb_sym_step(h, s, pos[cur], &next, &pj, nullptr, nullptr, v, m, is_device, st)
                         : nb_large_step(math, s, n, 0, n, pos[cur], next, v, m, is_device, work, st);
        if (!rc) cur ^= 1;
        return rc;
    }
    int unpack(double* q, cudaStream_t st) { return nb_large_unpack(n, pos[cur], q, st); }
    void release() {
        cudaFree(pos[0]), cudaFree(pos[1]), cudaFree(work);
        if (h) nb_sym_destroy(h);
        *this = LargeStepper{};
    }
};

// Steps per chunk of the query path on the large-N steppers: the host reads the events between chunks.  A step costs
// about n^2 (2.95 ms at 65 536 bodies on the B200), so 2^33 / n^2 steps, at least 4 (~12 ms at 65 536 bodies) and at most
// 512 (below ~4 096 bodies a step is bound by launch latency).
static int large_chunk(int n) {
    const long long c = (1LL << 33) / ((long long)n * n);
    return (int)std::min(512LL, std::max(4LL, c));
}

// ---- a batch of same-n systems resident on one GPU ---------------------------------------------------
struct DeviceBatch {
    int gpu = -1, S = 0, n = 0, math = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    double *q = nullptr, *v = nullptr, *m = nullptr;
    unsigned char* isdev = nullptr;
    int* devidx = nullptr;
    nb_events* ev = nullptr;
    TrajDesc* descs = nullptr;
    void* grid_ws = nullptr;
    size_t grid_ws_bytes = 0;
    std::vector<TrajDesc> h_descs;
    std::vector<nb_events> h_ev;
    nb_events* pin_ev = nullptr;  // pinned staging for the events + the grid kernel's status word: the D2H copies after a
    int* pin_status = nullptr;    // launch are then truly asynchronous and run() does the waiting itself (busy-wait)
    std::vector<int> cur_step;
    double gpu_seconds = 0.0;
    long long pairs = 0;
    // n > NB_MAX_SMALL_N: the steppers, shared by the systems (they are stepped in turn), and the events of the system being
    // stepped after each of the last two chunks (pinned staging, see run_large)
    LargeStepper large;
    nb_events* pin_chunk = nullptr;
    cudaEvent_t chunk_done[2] = {nullptr, nullptr};

    int init(int gpu_, int S_, int n_, int math_) {
        gpu = gpu_, S = S_, n = n_, math = math_;
        NB_CUDA(cudaSetDevice(gpu));
        NB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        NB_CUDA(cudaEventCreate(&e0));
        NB_CUDA(cudaEventCreate(&e1));
        NB_CUDA(cudaMalloc(&q, (size_t)S * 3 * n * sizeof(double)));
        NB_CUDA(cudaMalloc(&v, (size_t)S * 3 * n * sizeof(double)));
        NB_CUDA(cudaMalloc(&m, (size_t)S * n * sizeof(double)));
        NB_CUDA(cudaMalloc(&isdev, (size_t)S * n));
        NB_CUDA(cudaMalloc(&devidx, (size_t)S * NB_MAX_DEVICES * sizeof(int)));
        NB_CUDA(cudaMalloc(&ev, (size_t)S * sizeof(nb_events)));
        NB_CUDA(cudaMalloc(&descs, (size_t)S * sizeof(TrajDesc)));
        NB_CUDA(cudaHostAlloc(&pin_ev, (size_t)S * sizeof(nb_events), cudaHostAllocDefault));
        NB_CUDA(cudaHostAlloc(&pin_status, 64, cudaHostAllocDefault));
        h_descs.assign(S, TrajDesc{});
        h_ev.assign(S, nb_events{});
        cur_step.assign(S, 0);
        if (n > NB_MAX_SMALL_N) {
            const int rc = large.init(n, math, stream);
            if (rc) return rc;
            NB_CUDA(cudaHostAlloc(&pin_chunk, 2 * sizeof(nb_events), cudaHostAllocDefault));
            NB_CUDA(cudaEventCreateWithFlags(&chunk_done[0], cudaEventDisableTiming));
            NB_CUDA(cudaEventCreateWithFlags(&chunk_done[1], cudaEventDisableTiming));
        }
        return NB_OK;
    }
    void release() {
        if (gpu < 0) return;
        if (g_leak_on_exit.load()) {
            gpu = -1;
            return;
        }
        cudaSetDevice(gpu);
        cudaFree(q), cudaFree(v), cudaFree(m), cudaFree(isdev), cudaFree(devidx), cudaFree(ev), cudaFree(descs);
        if (grid_ws) cudaFree(grid_ws);
        if (pin_ev) cudaFreeHost(pin_ev);
        if (pin_status) cudaFreeHost(pin_status);
        pin_ev = nullptr, pin_status = nullptr;
        large.release();
        if (pin_chunk) cudaFreeHost(pin_chunk);
        pin_chunk = nullptr;
        for (cudaEvent_t& e : chunk_done)
            if (e) cudaEventDestroy(e), e = nullptr;
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (stream) cudaStreamDestroy(stream);
        gpu = -1;
    }
    static void fresh_events(nb_events& e) {
        e.min_d2 = std::numeric_limits<double>::infinity();
        e.argmin_step = -1;
        e.hit_step = -2;
        e.destroyed_step = -2;
        e.cost = std::numeric_limits<double>::infinity();
        e.steps_done = -1;
        e.n_reach = 0;
        for (int k = 0; k < NB_MAX_DEVICES; k++) e.reach_step[k] = -2;
    }
    // upload system s (host pointers), starting at `step0` with nothing observed yet
    int set_system(int s, const double* hq, const double* hv, const double* hm, const unsigned char* hdev, int planet,
                   int asteroid, int kind, int destroy_device, int step0) {
        if (planet < 0 || planet >= n || asteroid < 0 || asteroid >= n) return NB_ERR_ARG;
        if (kind == NB_KIND_Q3 && (destroy_device < 0 || destroy_device >= n)) return NB_ERR_ARG;
        std::vector<double> mm(hm, hm + n);
        std::vector<int> di;
        for (int i = 0; i < n; i++)
            if (hdev[i]) {
                di.push_back(i);
                if (kind == NB_KIND_Q1) mm[i] = 0.0;  // nbody.cc:109-113, hw5.cu:217-222,357
            }
        if ((int)di.size() > NB_MAX_DEVICES) return NB_ERR_UNSUPPORTED;
        NB_CUDA(cudaSetDevice(gpu));
        // hq / hv may be null: the caller fills q, v device-to-device afterwards (nb_traj_fork)
        if (hq) NB_CUDA(cudaMemcpyAsync(q + (size_t)s * 3 * n, hq, 3 * n * sizeof(double), cudaMemcpyHostToDevice, stream));
        if (hv) NB_CUDA(cudaMemcpyAsync(v + (size_t)s * 3 * n, hv, 3 * n * sizeof(double), cudaMemcpyHostToDevice, stream));
        NB_CUDA(cudaMemcpyAsync(m + (size_t)s * n, mm.data(), n * sizeof(double), cudaMemcpyHostToDevice, stream));
        NB_CUDA(cudaMemcpyAsync(isdev + (size_t)s * n, hdev, n, cudaMemcpyHostToDevice, stream));
        if (!di.empty())
            NB_CUDA(cudaMemcpyAsync(devidx + (size_t)s * NB_MAX_DEVICES, di.data(), di.size() * sizeof(int),
                                    cudaMemcpyHostToDevice, stream));
        fresh_events(h_ev[s]);
        h_ev[s].n_reach = (int)di.size();
        NB_CUDA(cudaMemcpyAsync(ev + s, &h_ev[s], sizeof(nb_events), cudaMemcpyHostToDevice, stream));
        NB_CUDA(cudaStreamSynchronize(stream));  // mm / di are stack-local
        TrajDesc& d = h_descs[s];
        d.n = n, d.planet = planet, d.asteroid = asteroid, d.kind = kind, d.destroy_device = destroy_device;
        d.n_dev = (int)di.size();
        d.q = q + (size_t)s * 3 * n, d.v = v + (size_t)s * 3 * n, d.m = m + (size_t)s * n;
        d.is_device = isdev + (size_t)s * n, d.dev_index = devidx + (size_t)s * NB_MAX_DEVICES, d.ev = ev + s;
        cur_step[s] = step0;
        return NB_OK;
    }
    // advance every system to step_end (or its stop event); blocks until done
    int run(int step_end, bool allow_grid) {
        int max_end = step_end;
        for (int s = 0; s < S; s++) {
            h_descs[s].step_begin = cur_step[s];
            h_descs[s].step_end = step_end > cur_step[s] ? step_end : cur_step[s];
        }
        const double* fst = nullptr;
        int rc = fst_table(gpu, max_end + 2, &fst);
        if (rc) return rc;
        NB_CUDA(cudaSetDevice(gpu));
        NB_CUDA(cudaMemcpyAsync(descs, h_descs.data(), S * sizeof(TrajDesc), cudaMemcpyHostToDevice, stream));
        NB_CUDA(cudaEventRecord(e0, stream));
        const auto h0 = std::chrono::steady_clock::now();
        int max_dev = 0;
        for (int s = 0; s < S; s++) max_dev = h_descs[s].n_dev > max_dev ? h_descs[s].n_dev : max_dev;
        // the grid kernel's observer warp keeps two devices per lane (NB_MAX_DEVICES = 64); STRICT needs the single block's
        // ascending-j sum
        bool grid = false;
        if (n > NB_MAX_SMALL_N) {
            rc = run_large();
        } else if (allow_grid && math == NB_MATH_FAST && max_dev <= 64 && grid_traj_supported(gpu, n)) {
            size_t need = grid_traj_workspace_bytes(n);
            if (need > grid_ws_bytes) {
                if (grid_ws) NB_CUDA(cudaFree(grid_ws));
                NB_CUDA(cudaMalloc(&grid_ws, need));
                grid_ws_bytes = need;
            }
            rc = launch_grid_traj(math, n, S, descs, fst, gpu, grid_ws, grid_ws_bytes, stream);
            grid = true;
            if (rc == NB_ERR_UNSUPPORTED) {
                // the grid's blocks cannot be co-resident here (MIG, MPS, a shared GPU); nothing was launched and no
                // state was touched: the single-block kernel gives the same answer, only slower
                static const bool verbose = getenv("NB_VERBOSE") != nullptr;
                if (verbose) fprintf(stderr, "nbody_b200: grid kernel unavailable (%s): single-block kernel instead\n", g_detail.c_str());
                rc = launch_traj_batch(math, n, S, descs, fst, stream);
                grid = false;
            }
        } else {
            rc = launch_traj_batch(math, n, S, descs, fst, stream);
        }
        if (rc) return rc;
        NB_CUDA(cudaEventRecord(e1, stream));  // e0 .. e1 = the kernels only: nothing below waits on the host in between
        {
            const double hms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
            static const bool verbose = getenv("NB_VERBOSE") != nullptr;
            if (verbose && hms > 2.0) fprintf(stderr, "nbody_b200:   host spent %.1f ms between the two event records\n", hms);
        }
        NB_CUDA(cudaMemcpyAsync(pin_ev, ev, S * sizeof(nb_events), cudaMemcpyDeviceToHost, stream));
        *pin_status = 0;
        pin_status[1] = 0;
        if (grid) NB_CUDA(cudaMemcpyAsync(pin_status, grid_traj_status(grid_ws, n), 2 * sizeof(int), cudaMemcpyDeviceToHost, stream));
        rc = spin_wait(stream);
        if (rc) return rc;
        memcpy(h_ev.data(), pin_ev, S * sizeof(nb_events));
        if (pin_status[1] != 0) g_torn_records += pin_status[1];  // records that failed the full self-check and were fetched again
        if (*pin_status != 0) {
            set_error_detail("grid trajectory kernel: exchange spin timed out (blocks not co-resident?)");
            return NB_ERR_CUDA;
        }
        float ms = 0;
        NB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        gpu_seconds += ms * 1e-3;
        for (int s = 0; s < S; s++) {
            long long steps = h_ev[s].steps_done - cur_step[s];
            if (steps > 0) pairs += steps * (long long)n * (n - 1);
            cur_step[s] = h_ev[s].steps_done;
        }
        return NB_OK;
    }
    static bool stopped(const nb_events& e, int kind) { return kind >= NB_KIND_Q2 && e.hit_step != -2; }
    // n > NB_MAX_SMALL_N: the systems one after another on the large-N steppers, each step followed by the one-warp observer
    // (large_observe_kernel), step_begin observed first unless it already was.  Steps go out in chunks of large_chunk(n):
    // while chunk c + 1 runs, the host reads the events after chunk c and enqueues nothing more once the stop event has
    // fired.  The q, v left in a stopped slot are therefore up to two chunks past the stop, while cur_step (= steps_done) is
    // the stop step: get_state would not return the state at cur_step there.  Nothing reads it - solve_chain reloads such
    // a slot, and later runs skip a stopped system - so it is not rewound.
    int run_large() {
        const int chunk = large_chunk(n);
        for (int s = 0; s < S; s++) {
            const TrajDesc& d = h_descs[s];
            if (stopped(h_ev[s], d.kind) || h_ev[s].steps_done >= d.step_end) continue;
            int rc = large.pack(d.q, d.m, d.is_device, d.step_begin + 1, stream);
            if (!rc) rc = launch_large_observe(d, large.pos[large.cur], d.step_begin, stream);
            for (int st = d.step_begin, c = 0; !rc && st < d.step_end; c++) {
                const int end = std::min(st + chunk, d.step_end);
                while (!rc && st < end) {
                    rc = large.step(++st, d.v, d.m, d.is_device, stream);
                    if (!rc) rc = launch_large_observe(d, large.pos[large.cur], st, stream);
                }
                if (rc || st >= d.step_end) break;
                NB_CUDA(cudaMemcpyAsync(pin_chunk + (c & 1), d.ev, sizeof(nb_events), cudaMemcpyDeviceToHost, stream));
                NB_CUDA(cudaEventRecord(chunk_done[c & 1], stream));
                if (c > 0) {  // chunk c is queued: read the events after chunk c - 1
                    rc = spin_wait(stream, chunk_done[(c - 1) & 1]);
                    if (!rc && stopped(pin_chunk[(c - 1) & 1], d.kind)) break;
                }
            }
            if (!rc) rc = large.unpack(d.q, stream);
            if (rc) return rc;
        }
        return NB_OK;
    }
    int get_state(int s, double* hq, double* hv, double* hm) {
        NB_CUDA(cudaSetDevice(gpu));
        if (hq) NB_CUDA(cudaMemcpyAsync(hq, q + (size_t)s * 3 * n, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, stream));
        if (hv) NB_CUDA(cudaMemcpyAsync(hv, v + (size_t)s * 3 * n, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, stream));
        if (hm) NB_CUDA(cudaMemcpyAsync(hm, m + (size_t)s * n, n * sizeof(double), cudaMemcpyDeviceToHost, stream));
        NB_CUDA(cudaStreamSynchronize(stream));
        return NB_OK;
    }
};

}  // namespace nb

using nb::DeviceBatch;

struct nb_traj {
    DeviceBatch b;
    int planet, asteroid, kind, destroy_device;
    std::vector<unsigned char> isdev;
};

extern "C" {

const char* nb_version(void) { return "nbody_b200 0.1 (sm_100a)"; }

const char* nb_strerror(int code) {
    switch (code) {
        case NB_OK: return "ok";
        case NB_ERR_ARG: return "invalid argument";
        case NB_ERR_CUDA: return "CUDA error";
        case NB_ERR_NO_GPU: return "no usable CUDA device (this library has no CPU fallback)";
        case NB_ERR_UNSUPPORTED: return "unsupported size or mode";
        case NB_ERR_IO: return "I/O or parse error";
        default: return "unknown error";
    }
}

const char* nb_last_error_detail(void) { return nb::g_detail.c_str(); }

int nb_device_count(int* count) {
    if (!count) return NB_ERR_ARG;
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess || c == 0) {
        (void)cudaGetLastError();
        *count = 0;
        nb::set_error_detail(std::string("no CUDA device: ") + cudaGetErrorString(e));
        return NB_ERR_NO_GPU;
    }
    *count = c;
    return NB_OK;
}

long long nb_kernel_launches(void) { return nb::g_launches.load(); }
long long nb_grid_torn_records(void) { return nb::g_torn_records.load(); }

// Everything a GPU needs before its first trajectory launch, callable from a helper thread while the input is still
// being parsed: driver initialisation + primary context, the |sin| table, the trajectory kernels' module.
void nb_internal_leak_on_exit(int on) { nb::g_leak_on_exit.store(on != 0); }

int nb_device_warm(int gpu) {
    int rc = nb::check_gpu(gpu);
    if (rc) return rc;
    NB_CUDA(cudaSetDevice(gpu));
    NB_CUDA(cudaFree(nullptr));
    const double* fst = nullptr;
    rc = nb::fst_table(gpu, NB_N_STEPS + 2, &fst);
    if (rc) return rc;
    nb::grid_traj_warm();
    return NB_OK;
}

// ---- trajectories ------------------------------------------------------------------------------------
int nb_traj_create(int gpu, const nb_system* sys, int kind, int destroy_device, int math, nb_traj** out) {
    if (!sys || !out || !sys->q || !sys->v || !sys->m || !sys->is_device) return NB_ERR_ARG;
    if (sys->n < 1) return NB_ERR_ARG;
    if (sys->n > NB_MAX_SMALL_N) return NB_ERR_UNSUPPORTED;
    if (kind < NB_KIND_PLAIN || kind > NB_KIND_Q3 || (math != NB_MATH_FAST && math != NB_MATH_STRICT)) return NB_ERR_ARG;
    int rc = nb::check_gpu(gpu);
    if (rc) return rc;
    nb_traj* t = new nb_traj();
    t->planet = sys->planet, t->asteroid = sys->asteroid, t->kind = kind, t->destroy_device = destroy_device;
    t->isdev.assign(sys->is_device, sys->is_device + sys->n);
    rc = t->b.init(gpu, 1, sys->n, math);
    if (!rc)
        rc = t->b.set_system(0, sys->q, sys->v, sys->m, sys->is_device, sys->planet, sys->asteroid, kind, destroy_device, 0);
    if (rc) {
        t->b.release();
        delete t;
        return rc;
    }
    *out = t;
    return NB_OK;
}

int nb_traj_run(nb_traj* t, int step_end, nb_events* ev) {
    if (!t || step_end < 0) return NB_ERR_ARG;
    int rc = t->b.run(step_end, true);
    if (rc) return rc;
    if (ev) *ev = t->b.h_ev[0];
    return NB_OK;
}

int nb_traj_state(nb_traj* t, double* q, double* v, double* m, int* step) {
    if (!t) return NB_ERR_ARG;
    if (step) *step = t->b.cur_step[0];
    return t->b.get_state(0, q, v, m);
}

// Fork = the reference's snapshot + restore (hw5.cu:275-284, 411-413, 482-483) without the host bounce: positions
// and velocities go device to device (cudaMemcpyPeerAsync over NVLink when the fork lives on another GPU); only the
// n base masses (Q1 zeroing, device list) pass through the host.
int nb_traj_fork_on(nb_traj* t, int gpu, int kind, int destroy_device, nb_traj** out) {
    if (!t || !out) return NB_ERR_ARG;
    if (kind < NB_KIND_PLAIN || kind > NB_KIND_Q3) return NB_ERR_ARG;
    int rc = nb::check_gpu(gpu);
    if (rc) return rc;
    const int n = t->b.n;
    std::vector<double> m(n);
    rc = t->b.get_state(0, nullptr, nullptr, m.data());
    if (rc) return rc;
    nb_traj* f = new nb_traj();
    f->planet = t->planet, f->asteroid = t->asteroid, f->kind = kind, f->destroy_device = destroy_device;
    f->isdev = t->isdev;
    rc = f->b.init(gpu, 1, n, t->b.math);
    if (!rc)
        rc = f->b.set_system(0, nullptr, nullptr, m.data(), f->isdev.data(), f->planet, f->asteroid, kind, destroy_device,
                             t->b.cur_step[0]);
    if (!rc) {
        const size_t bytes = 3 * (size_t)n * sizeof(double);
        cudaError_t e = cudaSuccess;
        if (gpu == t->b.gpu) {
            e = cudaMemcpyAsync(f->b.q, t->b.q, bytes, cudaMemcpyDeviceToDevice, f->b.stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(f->b.v, t->b.v, bytes, cudaMemcpyDeviceToDevice, f->b.stream);
        } else {
            e = cudaMemcpyPeerAsync(f->b.q, gpu, t->b.q, t->b.gpu, bytes, f->b.stream);
            if (e == cudaSuccess) e = cudaMemcpyPeerAsync(f->b.v, gpu, t->b.v, t->b.gpu, bytes, f->b.stream);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(f->b.stream);
        if (e != cudaSuccess) rc = nb::cuda_fail(e, "fork copy", __FILE__, __LINE__);
    }
    if (rc) {
        f->b.release();
        delete f;
        return rc;
    }
    *out = f;
    return NB_OK;
}

int nb_traj_fork(nb_traj* t, int kind, int destroy_device, nb_traj** out) {
    if (!t) return NB_ERR_ARG;
    return nb_traj_fork_on(t, t->b.gpu, kind, destroy_device, out);
}

int nb_traj_destroy(nb_traj* t) {
    if (!t) return NB_ERR_ARG;
    t->b.release();
    delete t;
    return NB_OK;
}

// ---- ensembles ---------------------------------------------------------------------------------------
int nb_ensemble_run(int gpu, int math, int kind, int n_systems, int n, double* q, double* v, const double* m,
                    const unsigned char* is_device, const int* planet, const int* asteroid, const int* destroy_device,
                    int step_begin, int step_end, nb_events* ev, double* gpu_seconds) {
    if (n_systems < 1 || n < 1 || !q || !v || !m || !is_device || step_begin < 0 || step_end < step_begin) return NB_ERR_ARG;
    if (n > NB_MAX_SMALL_N) return NB_ERR_UNSUPPORTED;
    if (kind < NB_KIND_PLAIN || kind > NB_KIND_Q3 || (math != NB_MATH_FAST && math != NB_MATH_STRICT)) return NB_ERR_ARG;
    if (kind == NB_KIND_Q3 && !destroy_device) return NB_ERR_ARG;
    int rc = nb::check_gpu(gpu);
    if (rc) return rc;
    DeviceBatch b;
    rc = b.init(gpu, n_systems, n, math);
    for (int s = 0; s < n_systems && !rc; s++)
        rc = b.set_system(s, q + (size_t)s * 3 * n, v + (size_t)s * 3 * n, m + (size_t)s * n, is_device + (size_t)s * n,
                          planet ? planet[s] : 0, asteroid ? asteroid[s] : 0, kind,
                          destroy_device ? destroy_device[s] : -1, step_begin);
    if (!rc && step_begin > 0) {
        // resuming: the caller has observed step_begin already
        for (int s = 0; s < n_systems; s++) b.h_ev[s].steps_done = step_begin;
        cudaError_t e = cudaMemcpy(b.ev, b.h_ev.data(), n_systems * sizeof(nb_events), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) rc = nb::cuda_fail(e, "cudaMemcpy(ev)", __FILE__, __LINE__);
    }
    if (!rc) rc = b.run(step_end, false);
    for (int s = 0; s < n_systems && !rc; s++) {
        rc = b.get_state(s, q + (size_t)s * 3 * n, v + (size_t)s * 3 * n, nullptr);
        if (ev) ev[s] = b.h_ev[s];
    }
    if (gpu_seconds) *gpu_seconds = b.gpu_seconds;
    b.release();
    return rc;
}

// ---- the step operator -------------------------------------------------------------------------------
// n > NB_MAX_SMALL_N on one GPU (LargeStepper), host buffers in and out.  The first failing call's code is returned;
// everything is freed on every path.
static int run_steps_large(int gpu, int math, int n, double* q, double* v, const double* m, const unsigned char* is_device,
                           int step_begin, int step_end) {
    NB_CUDA(cudaSetDevice(gpu));
    int rc = NB_OK;
    cudaStream_t st = nullptr;
    double *dq = nullptr, *dv = nullptr, *dm = nullptr;
    unsigned char* ddev = nullptr;
    nb::LargeStepper ls;
    auto chk = [&](cudaError_t e, const char* what) {
        if (e != cudaSuccess && rc == NB_OK) rc = nb::cuda_fail(e, what, __FILE__, __LINE__);
    };
    chk(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "cudaStreamCreate");
    chk(cudaMalloc(&dq, 3 * (size_t)n * sizeof(double)), "cudaMalloc q");
    chk(cudaMalloc(&dv, 3 * (size_t)n * sizeof(double)), "cudaMalloc v");
    chk(cudaMalloc(&dm, (size_t)n * sizeof(double)), "cudaMalloc m");
    chk(cudaMalloc(&ddev, (size_t)n), "cudaMalloc is_device");
    if (rc == NB_OK) rc = ls.init(n, math, st);
    if (rc == NB_OK) {
        chk(cudaMemcpyAsync(dq, q, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D q");
        chk(cudaMemcpyAsync(dv, v, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D v");
        chk(cudaMemcpyAsync(dm, m, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D m");
        chk(cudaMemcpyAsync(ddev, is_device, (size_t)n, cudaMemcpyHostToDevice, st), "H2D is_device");
    }
    if (rc == NB_OK) rc = ls.pack(dq, dm, ddev, step_begin + 1, st);
    for (int step = step_begin + 1; step <= step_end && rc == NB_OK; step++) rc = ls.step(step, dv, dm, ddev, st);
    if (rc == NB_OK) rc = ls.unpack(dq, st);
    if (rc == NB_OK) {
        chk(cudaMemcpyAsync(q, dq, 3 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H q");
        chk(cudaMemcpyAsync(v, dv, 3 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H v");
        chk(cudaStreamSynchronize(st), "sync");
    }
    cudaFree(dq), cudaFree(dv), cudaFree(dm), cudaFree(ddev);
    ls.release();
    if (st) cudaStreamDestroy(st);
    return rc;
}

int nb_run_steps(int gpu, int math, int n, double* q, double* v, const double* m, const unsigned char* is_device,
                 int step_begin, int step_end) {
    if (n < 1 || !q || !v || !m || !is_device || step_begin < 0 || step_end < step_begin) return NB_ERR_ARG;
    if (math != NB_MATH_FAST && math != NB_MATH_STRICT) return NB_ERR_ARG;
    int rc = nb::check_gpu(gpu);
    if (rc) return rc;
    if (n > NB_MAX_SMALL_N) return run_steps_large(gpu, math, n, q, v, m, is_device, step_begin, step_end);
    DeviceBatch b;
    rc = b.init(gpu, 1, n, math);
    if (!rc) rc = b.set_system(0, q, v, m, is_device, 0, 0, NB_KIND_PLAIN, -1, step_begin);
    if (!rc) rc = b.run(step_end, true);
    if (!rc) rc = b.get_state(0, q, v, nullptr);
    b.release();
    return rc;
}

// ---- the three queries -------------------------------------------------------------------------------
// Ensemble scheduler.  trajectory 0 = Q1, 1 = Q2, 2+k = Q3 with device k destroyed.  Two plans, no collective in
// either, only nb_events structs come back:
//   * INDEPENDENT (as many GPUs as trajectories, or NB_SOLVE_ALL_DEVICES): Q1, Q2 and one Q3 trajectory per device
//     are all simulated from step 0 (identical arithmetic gives each Q3 trajectory Q2's prefix: no snapshot
//     transport, no dependency on Q2 - SURVEY 7.2); trajectory t goes to part t % n_parts, one launch per part.
//   * CHAIN (fewer GPUs than trajectories; the reference's own plan, hw5.cu:396-413, 438-530, 575-588): Q2 runs in
//     chunks of NB_SOLVE_CHUNK steps with a device-to-device copy of its state before each chunk; a device whose
//     missile arrives inside a chunk gets that copy as its fork point, so its Q3 trajectory starts at most one
//     chunk before the arrival instead of at step 0 (a fork started before the arrival is bit-identical to a
//     run from step 0).  The candidates are then tried in order of arrival step = order of cost, and the search
//     stops at the first one that saves the planet (hw5.cu:491-492, 509-517): the others cost more.  Part 0 runs
//     Q1 (in lock step with the chain when it is the only part), part 1 the chain.  Further parts (2 < GPUs <
//     trajectories) SPECULATE: part 2 + s simulates, from step 0, the query-3 trajectory of the device that is s-th
//     nearest to the planet at step 0 (the missile flies at a fixed speed, so that is the likely order of arrival);
//     the chain leaves those devices out and nb_solve_combine picks the cheapest saviour among everything simulated.
static const int NB_SOLVE_CHUNK = [] {
    const int v = getenv("NB_SOLVE_CHUNK") ? atoi(getenv("NB_SOLVE_CHUNK")) : 8192;
    return v < 1 ? 1 : v;  // 0 or negative would never advance the chain
}();

static bool solve_chain_plan(int n_parts, int n_traj, int math_flags) {
    return n_parts < n_traj && !(math_flags & NB_SOLVE_ALL_DEVICES);
}

static int solve_jobs(const nb_system* sys, std::vector<int>& devs) {
    if (!sys || !sys->q || !sys->v || !sys->m || !sys->is_device || sys->n < 1) return NB_ERR_ARG;
    if (sys->planet < 0 || sys->planet >= sys->n || sys->asteroid < 0 || sys->asteroid >= sys->n) return NB_ERR_ARG;
    devs.clear();
    for (int i = 0; i < sys->n; i++)
        if (sys->is_device[i]) devs.push_back(i);
    if ((int)devs.size() > NB_MAX_DEVICES) return NB_ERR_UNSUPPORTED;
    return NB_OK;
}

int nb_solve_trajectory_count(const nb_system* sys, int* count) {
    std::vector<int> devs;
    int rc = solve_jobs(sys, devs);
    if (rc) return rc;
    if (!count) return NB_ERR_ARG;
    *count = 2 + (int)devs.size();
    return NB_OK;
}


// devices (indexes into devs) by distance to the planet at step 0, nearest first; ties by index
static std::vector<int> speculation_order(const nb_system* sys, const std::vector<int>& devs) {
    const int n = sys->n, P = sys->planet;
    std::vector<std::pair<double, int>> d;
    for (int k = 0; k < (int)devs.size(); k++) {
        const int b = devs[k];
        const double dx = sys->q[b] - sys->q[P], dy = sys->q[b + n] - sys->q[P + n], dz = sys->q[b + 2 * n] - sys->q[P + 2 * n];
        d.emplace_back(dx * dx + dy * dy + dz * dz, k);
    }
    std::sort(d.begin(), d.end());
    std::vector<int> order;
    for (auto& e : d) order.push_back(e.second);
    return order;
}

// CHAIN plan on one GPU (see above): slot 0 = Q1 (optional), last slot = Q2, then the Q3 candidates one after another;
// devices flagged in `speculated` are simulated elsewhere and left out
static int solve_chain(const nb_system* sys, const std::vector<int>& devs, const std::vector<char>& speculated, int gpu,
                       bool with_q1, bool with_chain, int n_steps, int math, nb_events* evs, double* gpu_seconds,
                       long long* pair_interactions) {
    const bool verbose = getenv("NB_VERBOSE") != nullptr;
    const int n = sys->n, dc = (int)devs.size();
    const size_t sbytes = 3 * (size_t)n * sizeof(double);
    int rc = nb::check_gpu(gpu);
    if (rc) return rc;
    DeviceBatch b;
    const int S = (with_q1 ? 1 : 0) + (with_chain ? 1 : 0), sl = S - 1;  // sl = slot of the chain
    const auto t_init = std::chrono::steady_clock::now();
    rc = b.init(gpu, S, n, math);
    if (verbose)
        fprintf(stderr, "nbody_b200: gpu %d buffers + pinned mailbox %.4f s\n", gpu,
                std::chrono::duration<double>(std::chrono::steady_clock::now() - t_init).count());
    if (!rc && with_q1) rc = b.set_system(0, sys->q, sys->v, sys->m, sys->is_device, sys->planet, sys->asteroid, NB_KIND_Q1, -1, 0);
    if (!rc && with_chain)
        rc = b.set_system(sl, sys->q, sys->v, sys->m, sys->is_device, sys->planet, sys->asteroid, NB_KIND_Q2, -1, 0);
    double* lag = nullptr;               // Q2's q, v at the start of the current chunk
    std::vector<double*> snap(dc, nullptr);  // fork point of device k: q, v at the start of the chunk its missile arrived in
    std::vector<int> snap_step(dc, -1);
    auto cleanup = [&](int r) {
        if (nb::g_leak_on_exit.load()) return r;
        cudaSetDevice(gpu);
        if (lag) cudaFree(lag);
        for (double* p : snap)
            if (p) cudaFree(p);
        b.release();
        return r;
    };
    if (rc) return cleanup(rc);
    int n_launch = 0;
    const auto t_run = std::chrono::steady_clock::now();
    if (!with_chain) {
        rc = b.run(n_steps, true);
        if (!rc) evs[0] = b.h_ev[0];
    } else {
        if (cudaMalloc(&lag, 2 * sbytes) != cudaSuccess) return cleanup(NB_ERR_CUDA);
        double* cq = b.q + (size_t)sl * 3 * n;
        double* cv = b.v + (size_t)sl * 3 * n;
        // ---- Q2 (and Q1 beside it), chunk by chunk while a missile is still under way
        int cur = 0;
        bool first = true;  // n_steps == 0 still observes step 0
        while (!rc && (first || (cur < n_steps && b.h_ev[sl].hit_step == -2))) {
            first = false;
            bool pending = false;
            for (int k = 0; k < dc; k++) pending |= snap_step[k] < 0;
            // chunks go on after the last arrival: Q1 (same launch) must not run ahead alone past Q2's hit, its remaining
            // steps pair with the Q3 candidate's in one launch
            const int next = cur + NB_SOLVE_CHUNK < n_steps ? cur + NB_SOLVE_CHUNK : n_steps;
            if (pending) {
                if (cudaMemcpyAsync(lag, cq, sbytes, cudaMemcpyDeviceToDevice, b.stream) != cudaSuccess ||
                    cudaMemcpyAsync(lag + 3 * n, cv, sbytes, cudaMemcpyDeviceToDevice, b.stream) != cudaSuccess)
                    return cleanup(NB_ERR_CUDA);
            }
            const double g_before = b.gpu_seconds;
            rc = b.run(next, true);
            n_launch++;
            if (verbose) fprintf(stderr, "nbody_b200:   Q2 chunk %d -> %d: kernels %.4f s\n", cur, next, b.gpu_seconds - g_before);
            for (int k = 0; k < dc && !rc; k++)
                if (snap_step[k] < 0 && b.h_ev[sl].reach_step[k] != -2) {
                    if (cudaMalloc(&snap[k], 2 * sbytes) != cudaSuccess ||
                        cudaMemcpyAsync(snap[k], lag, 2 * sbytes, cudaMemcpyDeviceToDevice, b.stream) != cudaSuccess)
                        return cleanup(NB_ERR_CUDA);
                    snap_step[k] = cur;
                }
            cur = next;
        }
        if (rc) return cleanup(rc);
        evs[1] = b.h_ev[sl];
        for (int k = 0; k < dc; k++) {  // "not simulated" until tried; a speculated device is another part's entry
            DeviceBatch::fresh_events(evs[2 + k]);
            if (speculated[k]) evs[2 + k].steps_done = -2;
        }
        // ---- Q3: candidates by arrival step (= by cost, hw5.cu:575-585), first saviour wins (hw5.cu:491-492)
        if (evs[1].hit_step != -2) {
            std::vector<int> order;
            for (int k = 0; k < dc; k++)
                if (snap_step[k] >= 0 && !speculated[k]) order.push_back(k);
            std::stable_sort(order.begin(), order.end(),
                             [&](int a, int c2) { return evs[1].reach_step[a] < evs[1].reach_step[c2]; });
            for (int k : order) {
                rc = b.set_system(sl, nullptr, nullptr, sys->m, sys->is_device, sys->planet, sys->asteroid, NB_KIND_Q3, devs[k],
                                  snap_step[k]);
                if (rc) return cleanup(rc);
                if (cudaMemcpyAsync(cq, snap[k], sbytes, cudaMemcpyDeviceToDevice, b.stream) != cudaSuccess ||
                    cudaMemcpyAsync(cv, snap[k] + 3 * n, sbytes, cudaMemcpyDeviceToDevice, b.stream) != cudaSuccess)
                    return cleanup(NB_ERR_CUDA);
                const double g_before = b.gpu_seconds;
                rc = b.run(n_steps, true);  // Q1, if still under way, rides along in the same launch
                n_launch++;
                if (verbose)
                    fprintf(stderr, "nbody_b200:   Q3 device %d from step %d: kernels %.4f s\n", devs[k], snap_step[k], b.gpu_seconds - g_before);
                if (rc) return cleanup(rc);
                evs[2 + k] = b.h_ev[sl];
                if (b.h_ev[sl].hit_step == -2 && b.h_ev[sl].destroyed_step != -2) break;  // saved: the rest cost more
            }
        }
        if (with_q1) {
            if (b.cur_step[0] < n_steps) {
                // nothing left to pair Q1 with: park the chain slot (a stopped trajectory never steps again)
                rc = b.run(n_steps, true);
                n_launch++;
            }
            if (!rc) evs[0] = b.h_ev[0];
        }
    }
    if (verbose)
        fprintf(stderr, "nbody_b200: gpu %d chain plan (%s%s): %d launches, run %.3f s (kernels %.3f s)\n", gpu,
                with_q1 ? "Q1 " : "", with_chain ? "Q2 -> Q3 candidates" : "", n_launch,
                std::chrono::duration<double>(std::chrono::steady_clock::now() - t_run).count(), b.gpu_seconds);
    if (gpu_seconds) *gpu_seconds = b.gpu_seconds;
    if (pair_interactions) *pair_interactions = b.pairs;
    return cleanup(rc);
}

int nb_solve_partial(const nb_system* sys, int gpu, int part, int n_parts, int n_steps, int math, nb_events* evs,
                     double* gpu_seconds, long long* pair_interactions) {
    std::vector<int> devs;
    int rc = solve_jobs(sys, devs);
    if (rc) return rc;
    if (!evs || n_parts < 1 || part < 0 || part >= n_parts || n_steps < 0) return NB_ERR_ARG;
    const int math_flags = math;
    math &= ~NB_SOLVE_ALL_DEVICES;
    if (math != NB_MATH_FAST && math != NB_MATH_STRICT) return NB_ERR_ARG;
    for (int t = 0; t < 2 + (int)devs.size(); t++) {  // entries of other parts stay marked "not mine"
        DeviceBatch::fresh_events(evs[t]);
        evs[t].steps_done = -2;
    }
    if (gpu_seconds) *gpu_seconds = 0;
    if (pair_interactions) *pair_interactions = 0;
    const int T = 2 + (int)devs.size();
    std::vector<int> mine;  // trajectories this part simulates from step 0 in one launch
    if (solve_chain_plan(n_parts, T, math_flags)) {
        std::vector<char> speculated(devs.size(), 0);
        const std::vector<int> order = speculation_order(sys, devs);
        for (int p = 2; p < n_parts && p - 2 < (int)order.size(); p++) speculated[order[p - 2]] = 1;
        if (part <= 1)
            return solve_chain(sys, devs, speculated, gpu, /*with_q1=*/part == 0, /*with_chain=*/n_parts == 1 || part == 1, n_steps,
                               math, evs, gpu_seconds, pair_interactions);
        if (part - 2 >= (int)order.size()) return NB_OK;
        mine.push_back(2 + order[part - 2]);
    } else {
        for (int t = part; t < T; t += n_parts) mine.push_back(t);
    }
    const bool verbose = getenv("NB_VERBOSE") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto secs_since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double>(now() - t).count(); };
    auto t_a = now();
    rc = nb::check_gpu(gpu);
    if (rc) return rc;
    const double s_driver = secs_since(t_a);
    if (gpu_seconds) *gpu_seconds = 0;
    if (pair_interactions) *pair_interactions = 0;
    if (mine.empty()) return NB_OK;
    DeviceBatch b;
    auto t_b = now();
    rc = b.init(gpu, (int)mine.size(), sys->n, math);
    const double s_ctx = secs_since(t_b);
    auto t_c = now();
    for (size_t s = 0; s < mine.size() && !rc; s++) {
        const int t = mine[s];
        const int kind = t == 0 ? NB_KIND_Q1 : (t == 1 ? NB_KIND_Q2 : NB_KIND_Q3);
        rc = b.set_system((int)s, sys->q, sys->v, sys->m, sys->is_device, sys->planet, sys->asteroid, kind,
                          t >= 2 ? devs[t - 2] : -1, 0);
    }
    const double s_upload = secs_since(t_c);
    auto t_d = now();
    if (!rc) rc = b.run(n_steps, true);
    const double s_run = secs_since(t_d);
    if (verbose)
        fprintf(stderr, "nbody_b200: gpu %d part %d/%d: driver init %.3f s, context+alloc %.3f s, upload %.3f s, "
                        "run %.3f s (kernels %.3f s)\n", gpu, part, n_parts, s_driver, s_ctx, s_upload, s_run, b.gpu_seconds);
    if (!rc)
        for (size_t s = 0; s < mine.size(); s++) evs[mine[s]] = b.h_ev[s];
    if (gpu_seconds) *gpu_seconds = b.gpu_seconds;
    if (pair_interactions) *pair_interactions = b.pairs;
    b.release();
    return rc;
}

int nb_solve_combine(const nb_system* sys, const nb_events* evs, nb_answer* ans) {
    std::vector<int> devs;
    int rc = solve_jobs(sys, devs);
    if (rc) return rc;
    if (!evs || !ans) return NB_ERR_ARG;
    const int dc = (int)devs.size();
    memset(ans, 0, sizeof *ans);
    ans->min_dist = sqrt(evs[0].min_d2);  // hw5.cu:407
    ans->argmin_step = evs[0].argmin_step;
    ans->hit_time_step = evs[1].hit_step;  // -2 when none (nbody.cc:125)
    ans->gravity_device_id = -1;           // hw5.cu:547-548
    ans->missile_cost = 0;
    ans->n_devices = dc;
    for (int k = 0; k < NB_MAX_DEVICES; k++) {
        ans->device_index[k] = k < dc ? devs[k] : -1;
        ans->reach_step[k] = k < dc ? evs[1].reach_step[k] : -2;
        ans->q3_hit_step[k] = -3;
        ans->q3_cost[k] = std::numeric_limits<double>::infinity();
    }
    if (evs[1].hit_step != -2) {  // hw5.cu:568
        double best = std::numeric_limits<double>::infinity();
        for (int k = 0; k < dc; k++) {
            const nb_events& e = evs[2 + k];
            if (e.steps_done < 0) continue;  // not simulated (chain plan: a cheaper device already saved the planet)
            ans->q3_hit_step[k] = e.hit_step;
            ans->q3_cost[k] = e.cost;
            // hw5.cu:509-517: saved (no hit through n_steps) and cheapest; ties -> lowest device index
            if (e.hit_step == -2 && e.destroyed_step != -2 && e.cost < best) {
                best = e.cost;
                ans->gravity_device_id = devs[k];
                ans->missile_cost = e.cost;
            }
        }
    }
    ans->n_trajectories = 2 + dc;
    return NB_OK;
}

int nb_solve(const nb_system* sys, const int* gpus, int n_gpus, int n_steps, int math, nb_answer* ans) {
    std::vector<int> devs;
    int rc = solve_jobs(sys, devs);
    if (rc) return rc;
    if (!ans || n_gpus < 1 || n_steps < 0) return NB_ERR_ARG;
    auto t_begin = std::chrono::steady_clock::now();
    const int T = 2 + (int)devs.size();
    const int G = n_gpus < T ? n_gpus : T;  // chain plan with more than two GPUs: the spare ones speculate (see above)
    std::vector<int> gl(G);
    for (int g = 0; g < G; g++) {
        gl[g] = gpus ? gpus[g] : g;
        rc = nb::check_gpu(gl[g]);
        if (rc) return rc;
    }
    std::vector<nb_events> evs(T);
    std::vector<int> rcs(G, 0);
    std::vector<std::string> details(G);
    std::vector<double> secs(G, 0.0);
    std::vector<long long> pairs(G, 0);
    std::vector<std::vector<nb_events>> part_evs(G, std::vector<nb_events>(T));
    auto worker = [&](int g) {
        rcs[g] = nb_solve_partial(sys, gl[g], g, G, n_steps, math, part_evs[g].data(), &secs[g], &pairs[g]);
        if (rcs[g]) details[g] = nb::g_detail;
    };
    std::vector<std::thread> th;  // one host thread per GPU (hw5.cu:566-567, 587-588)
    for (int g = 1; g < G; g++) th.emplace_back(worker, g);
    worker(0);
    for (auto& t : th) t.join();
    for (int g = 0; g < G; g++) {
        if (rcs[g]) {
            nb::set_error_detail(details[g]);
            return rcs[g];
        }
        for (int t = 0; t < T; t++)
            if (part_evs[g][t].steps_done != -2) evs[t] = part_evs[g][t];
    }
    rc = nb_solve_combine(sys, evs.data(), ans);
    if (rc) return rc;
    for (int g = 0; g < G; g++) {
        if (secs[g] > ans->gpu_seconds) ans->gpu_seconds = secs[g];
        ans->pair_interactions += pairs[g];
    }
    ans->n_gpus_used = G;
    ans->wall_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count();
    return NB_OK;
}

}  // extern "C"
