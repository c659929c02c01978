// Large-N step (n > 1024, e.g. the 65 536-body synthetic system), optionally body-sharded:
// this GPU integrates bodies [i_begin, i_begin+i_count) against ALL n bodies.
//
// Replaces compute_accelerations_gpu (one thread per ordered pair + 3 FP64 atomics per pair,
// hw5.cu:159-215) and update_positions_gpu (hw5.cu:231-239).  Arithmetic: nbody.cc:56-88.
//
// Data layout in HBM (L2-resident: 2 MiB at n = 65 536):
//     pos4[n] = {x, y, z, G*m_eff(step)}   one 32-byte record per body, double-buffered by step
// so that a j-tile is ONE contiguous block: tiles of TJ records are streamed into shared memory
// with 1-D TMA bulk copies (cp.async.bulk + mbarrier, SASS UBLKCP) through a STAGES-deep ring while
// the FP64 pipe works on the previous tile.  i-bodies live in registers (IPT per thread); every
// lane of a warp reads the same j record (shared-memory broadcast, 2 LDS.128 per IPT pairs).
//
// Grid = (i blocks) x (j splits): each block writes its partial acceleration to
// apart[split][3][i_count]; nb_large_integrate sums the splits in ascending order (deterministic,
// no atomics), applies v += a*dt, q += v*dt and emits the next pos4 record with G*m_eff(step+1).
// The split exists only to cut the work into enough equal pieces to balance 148 SMs.
#include <cstdint>
#include <cstring>
#include <vector>

#include "nb_async.cuh"
#include "nb_internal.h"
#include "nb_math.cuh"
#include "nb_observe.cuh"

namespace nb {
namespace {

constexpr int TJ = 256;      // bodies per j tile (8 KiB)
constexpr int STAGES = 3;    // TMA ring depth
constexpr int LT = 128;      // threads per block
constexpr int IPT = 4;       // i-bodies per thread (measured on B200 in round 1: 4 >= 2 > 1)
constexpr int MAX_JSPLIT = 128;

// P2P exchange only: the rows of source rank r are valid once counters[r] >= target (every block of r's
// integrate kernel has stored its rows here and released).  Blocks whose j range is local start at once -
// the grid is rotated so that they are scheduled first - and the others wait for exactly the ranks they
// read, so the arrival of the remote rows overlaps with the local tiles.
struct ArrivalWait {
    const unsigned long long* counters;  // [world] for the parity being read; nullptr = nothing to wait for
    unsigned long long target;
    int rows_per_rank, my_rank;
    int* status;
};

template <int MATH>
__global__ void __launch_bounds__(LT)
large_accel_kernel(const double4* __restrict__ pos4, int n, int i_begin, int i_count, int j_per_split,
                   double* __restrict__ apart, ArrivalWait aw) {
    __shared__ alignas(128) double4 tile[STAGES][TJ];
    __shared__ alignas(8) uint64_t full[STAGES];

    const int tid = threadIdx.x;
    int ysplit = blockIdx.y;
    if (aw.counters) ysplit = (int)((blockIdx.y + (unsigned)(aw.my_rank * aw.rows_per_rank) / j_per_split) % gridDim.y);
    const int j0 = ysplit * j_per_split;
    const int j1 = min(n, j0 + j_per_split);
    const int ntiles = (j1 - j0 + TJ - 1) / TJ;
    if (aw.counters) {
        if (tid == 0) {
            const int lo = j0 / aw.rows_per_rank, hi = (j1 - 1) / aw.rows_per_rank;
            const long long t0 = clock64();  // one deadline for all the sources
            for (int src = lo; src <= hi; src++)
                if (src != aw.my_rank) wait_counter(aw.counters + src, aw.target, aw.status, 1, t0);
            asm volatile("fence.proxy.async;" ::: "memory");  // the TMA (async proxy) reads what was just acquired
        }
        __syncthreads();
    }

    double xi[IPT], yi[IPT], zi[IPT], ax[IPT], ay[IPT], az[IPT];
    int il[IPT];
#pragma unroll
    for (int k = 0; k < IPT; k++) {
        il[k] = (blockIdx.x * IPT + k) * LT + tid;
        const double4 p = pos4[i_begin + min(il[k], i_count - 1)];
        xi[k] = p.x, yi[k] = p.y, zi[k] = p.z;
        ax[k] = ay[k] = az[k] = 0.0;
    }

    auto issue = [&](int t) {
        const int st = t % STAGES;
        const int jb = j0 + t * TJ;
        const uint32_t bytes = (uint32_t)(min(TJ, j1 - jb) * sizeof(double4));
        mbar_expect_tx(&full[st], bytes);
        tma_load_1d(&tile[st][0], pos4 + jb, bytes, &full[st]);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; s++) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0)
        for (int t = 0; t < STAGES && t < ntiles; t++) issue(t);

    for (int t = 0; t < ntiles; t++) {
        const int st = t % STAGES;
        mbar_wait(&full[st], (t / STAGES) & 1);
        const double4* tj = tile[st];
        const int cnt = min(TJ, j1 - (j0 + t * TJ));
        if (cnt == TJ) {
#pragma unroll 4
            for (int j = 0; j < TJ; j++) {
                const double4 b = tj[j];
                if (MATH == MATH_FAST) {
                    double c[IPT], dx[IPT], dy[IPT], dz[IPT];
#pragma unroll
                    for (int k = 0; k < IPT; k++) pair_coeff_fast(xi[k], yi[k], zi[k], b.x, b.y, b.z, b.w, c[k], dx[k], dy[k], dz[k]);
#pragma unroll
                    for (int k = 0; k < IPT; k++) pair_accum_fast(c[k], dx[k], dy[k], dz[k], ax[k], ay[k], az[k]);
                } else {
#pragma unroll
                    for (int k = 0; k < IPT; k++) pair<MATH>(xi[k], yi[k], zi[k], b.x, b.y, b.z, b.w, ax[k], ay[k], az[k]);
                }
            }
        } else {
            for (int j = 0; j < cnt; j++) {
                const double4 b = tj[j];
#pragma unroll
                for (int k = 0; k < IPT; k++) pair<MATH>(xi[k], yi[k], zi[k], b.x, b.y, b.z, b.w, ax[k], ay[k], az[k]);
            }
        }
        __syncthreads();  // everyone is done with stage st: refill it
        if (tid == 0 && t + STAGES < ntiles) issue(t + STAGES);
    }

    double* out = apart + (size_t)ysplit * 3 * i_count;
#pragma unroll
    for (int k = 0; k < IPT; k++)
        if (il[k] < i_count) {
            out[il[k]] = ax[k];
            out[il[k] + i_count] = ay[k];
            out[il[k] + 2 * i_count] = az[k];
        }
}

// The exchange fused into the integrate step (north star (d), second option): the new pos4 record of every
// local body is stored straight into EVERY rank's pos4_out buffer (peer-mapped pointers, NVLink P2P stores;
// the own buffer is peer `rank`), then each block raises every rank's arrival counter of this step's parity
// with a system-scope release.  No NCCL call, no staging copy: the all-gather is these stores.
constexpr int MAX_PEERS = 16;
struct PeerSet {
    double4* pos4_out[MAX_PEERS];
    unsigned long long* counter[MAX_PEERS];  // per rank: [2 parities][MAX_PEERS source ranks]
    int world, my_rank;
};

// sums the j-splits in ascending order, integrates (nbody.cc:77-88), writes the next pos4 record: to pos4_out, or with
// PUSH to every rank's buffer in `peers` followed by the release of their counters (`parity`); the other kind of
// destination is not read
template <bool PUSH>
__global__ void large_integrate_kernel(const double4* __restrict__ pos4, double4* __restrict__ pos4_out, PeerSet peers,
                                       double* __restrict__ vel, const double* __restrict__ m0,
                                       const unsigned char* __restrict__ is_device, const double* __restrict__ apart,
                                       int jsplit, int i_begin, int i_count, double fst_next, int parity) {
    const int il = blockIdx.x * blockDim.x + threadIdx.x;
    if (il < i_count) {
        double a[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            double s = apart[(size_t)c * i_count + il];
            for (int k = 1; k < jsplit; k++) s += apart[((size_t)k * 3 + c) * i_count + il];
            a[c] = s;
        }
        const int i = i_begin + il;
        const double4 p = pos4[i];
        double x = p.x, y = p.y, z = p.z;
        double vx = vel[il], vy = vel[il + i_count], vz = vel[il + 2 * i_count];
        kick_drift(a[0], vx, x);
        kick_drift(a[1], vy, y);
        kick_drift(a[2], vz, z);
        vel[il] = vx, vel[il + i_count] = vy, vel[il + 2 * i_count] = vz;
        const double4 rec = make_double4(x, y, z, gm_eff(m0[i], is_device[i] != 0, fst_next));
        if constexpr (PUSH)
            for (int pr = 0; pr < peers.world; pr++) peers.pos4_out[pr][i] = rec;  // coalesced 32 B per lane, per peer
        else
            pos4_out[i] = rec;
    }
    if constexpr (PUSH) {
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x < peers.world) red_release_sys(peers.counter[threadIdx.x] + parity * MAX_PEERS + peers.my_rank);
    }
}

// device-side wait, in stream order, until every counter (one thread per source rank) has reached target
__global__ void counter_wait_kernel(const unsigned long long* counters, unsigned long long target, int* status, int code) {
    wait_counter(counters + threadIdx.x, target, status, code);
}

__global__ void large_pack_kernel(int n, const double* __restrict__ q, const double* __restrict__ m0,
                                  const unsigned char* __restrict__ is_device, double fst_next,
                                  double4* __restrict__ pos4) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    pos4[i] = make_double4(q[i], q[i + n], q[i + 2 * n], gm_eff(m0[i], is_device[i] != 0, fst_next));
}

__global__ void large_unpack_kernel(int n, const double4* __restrict__ pos4, double* __restrict__ q) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double4 p = pos4[i];
    q[i] = p.x, q[i + n] = p.y, q[i + 2 * n] = p.z;
}

// The observers of step st of one trajectory on the large-N steppers: one warp, launched after the step's integrate kernel,
// reads the records {x, y, z, G*m_eff(st+1)} it wrote.  Lane l looks after devices l and l + 32 (NB_MAX_DEVICES = 64), as
// the grid kernel's observer warp does.  A stopped trajectory (Q2/Q3 hit) or an already observed step is left as it is,
// so steps enqueued past the stop change no event.  The Q3 destroy at st zeroes the device's base mass (Observed::store)
// and the mass of the record just read: the forces of step st+1 are the first without it (hw5.cu:299-307).
__global__ void __launch_bounds__(32) large_observe_kernel(const TrajDesc d, double4* __restrict__ pos4, int st) {
    const int lane = threadIdx.x;
    Observed ob;
    ob.load(d.ev);
    const bool stopped = (d.kind >= NB_KIND_Q2) && ob.hit_step != -2;
    if (stopped || d.ev->steps_done >= st) return;
    int my_dev[2], my_reach[2];
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int k = lane + 32 * h;
        my_dev[h] = k < d.n_dev ? d.dev_index[k] : -1;
        my_reach[h] = k < d.n_dev ? d.ev->reach_step[k] : -2;
    }
    const int DD = d.destroy_device;
    const bool armed = q3_armed(d.kind, DD, d.n, d.m);
    const int seen = observe_step<2>(ob, st, d.kind, d.planet, d.asteroid, armed, armed ? DD : 0, my_dev, my_reach,
                                     [&](int r, double& x, double& y, double& z) {
                                         const double4 p = pos4[r];
                                         x = p.x, y = p.y, z = p.z;
                                     });
    __syncwarp();  // every lane has read the events before lane 0 rewrites them
#pragma unroll
    for (int h = 0; h < 2; h++)
        if (lane + 32 * h < d.n_dev) d.ev->reach_step[lane + 32 * h] = my_reach[h];
    if (lane == 0) {
        ob.store(d, st);
        if (seen == OBS_DESTROYED) pos4[DD].w = 0.0;
    }
}

// optional per-thread profiling of the acceleration kernel (nb_profile_enable / nb_profile_read)
struct Prof {
    bool on = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> evs;
};
thread_local Prof g_prof;

int pick_jsplit(int math, int n, int i_count) {
    if (math == NB_MATH_STRICT) return 1;  // ascending-j sum == the oracle's order
    const int iblocks = (i_count + LT * IPT - 1) / (LT * IPT);
    int js = 1;
    // enough equal pieces (>= ~14 per SM) that the 148 SMs finish together, >= 2 tiles per piece;
    // measured on B200: 65 536 bodies, IPT 4: 1 split 43.8 %, 8 splits 54.6 %, 16 splits 54.9 % of peak;
    // an 8 192-body shard (P = 8) has only 16 i-blocks and needs 128 splits to fill the GPU
    while (js < MAX_JSPLIT && iblocks * js < 14 * 148 && n / (js * 2) >= 2 * TJ) js *= 2;
    return js;
}

}  // namespace

bool profile_on() { return g_prof.on; }
void profile_push(cudaEvent_t e0, cudaEvent_t e1) { g_prof.evs.emplace_back(e0, e1); }

int launch_counter_wait(const unsigned long long* counters, int count, unsigned long long target, int* status, int code,
                        cudaStream_t stream) {
    counter_wait_kernel<<<1, count, 0, stream>>>(counters, target, status, code);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

int launch_large_observe(const TrajDesc& d, double* pos4_dev, int step, cudaStream_t stream) {
    large_observe_kernel<<<1, 32, 0, stream>>>(d, (double4*)pos4_dev, step);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

}  // namespace nb

using namespace nb;

extern "C" {

long long nb_large_scratch_bytes(int n, int i_count) {
    (void)n;
    if (i_count < 1) return 0;
    // the largest split count pick_jsplit can choose for this shard (STRICT uses 1)
    const int js = pick_jsplit(NB_MATH_FAST, n, i_count);
    return (long long)js * 3 * i_count * (long long)sizeof(double);
}

int nb_large_pack(int math, int n, const double* q_planar_dev, const double* m0_dev, const unsigned char* is_device_dev,
                  int step_next, double* pos4_dev, void* stream) {
    (void)math;
    if (n < 1 || !q_planar_dev || !m0_dev || !is_device_dev || !pos4_dev || step_next < 0) return NB_ERR_ARG;
    const double fst = fst_value(step_next);
    large_pack_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, q_planar_dev, m0_dev, is_device_dev, fst,
                                                                         (double4*)pos4_dev);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

int nb_large_unpack(int n, const double* pos4_dev, double* q_planar_dev, void* stream) {
    if (n < 1 || !pos4_dev || !q_planar_dev) return NB_ERR_ARG;
    large_unpack_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, (const double4*)pos4_dev, q_planar_dev);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

static int large_step_impl(int math, int step, int n, int i_begin, int i_count, const double* pos4_dev,
                           double* pos4_out_dev, const PeerSet* peers, const ArrivalWait& aw, double* vel_dev,
                           const double* m0_dev, const unsigned char* is_device_dev, void* scratch_dev, void* stream) {
    if (n < 1 || i_begin < 0 || i_count < 1 || i_begin + i_count > n || step < 1) return NB_ERR_ARG;
    if (!pos4_dev || (!pos4_out_dev && !peers) || !vel_dev || !m0_dev || !is_device_dev || !scratch_dev) return NB_ERR_ARG;
    if (math != NB_MATH_FAST && math != NB_MATH_STRICT) return NB_ERR_ARG;
    const int jsplit = pick_jsplit(math, n, i_count);
    int jps = (n + jsplit - 1) / jsplit;
    jps = ((jps + TJ - 1) / TJ) * TJ;  // whole tiles per split
    const int nsplit = (n + jps - 1) / jps;
    dim3 grid((i_count + LT * IPT - 1) / (LT * IPT), nsplit);
    cudaStream_t st = (cudaStream_t)stream;
    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    if (g_prof.on) {
        NB_CUDA(cudaEventCreate(&pe0));
        NB_CUDA(cudaEventCreate(&pe1));
        NB_CUDA(cudaEventRecord(pe0, st));
    }
    auto* accel = math == NB_MATH_STRICT ? large_accel_kernel<MATH_STRICT> : large_accel_kernel<MATH_FAST>;
    accel<<<grid, LT, 0, st>>>((const double4*)pos4_dev, n, i_begin, i_count, jps, (double*)scratch_dev, aw);
    count_launch();
    NB_CUDA(cudaGetLastError());
    if (g_prof.on) {
        NB_CUDA(cudaEventRecord(pe1, st));
        g_prof.evs.emplace_back(pe0, pe1);
    }
    const double fst_next = fst_value(step + 1);
    auto* integrate = peers ? large_integrate_kernel<true> : large_integrate_kernel<false>;
    integrate<<<(i_count + 127) / 128, 128, 0, st>>>((const double4*)pos4_dev, (double4*)pos4_out_dev,
                                                     peers ? *peers : PeerSet{}, vel_dev, m0_dev, is_device_dev,
                                                     (const double*)scratch_dev, nsplit, i_begin, i_count, fst_next,
                                                     step & 1);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

int nb_large_step(int math, int step, int n, int i_begin, int i_count, const double* pos4_dev, double* pos4_out_dev,
                  double* vel_dev, const double* m0_dev, const unsigned char* is_device_dev, void* scratch_dev,
                  void* stream) {
    return large_step_impl(math, step, n, i_begin, i_count, pos4_dev, pos4_out_dev, nullptr, ArrivalWait{}, vel_dev,
                           m0_dev, is_device_dev, scratch_dev, stream);
}

int nb_large_step_p2p(int math, int step, int n, int i_begin, int i_count, const double* pos4_dev,
                      double* const* peer_pos4_out, unsigned long long* const* peer_counters, int world, int rank,
                      unsigned long long wait_target, int* status_dev, double* vel_dev, const double* m0_dev,
                      const unsigned char* is_device_dev, void* scratch_dev, void* stream) {
    if (!peer_pos4_out || !peer_counters || world < 1 || world > MAX_PEERS || rank < 0 || rank >= world) return NB_ERR_ARG;
    if (n % world != 0 || i_count != n / world || i_begin != rank * i_count || !status_dev) return NB_ERR_ARG;
    PeerSet ps;
    ps.world = world;
    ps.my_rank = rank;
    ArrivalWait aw{};
    if (wait_target > 0 && world > 1) {  // rows of step-1 live in the buffer being read; their counters have parity (step-1)&1
        aw.counters = peer_counters[rank] + ((step - 1) & 1) * MAX_PEERS;
        aw.target = wait_target;
        aw.rows_per_rank = i_count;
        aw.my_rank = rank;
        aw.status = status_dev;
    }
    for (int p = 0; p < world; p++) {
        if (!peer_pos4_out[p] || !peer_counters[p]) return NB_ERR_ARG;
        ps.pos4_out[p] = (double4*)peer_pos4_out[p];
        ps.counter[p] = peer_counters[p];
    }
    return large_step_impl(math, step, n, i_begin, i_count, pos4_dev, nullptr, &ps, aw, vel_dev, m0_dev, is_device_dev,
                           scratch_dev, stream);
}

int nb_large_blocks_per_step(int i_count) { return i_count < 1 ? 0 : (i_count + 127) / 128; }

int nb_large_p2p_counter_bytes(void) { return 2 * MAX_PEERS * (int)sizeof(unsigned long long); }

int nb_large_wait_p2p(const unsigned long long* my_counters, int parity, int world, unsigned long long target,
                      int* status_dev, void* stream) {
    if (!my_counters || !status_dev || world < 1 || world > MAX_PEERS || parity < 0 || parity > 1) return NB_ERR_ARG;
    return launch_counter_wait(my_counters + parity * MAX_PEERS, world, target, status_dev, 1, (cudaStream_t)stream);
}

// ---- raw device memory + CUDA IPC, for the peer-mapped buffers of the P2P exchange (one process per GPU) ----
int nb_dev_alloc(long long bytes, void** dev_ptr) {
    if (bytes < 1 || !dev_ptr) return NB_ERR_ARG;
    NB_CUDA(cudaMalloc(dev_ptr, (size_t)bytes));
    NB_CUDA(cudaMemset(*dev_ptr, 0, (size_t)bytes));
    return NB_OK;
}
int nb_dev_free(void* dev_ptr) {
    NB_CUDA(cudaFree(dev_ptr));
    return NB_OK;
}
int nb_dev_copy(void* dst, const void* src, long long bytes, int kind, void* stream) {
    if (!dst || !src || bytes < 0 || kind < 0 || kind > 2) return NB_ERR_ARG;
    const cudaMemcpyKind k = kind == 0 ? cudaMemcpyHostToDevice : kind == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    NB_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, k, (cudaStream_t)stream));
    NB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return NB_OK;
}
int nb_ipc_export(void* dev_ptr, unsigned char* handle64) {
    if (!dev_ptr || !handle64) return NB_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    cudaIpcMemHandle_t h;
    NB_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle64, &h, 64);
    return NB_OK;
}
int nb_ipc_open(const unsigned char* handle64, void** dev_ptr) {
    if (!handle64 || !dev_ptr) return NB_ERR_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    NB_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return NB_OK;
}
int nb_ipc_close(void* dev_ptr) {
    NB_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return NB_OK;
}

int nb_profile_enable(int on) {
    for (auto& p : g_prof.evs) cudaEventDestroy(p.first), cudaEventDestroy(p.second);
    g_prof.evs.clear();
    g_prof.on = on != 0;
    return NB_OK;
}

int nb_profile_read(double* accel_ms, long long* accel_launches) {
    double total = 0;
    for (auto& p : g_prof.evs) {
        NB_CUDA(cudaEventSynchronize(p.second));
        float ms = 0;
        NB_CUDA(cudaEventElapsedTime(&ms, p.first, p.second));
        total += ms;
    }
    if (accel_ms) *accel_ms = total;
    if (accel_launches) *accel_launches = (long long)g_prof.evs.size();
    return NB_OK;
}

}  // extern "C"
