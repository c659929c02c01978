// Ensembles of NB_MAX_SMALL_N < n <= NB_MAX_ENSEMBLE_N bodies (nb_ensemble_run): every system of a group advanced by one
// launch per kernel and step, grid = (work item, system).  DESIGN.md §4.7.
//
// Per system, in the group's scratch (EnsGroup, nb_internal.h):
//     pos4[parity][n_pad] = {x, y, z, G*m_eff(step)}   parity = step & 1; bodies n .. n_pad-1 are zero records, never written
//     slots[B][3][n_pad]                               partial accelerations; B = n_pad / ENS_T slots (FAST), 1 (STRICT)
// A step st is three launches for the whole group:
//   sym_ens_tile_kernel         FAST.  One warp per (upper-triangle tile (I, J) of ENS_T x ENS_T bodies, system).  The j
//                               tile is staged in shared memory; the warp holds the ENS_T i bodies in registers, ENS_IPT
//                               per lane.  An off-diagonal tile evaluates every unordered pair once (pair_sym): the j
//                               bodies rotate through the lanes by shuffles with their accumulators, as in
//                               traj_sym_kernel.  A diagonal tile is one-sided (pair_coeff_fast / pair_accum_fast; the
//                               self term is exactly zero).  Tile (I, J) writes its a_i row into slot J of row I and its
//                               a_j row into slot I of row J, so every slot of every body is written once per step and
//                               no atomics are needed.
//   large_ens_strict_kernel     STRICT.  One thread per i body, j ascending through shared-memory tiles with
//                               pair<MATH_STRICT>: the oracle's order, the whole sum into slot 0.
//   large_ens_integrate_kernel  adds a body's slots in ascending order, kick_drift on the system's planar v, and writes
//                               the next record with the masses of step st+1 (gm_eff, as large_integrate_kernel).
// followed by large_ens_observe_kernel (one warp per system, the observer of large_observe_kernel).
// A system whose Q2/Q3 stop event has fired returns at the top of every kernel: its q, v and records stay at the hit step.
// Every sum has a fixed order that depends on n only, so a system's result does not depend on the other systems.
#include "nb_internal.h"
#include "nb_math.cuh"
#include "nb_observe.cuh"

namespace nb {
namespace {

// Measured on B200 (profiles/r05_large_ensembles.md): one warp and 4 i bodies per lane (tile edge 128) against tile edge
// 256 (two such warps, or one warp with 8 per lane): equal at 2048 and 8192 bodies, 1.24x faster at 1025 (less padding).
constexpr int ENS_IPT = 4;              // i bodies per lane
constexpr int ENS_T = 32 * ENS_IPT;     // tile edge: the warp's i bodies = its j tile
constexpr int STRICT_THREADS = 128;     // STRICT: i bodies per block = j records per shared tile
constexpr int INTEGRATE_THREADS = 128;
static_assert(ENS_T % STRICT_THREADS == 0, "n_pad is a whole number of STRICT j tiles");

// a system's stop event has fired (Q2 / Q3 hit): the observer of the previous step ran earlier in the stream
__device__ __forceinline__ bool ens_stopped(const TrajDesc* descs, int g) {
    return descs[g].kind >= NB_KIND_Q2 && descs[g].ev->hit_step != -2;
}

__global__ void __launch_bounds__(32) sym_ens_tile_kernel(const EnsGroup e, int parity) {
    __shared__ double4 jt[ENS_T];
    const int g = blockIdx.y;
    if (ens_stopped(e.descs, g)) return;
    int I, J;
    tile_of(blockIdx.x, I, J);
    const double4* p = e.pos4 + ((size_t)parity * e.G + g) * e.n_pad;
    double* slot = e.slots + (size_t)g * e.n_slots * 3 * e.n_pad;
    const int lane = threadIdx.x;
    const int src_lane = (lane + 1) & 31;
    for (int k = lane; k < ENS_T; k += 32) jt[k] = p[J * ENS_T + k];
    // i body of register slot k: ib + 32k
    const int ib = I * ENS_T + lane;
    double xi[ENS_IPT], yi[ENS_IPT], zi[ENS_IPT], gi[ENS_IPT], ax[ENS_IPT], ay[ENS_IPT], az[ENS_IPT];
#pragma unroll
    for (int k = 0; k < ENS_IPT; k++) {
        const double4 r = p[ib + 32 * k];
        xi[k] = r.x, yi[k] = r.y, zi[k] = r.z, gi[k] = r.w;
        ax[k] = ay[k] = az[k] = 0.0;
    }
    __syncwarp();
    if (I == J) {
        // diagonal tile, one-sided: every lane reads the same j record
#pragma unroll 2
        for (int j = 0; j < ENS_T; j++) {
            const double4 b = jt[j];
            double c[ENS_IPT], dx[ENS_IPT], dy[ENS_IPT], dz[ENS_IPT];
#pragma unroll
            for (int k = 0; k < ENS_IPT; k++) pair_coeff_fast(xi[k], yi[k], zi[k], b.x, b.y, b.z, b.w, c[k], dx[k], dy[k], dz[k]);
#pragma unroll
            for (int k = 0; k < ENS_IPT; k++) pair_accum_fast(c[k], dx[k], dy[k], dz[k], ax[k], ay[k], az[k]);
        }
    } else {
        // off-diagonal tile, symmetric: 32 j bodies at a time, one per lane, home again after 32 moves
#pragma unroll 1
        for (int s0 = 0; s0 < ENS_T; s0 += 32) {
            const double4 b = jt[s0 + lane];
            double jx = b.x, jy = b.y, jz = b.z, jg = b.w;
            double ajx = 0.0, ajy = 0.0, ajz = 0.0;
#pragma unroll 2
            for (int r = 0; r < 32; r++) {
                const double nx = __shfl_sync(0xffffffffu, jx, src_lane), ny = __shfl_sync(0xffffffffu, jy, src_lane),
                             nz = __shfl_sync(0xffffffffu, jz, src_lane), ng = __shfl_sync(0xffffffffu, jg, src_lane);
#pragma unroll
                for (int k = 0; k < ENS_IPT; k++)
                    pair_sym(xi[k], yi[k], zi[k], gi[k], jx, jy, jz, jg, ax[k], ay[k], az[k], ajx, ajy, ajz);
                ajx = __shfl_sync(0xffffffffu, ajx, src_lane), ajy = __shfl_sync(0xffffffffu, ajy, src_lane),
                ajz = __shfl_sync(0xffffffffu, ajz, src_lane);
                jx = nx, jy = ny, jz = nz, jg = ng;
            }
            // a_j row of the tile: slot I of row J
            double* out = slot + (size_t)I * 3 * e.n_pad + J * ENS_T + s0 + lane;
            out[0] = ajx, out[e.n_pad] = ajy, out[2 * e.n_pad] = ajz;
        }
    }
    // a_i row of the tile: slot J of row I
    double* out = slot + (size_t)J * 3 * e.n_pad;
#pragma unroll
    for (int k = 0; k < ENS_IPT; k++) {
        out[ib + 32 * k] = ax[k];
        out[e.n_pad + ib + 32 * k] = ay[k];
        out[2 * e.n_pad + ib + 32 * k] = az[k];
    }
}

__global__ void __launch_bounds__(STRICT_THREADS) large_ens_strict_kernel(const EnsGroup e, int parity) {
    __shared__ double4 jt[STRICT_THREADS];
    const int g = blockIdx.y;
    if (ens_stopped(e.descs, g)) return;
    const double4* p = e.pos4 + ((size_t)parity * e.G + g) * e.n_pad;
    const int i = blockIdx.x * STRICT_THREADS + threadIdx.x;  // < n_pad
    const double4 r = p[i];
    double ax = 0.0, ay = 0.0, az = 0.0;
    for (int j0 = 0; j0 < e.n; j0 += STRICT_THREADS) {
        __syncthreads();  // everyone is done with the previous tile
        jt[threadIdx.x] = p[j0 + threadIdx.x];
        __syncthreads();
        const int cnt = min(STRICT_THREADS, e.n - j0);
        for (int j = 0; j < cnt; j++) {
            const double4 b = jt[j];
            pair<MATH_STRICT>(r.x, r.y, r.z, b.x, b.y, b.z, b.w, ax, ay, az);
        }
    }
    if (i < e.n) {
        double* out = e.slots + (size_t)g * e.n_slots * 3 * e.n_pad;
        out[i] = ax, out[e.n_pad + i] = ay, out[2 * e.n_pad + i] = az;
    }
}

__global__ void __launch_bounds__(INTEGRATE_THREADS) large_ens_integrate_kernel(const EnsGroup e, int parity,
                                                                                  double fst_next) {
    const int g = blockIdx.y;
    if (ens_stopped(e.descs, g)) return;
    const int i = blockIdx.x * INTEGRATE_THREADS + threadIdx.x;
    const int n = e.n;
    if (i >= n) return;
    const TrajDesc& d = e.descs[g];
    const double* slot = e.slots + (size_t)g * e.n_slots * 3 * e.n_pad;
    double a[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        double s = slot[(size_t)c * e.n_pad + i];
        for (int k = 1; k < e.n_slots; k++) s += slot[((size_t)k * 3 + c) * e.n_pad + i];
        a[c] = s;
    }
    const double4 p = e.pos4[((size_t)parity * e.G + g) * e.n_pad + i];
    double x = p.x, y = p.y, z = p.z;
    double* v = d.v;
    double vx = v[i], vy = v[i + n], vz = v[i + 2 * n];
    kick_drift(a[0], vx, x);
    kick_drift(a[1], vy, y);
    kick_drift(a[2], vz, z);
    v[i] = vx, v[i + n] = vy, v[i + 2 * n] = vz;
    e.pos4[((size_t)(parity ^ 1) * e.G + g) * e.n_pad + i] = make_double4(x, y, z, gm_eff(d.m[i], d.is_device[i] != 0, fst_next));
}

__global__ void __launch_bounds__(32) large_ens_observe_kernel(const EnsGroup e, int parity, int st) {
    const int g = blockIdx.x;
    observe_large(e.descs[g], e.pos4 + ((size_t)parity * e.G + g) * e.n_pad, st);
}

}  // namespace

int ens_pad(int n) { return (n + ENS_T - 1) / ENS_T * ENS_T; }

int ens_slots(int math, int n) { return math == NB_MATH_STRICT ? 1 : ens_pad(n) / ENS_T; }

int ens_step(int math, const EnsGroup& e, int step, cudaStream_t stream) {
    const int parity = (step - 1) & 1;  // the records of step - 1
    if (math == NB_MATH_STRICT) {
        large_ens_strict_kernel<<<dim3(e.n_pad / STRICT_THREADS, e.G), STRICT_THREADS, 0, stream>>>(e, parity);
    } else {
        const int B = e.n_pad / ENS_T;
        sym_ens_tile_kernel<<<dim3(B * (B + 1) / 2, e.G), 32, 0, stream>>>(e, parity);
    }
    count_launch();
    NB_CUDA(cudaGetLastError());
    large_ens_integrate_kernel<<<dim3((e.n + INTEGRATE_THREADS - 1) / INTEGRATE_THREADS, e.G), INTEGRATE_THREADS, 0, stream>>>(
        e, parity, fst_value(step + 1));
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

int ens_observe(const EnsGroup& e, int step, cudaStream_t stream) {
    large_ens_observe_kernel<<<e.G, 32, 0, stream>>>(e, step & 1, step);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

}  // namespace nb
