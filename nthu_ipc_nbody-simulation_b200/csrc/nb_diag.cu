// Diagnostics of a state (nb_diagnostics, nb_traj_diagnostics): mass, kinetic and potential energy, linear and angular
// momentum of every system of a batch, with the effective masses of the state's step (nbody.cc:14-16, 63).
//
// Two kernels, no floating-point atomics, every sum in a fixed order (DESIGN.md §4.6):
//   sym_potential_kernel  one block per (upper-triangle tile of DIAG_T x DIAG_T body pairs, system).  The j tile is staged
//                         in shared memory as {x, y, z, m} records; each of the DIAG_THREADS threads holds DIAG_IPT i
//                         bodies and accumulates sum_j m_j / r_ij over the tile with one FMA per pair (pair_rinv,
//                         nb_math.cuh), then sum_t m_i(t) * acc_t.  Diagonal tiles take j > i only, and add the O(n)
//                         terms (mass, m|v|^2, m v, m q x v) of their i bodies.  The block's nine sums go through a
//                         shuffle tree to one partial record per tile.
//   sym_diag_sum_kernel   one block per system: each thread sums every DIAG_SUM_THREADS-th tile partial in tile order, a
//                         shuffle + shared-memory tree combines the threads.  kinetic = 0.5 * sum, potential = -G * sum.
// A system's partials and their order depend on n only, never on the other systems of the batch.
#include <climits>

#include "nb_internal.h"
#include "nb_math.cuh"

namespace nb {

namespace {

constexpr int DIAG_THREADS = 64;
constexpr int DIAG_IPT = DIAG_T / DIAG_THREADS;
constexpr int DIAG_SUM_THREADS = 1024;
static_assert(DIAG_IPT * DIAG_THREADS == DIAG_T, "tile edge = threads x i bodies per thread");

// partial record: mass, sum m|v|^2, sum_{i<j} m_i m_j / r_ij, P[3], L[3]
enum { Q_MASS, Q_KIN, Q_POT, Q_PX, Q_PY, Q_PZ, Q_LX, Q_LY, Q_LZ, DIAG_Q };

struct PairSys {
    const double* q;                  // [S][3n] planar
    const double* v;                  // [S][3n] planar
    const double* m;                  // [S][n] base masses
    const unsigned char* is_device;  // [S][n]
};

template <bool DIAG>
__device__ __forceinline__ void tile_pairs(const double4* rec, const double (&xi)[DIAG_IPT], const double (&yi)[DIAG_IPT],
                                           const double (&zi)[DIAG_IPT], double (&acc)[DIAG_IPT]) {
#pragma unroll 2
    for (int jj = 0; jj < DIAG_T; jj++) {
        const double4 r = rec[jj];
#pragma unroll
        for (int t = 0; t < DIAG_IPT; t++) {
            // diagonal tile: local index of i body t is t * DIAG_THREADS + threadIdx.x; j > i only (the self pair too
            // gets a finite r^-1 = 1/eps and weight 0)
            const double mj = DIAG ? (jj > t * DIAG_THREADS + (int)threadIdx.x ? r.w : 0.0) : r.w;
            acc[t] = fma(mj, pair_rinv(xi[t], yi[t], zi[t], r.x, r.y, r.z), acc[t]);
        }
    }
}

__device__ __forceinline__ double warp_tree(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    return x;
}

__global__ void __launch_bounds__(DIAG_THREADS) sym_potential_kernel(PairSys sys, int n, int s0, int S, int n_tiles,
                                                                       double fst, double* __restrict__ part) {
    __shared__ double4 rec[DIAG_T];
    __shared__ double red[DIAG_THREADS / 32][DIAG_Q];
    const int s = s0 + blockIdx.y, k = blockIdx.x;
    int I, J;
    tile_of(k, I, J);
    const double* q = sys.q + (size_t)s * 3 * n;
    const double* m = sys.m + (size_t)s * n;
    const unsigned char* dev = sys.is_device + (size_t)s * n;
    for (int jj = threadIdx.x; jj < DIAG_T; jj += DIAG_THREADS) {
        const int j = J * DIAG_T + jj;
        rec[jj] = j < n ? make_double4(q[j], q[j + n], q[j + 2 * n], m_eff(m[j], dev[j] != 0, fst))
                        : make_double4(0.0, 0.0, 0.0, 0.0);
    }
    double xi[DIAG_IPT], yi[DIAG_IPT], zi[DIAG_IPT], mi[DIAG_IPT], acc[DIAG_IPT];
#pragma unroll
    for (int t = 0; t < DIAG_IPT; t++) {
        const int i = I * DIAG_T + t * DIAG_THREADS + threadIdx.x;
        const bool in = i < n;
        xi[t] = in ? q[i] : 0.0, yi[t] = in ? q[i + n] : 0.0, zi[t] = in ? q[i + 2 * n] : 0.0;
        mi[t] = in ? m_eff(m[i], dev[i] != 0, fst) : 0.0;
        acc[t] = 0.0;
    }
    __syncthreads();
    if (I == J)
        tile_pairs<true>(rec, xi, yi, zi, acc);
    else
        tile_pairs<false>(rec, xi, yi, zi, acc);
    double r[DIAG_Q] = {};
#pragma unroll
    for (int t = 0; t < DIAG_IPT; t++) r[Q_POT] = fma(mi[t], acc[t], r[Q_POT]);
    if (I == J) {  // the O(n) terms of the tile's i bodies, once per body
        const double* v = sys.v + (size_t)s * 3 * n;
#pragma unroll
        for (int t = 0; t < DIAG_IPT; t++) {
            const int i = I * DIAG_T + t * DIAG_THREADS + threadIdx.x;
            if (i >= n) break;
            const double vx = v[i], vy = v[i + n], vz = v[i + 2 * n], w = mi[t];
            r[Q_MASS] += w;
            r[Q_KIN] = fma(w, fma(vx, vx, fma(vy, vy, vz * vz)), r[Q_KIN]);
            r[Q_PX] = fma(w, vx, r[Q_PX]);
            r[Q_PY] = fma(w, vy, r[Q_PY]);
            r[Q_PZ] = fma(w, vz, r[Q_PZ]);
            r[Q_LX] = fma(w, fma(yi[t], vz, -(zi[t] * vy)), r[Q_LX]);
            r[Q_LY] = fma(w, fma(zi[t], vx, -(xi[t] * vz)), r[Q_LY]);
            r[Q_LZ] = fma(w, fma(xi[t], vy, -(yi[t] * vx)), r[Q_LZ]);
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < DIAG_Q; c++) r[c] = warp_tree(r[c]);
    if (lane == 0)
#pragma unroll
        for (int c = 0; c < DIAG_Q; c++) red[warp][c] = r[c];
    __syncthreads();
    if (threadIdx.x < DIAG_Q) {
        const int c = threadIdx.x;
        double x = red[0][c];
#pragma unroll
        for (int w = 1; w < DIAG_THREADS / 32; w++) x += red[w][c];
        part[((size_t)c * S + s) * n_tiles + k] = x;
    }
}

__global__ void __launch_bounds__(DIAG_SUM_THREADS) sym_diag_sum_kernel(const double* __restrict__ part, int S, int n_tiles,
                                                                         double* __restrict__ out) {
    __shared__ double red[DIAG_SUM_THREADS / 32][DIAG_Q];
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int c = 0; c < DIAG_Q; c++) {
        const double* p = part + ((size_t)c * S + s) * n_tiles;
        double x = 0.0;
        for (int k = threadIdx.x; k < n_tiles; k += DIAG_SUM_THREADS) x += p[k];
        x = warp_tree(x);
        if (lane == 0) red[warp][c] = x;
    }
    __syncthreads();
    if (warp == 0) {
        double* o = out + (size_t)s * DIAG_Q;
        for (int c = 0; c < DIAG_Q; c++) {
            const double x = warp_tree(red[lane][c]);
            if (lane == 0) o[c] = c == Q_KIN ? 0.5 * x : (c == Q_POT ? -(G * x) : x);
        }
    }
}

long long diag_tiles(int n) {
    const long long t = (n + DIAG_T - 1) / DIAG_T;
    return t * (t + 1) / 2;
}

}  // namespace

size_t diag_scratch_bytes(int S, int n) { return (size_t)DIAG_Q * S * diag_tiles(n) * sizeof(double); }

int diag_launch(int S, int n, const double* q, const double* v, const double* m, const unsigned char* is_device, double fst,
                void* scratch, double* out, cudaStream_t stream) {
    const long long tiles = diag_tiles(n);
    if (tiles > INT_MAX) return NB_ERR_UNSUPPORTED;
    const PairSys sys{q, v, m, is_device};
    for (int s0 = 0; s0 < S; s0 += 65535) {  // gridDim.y limit
        const int cnt = S - s0 < 65535 ? S - s0 : 65535;
        sym_potential_kernel<<<dim3((unsigned)tiles, cnt), DIAG_THREADS, 0, stream>>>(sys, n, s0, S, (int)tiles, fst,
                                                                                       (double*)scratch);
        count_launch();
        NB_CUDA(cudaGetLastError());
    }
    sym_diag_sum_kernel<<<S, DIAG_SUM_THREADS, 0, stream>>>((const double*)scratch, S, (int)tiles, out);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

}  // namespace nb
