// Persistent single-block trajectory kernel (n <= 1024): one thread block owns one system, keeps
// every body resident in shared memory and runs all steps AND all observers without returning to
// the host.  blockIdx.x selects the system, so one launch advances a whole ensemble.
//
// Replaces, per step, the reference's compute_accelerations_gpu<<<2D>>> + update_positions_gpu +
// <<<1,1>>> observer launches (hw5.cu:371-377, 390-397, 496-502) and the host loop around them.
// Arithmetic: nbody.cc:51-89 (see nb_math.cuh for the two variants).
//
// Thread map: thread t -> body i = t / JS, j-slice s = t % JS (JS a power of two <= 32, chosen so
// that n*JS <= 1024).  Slice s sums j = s, s+JS, ... in ascending order; slices are combined with
// a warp-shuffle butterfly.  JS == 1 (always used for STRICT) is the reference's ascending-j sum.
//
// Shared memory: xy[2][n] (double2) and zg[2][n] (double2 {z, G*m_eff}), double-buffered by step
// parity so that a step needs two block barriers:
//     [device G*m_eff(step) -> zg[cur]]  B  [forces from buf cur; owner integrates -> buf cur^1]  B  [observers]

#include "nb_internal.h"
#include "nb_math.cuh"
#include "nb_observe.cuh"

namespace nb {

namespace {

template <int MATH, int JS>
__global__ void __launch_bounds__(1024, 1)
traj_kernel(const TrajDesc* __restrict__ descs, const double* __restrict__ fst) {
    extern __shared__ double2 smem2[];
    const TrajDesc d = descs[blockIdx.x];
    const int n = d.n;
    double2* xy = smem2;          // [2][n]
    double2* zg = smem2 + 2 * n;  // [2][n]
    const int tid = threadIdx.x;
    const int i_raw = tid / JS;
    const int s = tid % JS;
    const bool active = i_raw < n;
    const int i = active ? i_raw : n - 1;
    const bool owner = active && (s == 0);

    // owner state
    double vx = 0, vy = 0, vz = 0;
    if (owner) {
        double x = d.q[i], y = d.q[i + n], z = d.q[i + 2 * n];
        vx = d.v[i];
        vy = d.v[i + n];
        vz = d.v[i + 2 * n];
        double gm = d.is_device[i] ? 0.0 : gm_eff(d.m[i], false, 0.0);
        xy[i] = make_double2(x, y);
        xy[n + i] = make_double2(x, y);
        zg[i] = make_double2(z, gm);
        zg[n + i] = make_double2(z, gm);
    }
    // device bookkeeping: thread k < n_dev looks after device k
    int my_dev = -1, my_reach = -2;
    double my_m0 = 0.0;
    if (tid < d.n_dev) {
        my_dev = d.dev_index[tid];
        my_m0 = d.m[my_dev];
        my_reach = d.ev->reach_step[tid];
    }
    Observed ob;
    ob.load(d.ev);
    const int kind = d.kind;
    const int P = d.planet, A = d.asteroid, DD = d.destroy_device;
    const bool armed = q3_armed(kind, DD, n, d.m);
    __syncthreads();

    int cur = 0;
    int step = d.step_begin;
    bool stop = (kind >= NB_KIND_Q2) && ob.hit_step != -2;

    // the observers' record reader of buffer b (built per call: a reader that captured `cur` would move instructions of the
    // pair loop, measured in the SASS of traj_kernel<FAST, 1>)
    auto records = [&](int b) {
        return [=](int r, double& x, double& y, double& z) {
            const double2 rxy = xy[b * n + r], rzg = zg[b * n + r];
            x = rxy.x, y = rxy.y, z = rzg.x;
        };
    };

    // the observers of this step; the traj kernels stop at the hit
    auto observe = [&]() {
        if (observe_step<1>(ob, step, kind, P, A, armed, DD, &my_dev, &my_reach, records(cur)) & OBS_HIT) stop = true;
    };
    if (d.ev->steps_done < step && !stop) observe();

    while (!stop && step < d.step_end) {
        ++step;
        // (1) G*m_eff of the devices for this step (nbody.cc:61-64); a destroyed device has mass 0
        if (my_dev >= 0) zg[cur * n + my_dev].y = device_gm(kind, my_dev, DD, ob, my_m0, fst, step);
        __syncthreads();
        // (2) forces on body i from slice s of the bodies (nbody.cc:56-74)
        const double2* cxy = xy + cur * n;
        const double2* czg = zg + cur * n;
        const double2 ixy = cxy[i], izg = czg[i];
        const double xi = ixy.x, yi = ixy.y, zi = izg.x;
        double ax = 0.0, ay = 0.0, az = 0.0;
        if (JS == 1) {
#pragma unroll 4
            for (int j = 0; j < n; ++j) {
                const double2 jxy = cxy[j], jzg = czg[j];
                pair<MATH>(xi, yi, zi, jxy.x, jxy.y, jzg.x, jzg.y, ax, ay, az);
            }
        } else {
#pragma unroll 2
            for (int j = s; j < n; j += JS) {
                const double2 jxy = cxy[j], jzg = czg[j];
                pair<MATH>(xi, yi, zi, jxy.x, jxy.y, jzg.x, jzg.y, ax, ay, az);
            }
#pragma unroll
            for (int o = JS / 2; o > 0; o >>= 1) {
                ax += __shfl_xor_sync(0xffffffffu, ax, o);
                ay += __shfl_xor_sync(0xffffffffu, ay, o);
                az += __shfl_xor_sync(0xffffffffu, az, o);
            }
        }
        // (3) v += a*dt; q += v*dt (nbody.cc:77-88) into the other buffer
        if (owner) {
            double x = xi, y = yi, z = zi;
            kick_drift(ax, vx, x);
            kick_drift(ay, vy, y);
            kick_drift(az, vz, z);
            xy[(cur ^ 1) * n + i] = make_double2(x, y);
            zg[(cur ^ 1) * n + i].x = z;
        }
        __syncthreads();
        cur ^= 1;
        observe();
    }

    // write back
    if (owner) {
        const double2 fxy = xy[cur * n + i], fzg = zg[cur * n + i];
        d.q[i] = fxy.x;
        d.q[i + n] = fxy.y;
        d.q[i + 2 * n] = fzg.x;
        d.v[i] = vx;
        d.v[i + n] = vy;
        d.v[i + 2 * n] = vz;
    }
    if (tid < d.n_dev) d.ev->reach_step[tid] = my_reach;
    if (tid == 0) ob.store(d, step);
}


// ---- symmetric variant for 896 < n <= 1024 (the 1024-body ensemble of BASELINE config 4) -------------------------------
// Same contract as traj_kernel, FAST math only.  Every UNORDERED pair of bodies in different groups is evaluated once and
// feeds both accelerations (20 FP64 instructions per unordered pair instead of 2 x 16), as in nb_sym.cu:
//   * 8 warps, warp w owns group w = bodies [128w, 128w + 128), 4 per lane, in registers {x, y, z, G*m, ax, ay, az, vx, vy, vz};
//   * group pairs (w, w+1), (w, w+2), (w, w+3) (mod 8) are warp w's, symmetric: the 128 j bodies of the other group pass
//     through the warp 32 at a time, one per lane, rotating through the lanes by warp shuffles with their own
//     acceleration accumulators; what a j body has collected is left in shared memory for its owner;
//   * the warp's own group (w, w) is evaluated one-sided (ordered pairs, broadcast reads); the opposite group (w, w+4)
//     is shared half and half with its owner, symmetric too;
//   * after one block barrier every lane adds the three partial sums other warps left for its bodies (fixed order:
//     deterministic), integrates (nbody.cc:77-88) and writes the new record; observers as in traj_kernel.
// FP64 instructions per body-step: 128*16 + 3*128*20 + 64*20 = 86 per j group against 8*16 = 128 for the one-sided kernel.
constexpr int TS_WARPS = 8, TS_G = 128, TS_I = 4;

__global__ void __launch_bounds__(32 * TS_WARPS, 1)
traj_sym_kernel(const TrajDesc* __restrict__ descs, const double* __restrict__ fst) {
    extern __shared__ __align__(32) unsigned char ts_smem[];
    double4* pos = reinterpret_cast<double4*>(ts_smem);                                   // [2][1024] {x, y, z, G*m_eff}
    double* stg = reinterpret_cast<double*>(ts_smem + 2 * 1024 * sizeof(double4));        // [8 warps][4 targets][3][128]
    const TrajDesc d = descs[blockIdx.x];
    const int n = d.n;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int src_lane = (lane + 1) & 31;

    // owner state: body b(k) = 128w + 32k + lane
    double vx[TS_I], vy[TS_I], vz[TS_I];
#pragma unroll
    for (int k = 0; k < TS_I; k++) {
        const int b = TS_G * w + 32 * k + lane;
        double x = 0, y = 0, z = 0, gm = 0;
        vx[k] = vy[k] = vz[k] = 0.0;
        if (b < n) {
            x = d.q[b], y = d.q[b + n], z = d.q[b + 2 * n];
            vx[k] = d.v[b], vy[k] = d.v[b + n], vz[k] = d.v[b + 2 * n];
            gm = d.is_device[b] ? 0.0 : gm_eff(d.m[b], false, 0.0);
        }
        pos[b] = make_double4(x, y, z, gm);  // bodies n .. 1023: zero mass at the origin (never written back)
        pos[1024 + b] = make_double4(x, y, z, gm);
    }
    int my_dev = -1, my_reach = -2;
    double my_m0 = 0.0;
    if (tid < d.n_dev) {
        my_dev = d.dev_index[tid];
        my_m0 = d.m[my_dev];
        my_reach = d.ev->reach_step[tid];
    }
    Observed ob;
    ob.load(d.ev);
    const int kind = d.kind;
    const int P = d.planet, A = d.asteroid, DD = d.destroy_device;
    const bool armed = q3_armed(kind, DD, n, d.m);
    __syncthreads();

    int cur = 0;
    int step = d.step_begin;
    bool stop = (kind >= NB_KIND_Q2) && ob.hit_step != -2;

    auto records = [&](int b) {
        return [=](int r, double& x, double& y, double& z) {
            const double4 p = pos[b * 1024 + r];
            x = p.x, y = p.y, z = p.z;
        };
    };

    // the observers of this step; the traj kernels stop at the hit
    auto observe = [&]() {
        if (observe_step<1>(ob, step, kind, P, A, armed, DD, &my_dev, &my_reach, records(cur)) & OBS_HIT) stop = true;
    };
    if (d.ev->steps_done < step && !stop) observe();

    while (!stop && step < d.step_end) {
        ++step;
        // (1) G*m_eff of the devices for this step (nbody.cc:61-64); a destroyed device has mass 0
        if (my_dev >= 0) pos[cur * 1024 + my_dev].w = device_gm(kind, my_dev, DD, ob, my_m0, fst, step);
        __syncthreads();
        const double4* cp = pos + cur * 1024;
        double xi[TS_I], yi[TS_I], zi[TS_I], gi[TS_I], ax[TS_I], ay[TS_I], az[TS_I];
#pragma unroll
        for (int k = 0; k < TS_I; k++) {
            const double4 p = cp[TS_G * w + 32 * k + lane];
            xi[k] = p.x, yi[k] = p.y, zi[k] = p.z, gi[k] = p.w;
            ax[k] = ay[k] = az[k] = 0.0;
        }
        // (2a) own group, one-sided: every lane reads the same j record; the self term is exactly zero
        {
            const double4* gj = cp + TS_G * w;
#pragma unroll 2
            for (int j = 0; j < TS_G; j++) {
                const double4 b = gj[j];
                double c[TS_I], dx[TS_I], dy[TS_I], dz[TS_I];
#pragma unroll
                for (int k = 0; k < TS_I; k++) pair_coeff_fast(xi[k], yi[k], zi[k], b.x, b.y, b.z, b.w, c[k], dx[k], dy[k], dz[k]);
#pragma unroll
                for (int k = 0; k < TS_I; k++) pair_accum_fast(c[k], dx[k], dy[k], dz[k], ax[k], ay[k], az[k]);
            }
        }
        // (2b) groups w+1, w+2, w+3: symmetric, the j bodies rotate through the lanes.  The opposite group w+4 is shared
        //      with its owner: warps 0..3 take the first 64 bodies of it against all their own, warps 4..7 take all 128
        //      bodies of it against the second 64 of their own (register slots 2 and 3) - together every pair once.
#pragma unroll 1
        for (int dg = 1; dg <= 4; dg++) {
            const double4* gj = cp + TS_G * ((w + dg) & 7);
            double* out = stg + ((w * 4 + (dg - 1)) * 3) * TS_G;
            const int jn = (dg == 4 && w < 4) ? TS_G / 2 : TS_G;
            if (dg == 4 && w >= 4) {
#pragma unroll 1
                for (int s0 = 0; s0 < TS_G; s0 += 32) {
                    const double4 b = gj[s0 + lane];
                    double jx = b.x, jy = b.y, jz = b.z, jg = b.w;
                    double ajx = 0.0, ajy = 0.0, ajz = 0.0;
#pragma unroll 4
                    for (int r = 0; r < 32; r++) {
                        const double nx = __shfl_sync(0xffffffffu, jx, src_lane), ny = __shfl_sync(0xffffffffu, jy, src_lane),
                                     nz = __shfl_sync(0xffffffffu, jz, src_lane), ng = __shfl_sync(0xffffffffu, jg, src_lane);
#pragma unroll
                        for (int k = TS_I / 2; k < TS_I; k++)
                            pair_sym(xi[k], yi[k], zi[k], gi[k], jx, jy, jz, jg, ax[k], ay[k], az[k], ajx, ajy, ajz);
                        ajx = __shfl_sync(0xffffffffu, ajx, src_lane), ajy = __shfl_sync(0xffffffffu, ajy, src_lane),
                        ajz = __shfl_sync(0xffffffffu, ajz, src_lane);
                        jx = nx, jy = ny, jz = nz, jg = ng;
                    }
                    out[s0 + lane] = ajx, out[TS_G + s0 + lane] = ajy, out[2 * TS_G + s0 + lane] = ajz;
                }
                continue;
            }
#pragma unroll 1
            for (int s0 = 0; s0 < jn; s0 += 32) {
                const double4 b = gj[s0 + lane];
                double jx = b.x, jy = b.y, jz = b.z, jg = b.w;
                double ajx = 0.0, ajy = 0.0, ajz = 0.0;
#pragma unroll 2
                for (int r = 0; r < 32; r++) {
                    const double nx = __shfl_sync(0xffffffffu, jx, src_lane), ny = __shfl_sync(0xffffffffu, jy, src_lane),
                                 nz = __shfl_sync(0xffffffffu, jz, src_lane), ng = __shfl_sync(0xffffffffu, jg, src_lane);
#pragma unroll
                    for (int k = 0; k < TS_I; k++)
                        pair_sym(xi[k], yi[k], zi[k], gi[k], jx, jy, jz, jg, ax[k], ay[k], az[k], ajx, ajy, ajz);
                    ajx = __shfl_sync(0xffffffffu, ajx, src_lane), ajy = __shfl_sync(0xffffffffu, ajy, src_lane),
                    ajz = __shfl_sync(0xffffffffu, ajz, src_lane);
                    jx = nx, jy = ny, jz = nz, jg = ng;
                }
                out[s0 + lane] = ajx, out[TS_G + s0 + lane] = ajy, out[2 * TS_G + s0 + lane] = ajz;  // home again after 32 moves
            }
        }
        __syncthreads();
        // (3) a = own sums + what warps w-1, w-2, w-3 left for this group; v += a*dt; q += v*dt (nbody.cc:77-88)
        double4* np = pos + (cur ^ 1) * 1024;
#pragma unroll
        for (int k = 0; k < TS_I; k++) {
            const int off = 32 * k + lane;
            double a0 = ax[k], a1 = ay[k], a2 = az[k];
#pragma unroll
            for (int dg = 1; dg <= 4; dg++) {
                // the opposite warp (dg == 4): warps 0..3 left sums for the first 64 bodies of this group only
                if (dg == 4 && w >= 4 && k >= TS_I / 2) continue;
                const double* in = stg + ((((w - dg) & 7) * 4 + (dg - 1)) * 3) * TS_G;
                a0 += in[off], a1 += in[TS_G + off], a2 += in[2 * TS_G + off];
            }
            double x = xi[k], y = yi[k], z = zi[k];
            kick_drift(a0, vx[k], x);
            kick_drift(a1, vy[k], y);
            kick_drift(a2, vz[k], z);
            double4* rec = np + TS_G * w + off;
            rec->x = x, rec->y = y, rec->z = z;  // .w: static G*m (devices: rewritten at the top of every step)
        }
        __syncthreads();
        cur ^= 1;
        observe();
    }

    // write back
#pragma unroll
    for (int k = 0; k < TS_I; k++) {
        const int b = TS_G * w + 32 * k + lane;
        if (b < n) {
            const double4 p = pos[cur * 1024 + b];
            d.q[b] = p.x, d.q[b + n] = p.y, d.q[b + 2 * n] = p.z;
            d.v[b] = vx[k], d.v[b + n] = vy[k], d.v[b + 2 * n] = vz[k];
        }
    }
    if (tid < d.n_dev) d.ev->reach_step[tid] = my_reach;
    if (tid == 0) ob.store(d, step);
}

int launch_sym(int n_traj, const TrajDesc* descs, const double* fst, cudaStream_t stream) {
    const size_t smem = 2 * 1024 * sizeof(double4) + (size_t)TS_WARPS * 4 * 3 * TS_G * sizeof(double);
    NB_CUDA(cudaFuncSetAttribute(traj_sym_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    traj_sym_kernel<<<n_traj, 32 * TS_WARPS, smem, stream>>>(descs, fst);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

template <int MATH, int JS>
int launch(int n, int n_traj, const TrajDesc* descs, const double* fst, cudaStream_t stream) {
    const size_t smem = (size_t)4 * n * sizeof(double2);
    NB_CUDA(cudaFuncSetAttribute(traj_kernel<MATH, JS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = ((n * JS + 31) / 32) * 32;
    traj_kernel<MATH, JS><<<n_traj, threads, smem, stream>>>(descs, fst);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

}  // namespace

int traj_js_for(int math, int n) {
    if (math == NB_MATH_STRICT) return 1;
    int js = 1;
    while (js < 32 && n * js * 2 <= 1024) js *= 2;
    return js;
}

int launch_traj_batch(int math, int n, int n_traj, const TrajDesc* descs, const double* fst, cudaStream_t stream) {
    if (n < 1 || n > NB_MAX_SMALL_N || n_traj < 1) return NB_ERR_ARG;
    if (math == NB_MATH_STRICT) return launch<MATH_STRICT, 1>(n, n_traj, descs, fst, stream);
    if (math != NB_MATH_FAST) return NB_ERR_ARG;
    // 896 < n <= 1024 (the 1024-body ensemble): the symmetric kernel (DESIGN 4.2: 115 us per step against the one-sided
    // kernel's 157 us)
    if (n > 1024 - TS_G && n <= 1024) return launch_sym(n_traj, descs, fst, stream);
    switch (traj_js_for(math, n)) {
        case 1: return launch<MATH_FAST, 1>(n, n_traj, descs, fst, stream);
        case 2: return launch<MATH_FAST, 2>(n, n_traj, descs, fst, stream);
        case 4: return launch<MATH_FAST, 4>(n, n_traj, descs, fst, stream);
        case 8: return launch<MATH_FAST, 8>(n, n_traj, descs, fst, stream);
        case 16: return launch<MATH_FAST, 16>(n, n_traj, descs, fst, stream);
        default: return launch<MATH_FAST, 32>(n, n_traj, descs, fst, stream);
    }
}

}  // namespace nb
