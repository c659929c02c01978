// Whole-GPU persistent trajectory kernel: ONE system (or two systems of the same n in lock step) spread over
// up to 128 SMs, all steps and observers in one launch.  This is the low-step-latency path for the b128 ... b1024
// queries: a single block needs ~133 us per b1024 step (nb_traj.cu), the FP64 floor over 128 SMs is ~1.05 us.
//
// Replaces the host-driven per-step launch sequence of the reference (hw5.cu:368-404, 387-403, 489-508: 3-4
// kernel launches per step, 600 000-800 000 per trajectory).  Arithmetic: nbody.cc:51-89.
//
// Block c owns bodies [8c, 8c+8).  Every step each block needs the new positions of ALL bodies, so the step
// latency is  hop (publish -> everybody has it)  +  pair loop  +  reduction/integration,  and the design goal
// is a hop of about one L2 round trip:
//
//   * publish: a body leaves as one naturally aligned 32-byte sector {x, y, z, self-checking tag} (one 256-bit store)
//     into a global record array double-buffered by step parity (L2 resident).  No fence, no atomic, no flag:
//     a sector is the unit the L2 reads and writes, so a reader sees it entirely old or entirely new and the
//     tag validates the data it travels with.
//   * fetch: one elected thread per block copies records with 1-D TMA bulk copies (cp.async.bulk, SASS UBLKCP)
//     straight into shared memory, WITHOUT polling first: all blocks run in lock step, so a block's own
//     publish time predicts everybody else's; the copy is issued a tuned delay after it.  Blocks form clusters
//     of CS (default 4): block r of a cluster copies slice r of the record array and MULTICASTS it into the
//     shared memory of all CS blocks, so the L2 serves 1/CS of the all-to-all traffic (4 MB -> 1 MB per b1024
//     step; the L2 read bandwidth, not only its latency, bounds a 128-reader all-to-all).
//   * validate: when the copies have landed, the 256 compute threads check every record's tag (4 each).  A record
//     that was copied before its publication is stale: its thread polls that one sector in global memory and
//     patches shared memory.  This is also what keeps the blocks in lock step - a block that runs ahead finds
//     the slowest block's records stale and waits for them, nothing else synchronises the grid.  Correctness
//     therefore never depends on the delay, only the speed does.
//   * buffer reuse is safe without fences by data dependence: a block overwrites its step s-2 sectors (and a
//     TMA overwrites the step s-2 stage in shared memory) only after its step s-1 data reached everybody, and
//     every block publishes step s-1 only after it finished reading step s-2.
//
// Warp roles (384 threads = 12 warps: compute warp groups 0-3 and 4-7, helper warp group 8-11; registers are re-allocated
// between them with setmaxnreg, see REG_COMPUTE below):
//   * 8 COMPUTE warps = 2 body groups x 4 j-quarters: warp w holds bodies 8c + 4(w>>2) .. +3 in registers and
//     takes records 128k + 32(w&3) + lane: four i-bodies share every j record read from shared memory
//     (conflict-free LDS.128 pairs: lanes with bit 2 set read the record's second half first).  A transposing
//     xor butterfly (18 64-bit shuffles for 12 sums) leaves the sums in lanes 0/8/16/24; the four quarters
//     meet in shared memory and 24 threads of warp 0 integrate one body component each (v += a*dt,
//     q += v*dt), gather x, y, z by shuffle and publish.
//   * 1 OBSERVER warp: hit test, minimum distance, missile reach/destroy (hw5.cu:241-309) on the complete
//     positions of every step, off the critical path.  It also owns the gravity devices' masses: the mass
//     column is double-buffered by step parity and the observer writes G*m_eff(step+2) of every device into
//     the next stage, so the pair loop is oblivious to devices.  The one step on which a device is destroyed
//     (its mass was written speculatively) is redone by the compute warps with the corrected column.
//   * 1 PRODUCER thread: arms the stage's mbarrier with the expected byte count and issues the TMA copies.
//   * lock-step launches (two systems per launch): 1 INTEGRATOR warp takes the serial tail of a step (sum of the j-parts,
//     integration, publication) from warp 0, the compute warps only arrive at its barrier and go on to the other system.
//   * the last warp of the helper warp group is idle.
//
// Spins are bounded (clock64) and raise `status`; co-residency comes from the cooperative launch
// (grid <= SM count, 1 block/SM).
//
// Measured on B200, b1024 (profiles/r01_grid_exchange_v2.md, r02_grid_exchange.md): 3.30 us/step for one system (round 1,
// step-only tags: 3.2-3.4) against 4.4-4.9 us for the first exchange (per-producer sentinel poll, then LDG
// fetch warps: two dependent L2 round trips per step); in-kernel phases per step at 1.96 GHz: copy wait 1450 clk
// (closed-loop delay + TMA round trip), validate 1130, pairs 2430 (FP64 floor 2184), butterfly 415, integrate+publish 550.
// Tried and measured worse: validating inside the pair loop (a vote per record batch serialises the loop),
// optimistic pair loop + redo on a stale record (a redone block is late, all others find it stale: cascade),
// per-block adaptive delays (creep up together), rotating the tag slot for conflict-free validation loads.
#include <cstdint>
#include <cstdio>
#include <chrono>
#include <cstdlib>
#include <map>
#include <mutex>
#include <set>
#include <string>
#include <tuple>

#include "nb_internal.h"
#include "nb_math.cuh"
#include "nb_observe.cuh"

namespace nb {

namespace {

// Register re-allocation between the warp roles (setmaxnreg, sm_90a+).  With 10 warps two of the four schedulers hold three
// warps, so no thread can have more than 168 registers, and at 166 ptxas serialises the four pair chains of a record
// (its own stall counts: 363 cycles per 8 pairs, 416 - 462 in the two-system kernel).  The block is launched with 12 warps
// instead (the helper warp group 8 - 11: observer, producer, integrator, idle warp), the helpers shrink to REG_HELPER
// registers and the eight compute warps grow to REG_COMPUTE: 320 cycles per 8 pairs, pairs phase 2860 -> 2430 clk
// (FP64 pipe 76 -> 90 % busy in that phase), b1024 3.38 -> 3.30 us per step, 1-GPU solve 1.23 -> 1.19 s (224 / 56: 3.36 /
// 1.205, the observer spills; 216 / 72: 3.30 / 1.19; 200 / 104: 3.37 / 1.19).  The pool is what the launch allocated: the
// increase WAITS until 8 x compute + 4 x helper <= 12 x 168 - a larger request hangs the kernel.
constexpr int REG_COMPUTE = 208, REG_HELPER = 88;
static_assert(8 * REG_COMPUTE + 4 * REG_HELPER <= 12 * 168 && REG_COMPUTE % 8 == 0 && REG_HELPER % 8 == 0 && REG_HELPER >= 24 &&
                  REG_COMPUTE <= 232,
              "setmaxnreg: the compute warps' increase must fit into what the helper warps release");

constexpr int PAIR_UNROLL = 2;   // records per trip of the pair loop (4 pairs each)
constexpr int GB = 8;            // bodies per block
constexpr int BPW = 4;           // bodies per compute warp
constexpr int NJ = 4;            // compute warps = 2 body groups x NJ j-parts; then the helper warp group
constexpr int NTHREADS = 384;    // 8 compute warps + observer, producer (lane 0 only), integrator and idle warp
constexpr int MAX_T = 2;         // systems per launch (shared memory: 80 B per record each)
constexpr int MAX_CS = 8;        // largest cluster
constexpr int RPAD = 256;        // shared-memory stages hold a multiple of this many records (the tail beyond R: zero mass)
constexpr int FLAG_STOP = 1, FLAG_REDO = 2;
constexpr long long SPIN_LIMIT = 4000000000LL;  // ~2 s of SM clocks
constexpr int NPROF = 24;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// one naturally aligned 32-byte sector per access (SASS LDG/STG.E.ENL2.256)
__device__ __forceinline__ void ld_sector(const double* p, double& a, double& b, double& c, double& d) {
    asm volatile("ld.relaxed.gpu.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_sector(double* p, double a, double b, double c, double d) {
    asm volatile("st.relaxed.gpu.global.v4.f64 [%4], {%0,%1,%2,%3};" ::"d"(a), "d"(b), "d"(c), "d"(d), "l"(p) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// 1-D TMA bulk copy global -> shared memory of this block; completion (bytes) counted on the block's mbarrier
__device__ __forceinline__ void tma_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// the same, delivered to the same shared-memory offset (and mbarrier) of every block in cta_mask
__device__ __forceinline__ void tma_load_multicast(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
// named barrier 1: the compute warps
__device__ __forceinline__ void compute_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * 2 * NJ) : "memory"); }

// Record layout: one 32-byte sector {x, y, z, tag}.  The tag is SELF-CHECKING: step in the upper 32 bits, a 32-bit
// fold of the bit patterns of x, y and z in the lower 32, so a record is accepted only if all four words belong
// together.  The design relies on a naturally aligned 32-byte access being one L2 sector transaction (see the header
// comment), which the PTX memory model does not promise for vector or bulk accesses; with this tag a torn record - any
// mixture of words of two publications - fails the check (up to a 2^-32 coincidence per torn record) and is fetched
// again instead of being consumed.  Two checks: the STEP check needs the tag word only (a record that was copied
// before its publication is old in all four words: the common case, handled in the validation pass); both are made in
// the validation pass (validate_stage, kept out of line so that the pair loop's code generation does not depend on it).
__device__ __forceinline__ unsigned fold32(double x, double y, double z) {
    // rot13(the four words of the record's first half) ^ the two words of z: two 3-input LOP3, one funnel shift, one LOP3 -
    // the check is on the serial path of every step (publication) and is made for every record of every step (validation)
    const unsigned lx = (unsigned)__double2loint(x), hx = (unsigned)__double2hiint(x), ly = (unsigned)__double2loint(y),
                   hy = (unsigned)__double2hiint(y), lz = (unsigned)__double2loint(z), hz = (unsigned)__double2hiint(z);
    const unsigned h = lx ^ hx ^ ly ^ hy;
    return __funnelshift_l(h, h, 13) ^ lz ^ hz;
}
// the same check on a record as the validation pass holds it: two 16-byte halves A (read first) and B, which of them is the
// record's first half depends on the lane (hsel: conflict-free LDS.128 pairs).  Four selects instead of swapping eight words.
__device__ __forceinline__ bool halves_ok(double2 A, double2 B, int hsel, int step) {
    const unsigned pa = (unsigned)__double2loint(A.x) ^ (unsigned)__double2hiint(A.x) ^ (unsigned)__double2loint(A.y);
    const unsigned pb = (unsigned)__double2loint(B.x) ^ (unsigned)__double2hiint(B.x) ^ (unsigned)__double2loint(B.y);
    const unsigned sa = (unsigned)__double2hiint(A.y), sb = (unsigned)__double2hiint(B.y);
    // first half {x, y}: all four words; second half {z, tag}: z's two words and the tag's low word, the tag's high word is the step
    const unsigned first = (hsel ? pb ^ sb : pa ^ sa), second = hsel ? pa : pb, stp = hsel ? sa : sb;
    return (int)stp == step && (__funnelshift_l(first, first, 13) ^ second) == 0u;
}
__device__ __forceinline__ double make_tag(int step, double x, double y, double z) {
    return __hiloint2double(step, (int)fold32(x, y, z));
}
__device__ __forceinline__ bool tag_step_is(double tg, int step) { return __double2hiint(tg) == step; }
__device__ __forceinline__ bool tag_ok(double tg, int step, double x, double y, double z) {
    return __double2hiint(tg) == step && (unsigned)__double2loint(tg) == fold32(x, y, z);
}

struct Shared {
    // stage = step parity.  full: the copies of all R records have landed (1 arrival = the producer's expect_tx, plus
    // the bytes); obs: the observer has judged the step (1 arrival).  Each completes once per two steps.
    alignas(8) uint64_t full[MAX_T][2];
    alignas(8) uint64_t obs[MAX_T][2];
    alignas(8) uint64_t trig[MAX_T][2];  // producer trigger: this block's sums of the step are complete (1 arrival)
    volatile int flags[MAX_T][2];   // FLAG_* of the step held by the stage, valid once obs completed
    volatile int stop[MAX_T];
    volatile int abort;
    volatile int delay[MAX_T];      // copy delay after the trigger (clk): a constant, or steered by stale_own (adaptive mode)
    volatile int stale_own[MAX_T];  // this step's validation found stale records in the slice this block's producer copied
    double part[MAX_T][2][2 * NJ][3 * BPW];  // per compute warp: sums {ax, ay, az} of its 4 bodies over its j-part
};

struct ObsState {  // per system, observer warp
    int n_dev, kind, Prec, Arec, DDrec, DD, step, step_begin, step_end;
    bool q3_armed, active, observed;
    Observed ev;
    int my_dev[2], my_reach[2];  // devices lane and lane + 32 of the system's list (-1: none): up to NB_MAX_DEVICES = 64
    double my_m0[2];
};

// The validation pass of the compute warps (256 threads, thread tid checks records tid + 256k): every record of the stage
// must pass the FULL self-check for step `st`.  A record that does not was copied before its publication (stale: the
// common case, and how the fast blocks wait for the slowest) or is torn: its thread polls that sector in global memory
// until it passes and patches shared memory.  A function of its own, force-inlined: the FP64 pair loop's register allocation
// is sensitive to what is inlined around it (measured on B200, b1024, us per step: validation written inline in the step loop
// 3.80, this function force-inlined 3.40, out of line 3.49; round 1's tag-only check 3.21).
__device__ __forceinline__ bool validate_stage(double* pos, const double* grec, int R, int st, int tid, int hsel, volatile int* abort_flag,
                                               int* status, unsigned long long* n_stale, int own_lo, int own_hi, volatile int* stale_own) {
    bool patched = false;
    constexpr int NTHR = 32 * 2 * NJ;             // the compute warps
    constexpr int NK = (1024 + NTHR - 1) / NTHR;  // records per thread (n <= 1024)
    double2 va[NK], vb[NK];  // whole records, conflict-free LDS.128 pairs (lanes with bit 2 set read the second half first)
#pragma unroll
    for (int k = 0; k < NK; k++) {
        const int r = min(tid + NTHR * k, R - 1);
        va[k] = *reinterpret_cast<const double2*>(pos + 4 * r + 2 * hsel);
        vb[k] = *reinterpret_cast<const double2*>(pos + 4 * r + 2 * (hsel ^ 1));
    }
#pragma unroll
    for (int k = 0; k < NK; k++) {
        const int r = tid + NTHR * k;
        if (r < R && !halves_ok(va[k], vb[k], hsel, st)) {
            double x, y, z, tg;
            const long long t0 = clock64();
            do {
                ld_sector(grec + 4 * (size_t)r, x, y, z, tg);
                if (*abort_flag) break;
                if (clock64() - t0 > SPIN_LIMIT) {
                    *abort_flag = 1;
                    atomicExch(status, 1);
                    break;
                }
            } while (!tag_ok(tg, st, x, y, z));
            // right step, wrong fold: a TORN record (word 1 of the status block)
            if (tag_step_is(hsel ? va[k].y : vb[k].y, st)) atomicAdd(status + 1, 1);
            pos[4 * r] = x, pos[4 * r + 1] = y, pos[4 * r + 2] = z;
            __threadfence_block();
            pos[4 * r + 3] = tg;
            patched = true;
            (*n_stale)++;
            if (r >= own_lo && r < own_hi) *stale_own = 1;
        }
    }
    return patched;
}

// PROFILE: block 0 thread 0 accumulates clock64 per phase (NB_GRID_PROFILE=1)
// T systems per launch: one set of compute warps steps them in turn (lock step)
template <int T, bool PROFILE>
__global__ void __launch_bounds__(NTHREADS, 1)
grid_traj_kernel(const TrajDesc* __restrict__ descs, const double* __restrict__ fst, double* __restrict__ gbuf,
                 long long* __restrict__ prof, int* __restrict__ status, int R, int delay_clk, int delay_single, int adapt_up,
                 int adapt_down) {
    extern __shared__ __align__(128) double smem[];
    __shared__ Shared sh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = blockIdx.x;
    const int n = descs[0].n;
    constexpr int NCW = 2 * NJ, W_OBS = NCW, W_PROD = W_OBS + 1, W_INT = W_PROD + 1, RQ = 32 * NJ;
    // With several systems in lock step, warp W_INT is the INTEGRATOR: the compute warps only ARRIVE at the barrier behind their
    // reduction and go on to the next system, the integrator waits there, sums the j-parts, integrates and publishes (two systems:
    // 1-GPU solve 1.18 -> 1.14 s).  With one system nothing else could use the time, and the hand-over costs it 130 clk per step
    // (measured: 3.30 -> 3.43 us), so warp 0 of the compute warps integrates.
    constexpr bool USE_INT = T > 1;
    constexpr int BAR_INT = 2;  // named barriers BAR_INT + t: the compute warps arrive, the integrator waits (32 * (NCW + 1) threads)
    const int RS = (R + RPAD - 1) / RPAD * RPAD;  // records per stage in shared memory (tail beyond R: zero mass, never copied)
    // per system: pos[2][RS] records {x, y, z, tag} then gm[2][RS]
    auto s_pos = [&](int t, int stage) { return smem + (size_t)t * 10 * RS + (size_t)stage * 4 * RS; };
    auto s_gm = [&](int t, int stage) { return smem + (size_t)t * 10 * RS + 8 * RS + (size_t)stage * RS; };
    auto g_rec = [&](int t, int st) { return gbuf + ((size_t)(st & 1) * T + t) * (size_t)R * 4; };

    if (PROFILE && tid == 0) {  // globaltimer (ns) at block entry: prof[8] = min, prof[9] = max over blocks
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        atomicMin((unsigned long long*)&prof[8], g);
        atomicMax((unsigned long long*)&prof[9], g);
    }
    if (tid == 0) {
        sh.abort = 0;
#pragma unroll
        for (int t = 0; t < T; t++) {
            // a trajectory that stopped in an earlier launch never steps again
            sh.stop[t] = (descs[t].kind >= NB_KIND_Q2 && descs[t].ev->hit_step != -2) ? 1 : 0;
            sh.delay[t] = delay_clk;
            sh.stale_own[t] = 0;
            for (int b = 0; b < 2; b++) {
                mbar_init(&sh.full[t][b], 1);
                mbar_init(&sh.obs[t][b], 1);
                mbar_init(&sh.trig[t][b], 1);
                sh.flags[t][b] = 0;
            }
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // positions of step_begin (tagged) into stage (step_begin & 1); static G*m in both mass columns, the devices'
    // G*m_eff(step_begin + 1) in the current one (the observer fills the other)
#pragma unroll
    for (int t = 0; t < T; t++) {
        const TrajDesc& d = descs[t];
        const int sb = d.step_begin;
        double* p0 = s_pos(t, sb & 1);
        double* p1 = s_pos(t, (sb & 1) ^ 1);
        double* g0 = s_gm(t, sb & 1);
        double* g1 = s_gm(t, (sb & 1) ^ 1);
        const double f1 = fst[sb + 1];
        for (int r = tid; r < RS; r += NTHREADS) {
            double x = 0, y = 0, z = 0, ga = 0, gb = 0;
            if (r < n) {
                x = d.q[r], y = d.q[r + n], z = d.q[r + 2 * n];
                const bool dev = d.is_device[r];
                ga = gm_eff(d.m[r], dev, f1);
                gb = dev ? 0.0 : ga;
            }
            p0[4 * r] = x, p0[4 * r + 1] = y, p0[4 * r + 2] = z, p0[4 * r + 3] = make_tag(sb, x, y, z);
            p1[4 * r] = 0.0, p1[4 * r + 1] = 0.0, p1[4 * r + 2] = 0.0, p1[4 * r + 3] = make_tag(-1, 0.0, 0.0, 0.0);
            g0[r] = ga, g1[r] = gb;
        }
    }
    // the stages were filled through the generic proxy; the TMA (async proxy) overwrites them from the next step on
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    cluster_sync_all();  // every block's mbarriers exist before anybody multicasts into them

    // the sector of record r once it carries the tag of step `st`, polled in global memory
    auto poll_rec = [&](const double* grec, int r, int st, double& x, double& y, double& z, double& tg) {
        const long long t0 = clock64();
        do {
            ld_sector(grec + 4 * (size_t)r, x, y, z, tg);
            if (sh.abort) break;
            if (clock64() - t0 > SPIN_LIMIT) {
                sh.abort = 1;
                atomicExch(status, 1);
                break;
            }
        } while (!tag_ok(tg, st, x, y, z));  // the FULL self-check: all four words of one publication
    };
    // A record of step `st` for the observer: out of shared memory if it passes the self-check, else out of global memory.
    auto load_rec = [&](const double* pos, const double* grec, int r, int st, double& x, double& y, double& z) {
        // a record caught half patched by a compute thread (patch_rec) fails the self-check like any torn record and is
        // fetched from global memory instead
        const volatile double* vp = pos + 4 * r;
        double tg = vp[3];
        x = vp[0], y = vp[1], z = vp[2];
        if (!tag_ok(tg, st, x, y, z)) poll_rec(grec, r, st, x, y, z, tg);
    };
    // fetch a stale record from global memory and patch shared memory: coordinates, fence, then the tag
    auto patch_rec = [&](double* pos, const double* grec, int r, int st) {
        double x, y, z, tg;
        poll_rec(grec, r, st, x, y, z, tg);
        pos[4 * r] = x, pos[4 * r + 1] = y, pos[4 * r + 2] = z;
        __threadfence_block();
        pos[4 * r + 3] = tg;
    };
    // bounded wait on an mbarrier phase; false = aborted
    auto wait_bar = [&](uint64_t* bar, uint32_t parity) {
        if (mbar_try_wait(bar, parity)) return true;
        const long long t0 = clock64();
        while (!mbar_try_wait(bar, parity)) {
            if (sh.abort) return false;
            if (clock64() - t0 > SPIN_LIMIT) {
                sh.abort = 1;
                atomicExch(status, 1);
                return false;
            }
        }
        return true;
    };

    // two branches, each behind its own setmaxnreg (warp-group aligned: warps 0-3 and 4-7 compute, 8-11 help)
    if (warp >= W_OBS) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REG_HELPER));
    if (USE_INT && warp == W_INT) {
        // ------------------------------------------------------------------ INTEGRATOR warp (lane < 24: body 8c + lane/3, component lane%3)
        const int ib = lane / 3, ik = lane - 3 * ib, my_body = c * GB + ib;
        const bool integ = lane < 3 * GB, mine = integ && my_body < n;
        int istep[T], ibegin[T], iend[T];
        bool iact[T];
        double iq[T], iv[T];
        bool any = false;
#pragma unroll
        for (int t = 0; t < T; t++) {
            const TrajDesc& d = descs[t];
            istep[t] = ibegin[t] = d.step_begin, iend[t] = d.step_end;
            iact[t] = !((d.kind >= NB_KIND_Q2) && d.ev->hit_step != -2);
            iq[t] = mine ? d.q[ik * n + my_body] : 0.0;
            iv[t] = mine ? d.v[ik * n + my_body] : 0.0;
            any |= iact[t];
        }
        bool aborted = false;
        while (any && !aborted) {
#pragma unroll
            for (int t = 0; t < T; t++) {
                if (!iact[t]) continue;
                const int st = istep[t], stage = st & 1;
                // the observer's verdict on step st, as the compute warps read it: on STOP they do not come to the barrier
                const int flags = wait_bar(&sh.obs[t][stage], (uint32_t)((st - ibegin[t]) >> 1) & 1u) ? (int)sh.flags[t][stage] : (int)FLAG_STOP;
                if (flags & FLAG_STOP) {
                    iact[t] = false;
                    continue;
                }
                asm volatile("bar.sync %0, %1;" ::"r"(BAR_INT + t), "n"(32 * (NCW + 1)) : "memory");  // the eight warps' sums are in sh.part
                if (sh.abort) {
                    aborted = true;
                    break;
                }
                // a = sum of the j-parts; v += a*dt; q += v*dt (nbody.cc:77-88); publish the body as one tagged sector, unfenced
                if (lane == 0) mbar_arrive(&sh.trig[t][(st + 1) & 1]);  // producer trigger: everybody publishes within ~150 clk
                if (integ) {
                    const double* p = &sh.part[t][stage][(ib >> 2) * NJ][3 * (ib & 3) + ik];
                    double a = p[0];
#pragma unroll
                    for (int j = 1; j < NJ; j++) a += p[j * 3 * BPW];  // fixed order: deterministic
                    if (my_body < n) kick_drift(a, iv[t], iq[t]);
                }
                const double qy = __shfl_down_sync(0xffffffffu, iq[t], 1);
                const double qz = __shfl_down_sync(0xffffffffu, iq[t], 2);
                if (integ && ik == 0) st_sector(g_rec(t, st + 1) + 4 * (size_t)my_body, iq[t], qy, qz, make_tag(st + 1, iq[t], qy, qz));
                istep[t] = st + 1;
            }
            any = false;
#pragma unroll
            for (int t = 0; t < T; t++) any |= iact[t];
        }
        if (mine) {
#pragma unroll
            for (int t = 0; t < T; t++) {
                descs[t].q[ik * n + my_body] = iq[t];
                descs[t].v[ik * n + my_body] = iv[t];
            }
        }
    } else if (warp >= W_INT) {
        // idle: the last warp of the helper warp group, and the integrator's with one system
    } else if (warp >= W_PROD) {
        // ------------------------------------------------------------------ PRODUCER thread
        if (lane == 0) {
            const uint32_t CS = cluster_nctarank(), rank = cluster_ctarank();
            const uint32_t slice = (uint32_t)R / CS;  // records per cluster rank (R is a multiple of 8*CS)
            const uint16_t mask = (uint16_t)((1u << CS) - 1u);
            int pstep[T];
            bool pact[T];
            bool any = false;
#pragma unroll
            for (int t = 0; t < T; t++) {
                pstep[t] = descs[t].step_begin;
                pact[t] = !sh.stop[t] && descs[t].step_end > descs[t].step_begin;
                any |= pact[t];
            }
            while (any && !sh.abort) {
                any = false;
#pragma unroll
                for (int t = 0; t < T; t++) {
                    if (!pact[t]) continue;
                    const int st = pstep[t] + 1;
                    // wait (hardware-suspended on the mbarrier, no issue slots taken from the compute warps) until this
                    // block's sums of step st are complete: it publishes within ~150 clk, and so does everybody
                    bool go = wait_bar(&sh.trig[t][st & 1], (uint32_t)((st - descs[t].step_begin - 1) >> 1) & 1u);
                    if (sh.stop[t]) go = false;
                    if (!go) {
                        pact[t] = false;
                        continue;
                    }
                    const long long t1 = clock64();
                    uint64_t* bar = &sh.full[t][st & 1];
                    mbar_arrive_expect_tx(bar, (uint32_t)R * 32u);
                    // Copy delay after the trigger: long enough for everybody's sectors of this step to be in the L2 when the
                    // copy reads them.  The blocks keep in step only through the data; whoever copies too early finds stale
                    // tags and polls (validation below), so the delay is a speed knob, not a correctness condition.
                    int dl = adapt_up > 0 ? sh.delay[t] : delay_clk;
                    if (T > 1 && adapt_up <= 0) {  // the only system still running in this launch waits for every copy: shortest delay
                        int n_act = 0;
#pragma unroll
                        for (int w = 0; w < T; w++) n_act += pact[w] ? 1 : 0;
                        if (n_act == 1) dl = delay_single;
                    }
                    while (clock64() - t1 < dl) {
                    }
                    double* dst = s_pos(t, st & 1) + (size_t)rank * slice * 4;
                    const double* src = g_rec(t, st) + (size_t)rank * slice * 4;
                    if (CS == 1)
                        tma_load(dst, src, slice * 32u, bar);
                    else
                        tma_load_multicast(dst, src, slice * 32u, bar, mask);
                    pstep[t] = st;
                    if (st >= descs[t].step_end) pact[t] = false;
                    any |= pact[t];
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ OBSERVER warp
        ObsState os[T];
        bool any = false;
#pragma unroll
        for (int t = 0; t < T; t++) {
            const TrajDesc& d = descs[t];
            ObsState& s = os[t];
            s.n_dev = d.n_dev, s.kind = d.kind, s.DD = d.destroy_device;
            s.Prec = d.planet, s.Arec = d.asteroid;
            s.DDrec = (s.DD >= 0 && s.DD < n) ? s.DD : 0;
            s.step = s.step_begin = d.step_begin, s.step_end = d.step_end;
            s.ev.load(d.ev);
            s.q3_armed = q3_armed(s.kind, s.DD, n, d.m);
            s.active = !((s.kind >= NB_KIND_Q2) && s.ev.hit_step != -2);
            s.observed = d.ev->steps_done >= s.step;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                s.my_dev[h] = -1, s.my_reach[h] = -2, s.my_m0[h] = 0.0;
                if (lane + 32 * h < s.n_dev) {
                    s.my_dev[h] = d.dev_index[lane + 32 * h];
                    s.my_m0[h] = d.m[s.my_dev[h]];
                    s.my_reach[h] = d.ev->reach_step[lane + 32 * h];
                }
            }
            any |= s.active;
        }
        while (any && !sh.abort) {
            any = false;
#pragma unroll
            for (int t = 0; t < T; t++) {
                ObsState& s = os[t];
                if (!s.active) continue;
                const int st = s.step, stage = st & 1;
                if (st > s.step_begin && !wait_bar(&sh.full[t][stage], (uint32_t)((st - s.step_begin - 1) >> 1) & 1u)) {
                    s.active = false;
                    continue;
                }
                const double* pos = s_pos(t, stage);
                const double* grec = g_rec(t, st);
                int flags = 0;
                if (!s.observed) {
                    const int seen = observe_step<2>(s.ev, st, s.kind, s.Prec, s.Arec, s.q3_armed, s.DDrec, s.my_dev, s.my_reach,
                                                     [&](int r, double& x, double& y, double& z) { load_rec(pos, grec, r, st, x, y, z); });
                    if (seen == OBS_HIT) flags |= FLAG_STOP;
                    if (seen == OBS_DESTROYED) {
                        // the pair loop of this step ran (or runs) with the device's mass: redo it without
                        if (st < s.step_end) flags |= FLAG_REDO;
                        if (lane == 0) s_gm(t, stage)[s.DDrec] = 0.0;
                    }
                }
                if (st >= s.step_end) flags |= FLAG_STOP;
#pragma unroll
                for (int h = 0; h < 2; h++)
                    if (!(flags & FLAG_STOP) && s.my_dev[h] >= 0)  // mass column of the next step's positions: step st + 2
                        s_gm(t, stage ^ 1)[s.my_dev[h]] = device_gm(s.kind, s.my_dev[h], s.DD, s.ev, s.my_m0[h], fst, st + 2);
                __syncwarp();
                if (lane == 0) {
                    sh.flags[t][stage] = flags;
                    mbar_arrive(&sh.obs[t][stage]);  // release: the mass column writes above are visible to the waiters
                }
                s.observed = false;
                if (flags & FLAG_STOP)
                    s.active = false;
                else
                    s.step = st + 1;
                any |= s.active;
            }
        }
        // events (block 0 reports; every block computed the same)
        if (c == 0) {
#pragma unroll
            for (int t = 0; t < T; t++) {
                const TrajDesc& d = descs[t];
                ObsState& s = os[t];
#pragma unroll
                for (int h = 0; h < 2; h++)
                    if (lane + 32 * h < s.n_dev) d.ev->reach_step[lane + 32 * h] = s.my_reach[h];
                if (lane == 0) s.ev.store(d, s.step);
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REG_COMPUTE));
        // ------------------------------------------------------------------ COMPUTE warps
        const int bg = warp / NJ, part0 = warp % NJ;  // body group, j-part
        const int body0 = c * GB + bg * BPW;  // the warp's four bodies (records body0 .. body0+3)
        const int hsel = (lane >> 2) & 1;     // conflict-free LDS.128 pairs: these lanes read the second half first
        // integrator threads of one system (warp 0, lane < 24): body 8c + lane/3, component lane%3
        const int ib = lane / 3, ik = lane - 3 * ib;
        const int my_body = c * GB + ib;
        const bool integ = warp == 0 && lane < 3 * GB;

        int cstep[T], cbegin[T], cend[T];
        bool cact[T];
        double iq = 0.0, iv = 0.0;  // one system: position / velocity component of the integrator threads
        long long pacc[6] = {0, 0, 0, 0, 0, 0}, pt = 0;
        unsigned long long n_stale = 0;
        auto tick = [&](int phase) {
            if (PROFILE) {
                const long long now = clock64();
                pacc[phase] += now - pt;
                pt = now;
            }
        };
        bool any = false;
#pragma unroll
        for (int t = 0; t < T; t++) {
            const TrajDesc& d = descs[t];
            cstep[t] = cbegin[t] = d.step_begin, cend[t] = d.step_end;
            cact[t] = !((d.kind >= NB_KIND_Q2) && d.ev->hit_step != -2);
            if (!USE_INT) {
                const bool mine = integ && my_body < n;
                iq = mine ? d.q[ik * n + my_body] : 0.0;
                iv = mine ? d.v[ik * n + my_body] : 0.0;
            }
            any |= cact[t];
        }
        long long g0 = 0, c0 = 0;
        if (PROFILE) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0));
            c0 = clock64();
        }
        bool aborted = false;

        while (any && !aborted) {
#pragma unroll
            for (int t = 0; t < T; t++) {
                if (!cact[t]) continue;  // uniform across the grid
                if (PROFILE) pt = clock64();
                const int st = cstep[t], stage = st & 1;
                const bool last = st >= cend[t];
                // a failed wait has raised sh.abort: the warps still meet at this step's barriers and leave together below
                if (!last && st > cbegin[t]) wait_bar(&sh.full[t][stage], (uint32_t)((st - cbegin[t] - 1) >> 1) & 1u);
                tick(0);
                double* pos = s_pos(t, stage);
                const double* cg = s_gm(t, stage);
                const double* grec = g_rec(t, st);
                double ax[BPW], ay[BPW], az[BPW];
                int flags = 0;
                if (!last) {
                    // (0) validate: every record of the stage must carry this step's tag (thread tid checks records
                    //     tid + 256k; the tags of 32 consecutive records share 8 banks, so this pass is shared-memory bound: ~256 clk at
                    //     n = 1024).  A stale record was copied
                    //     before its publication - this is how the fast blocks wait for the slowest: poll that sector in global
                    //     memory and patch shared memory, each stale record by exactly one thread of the block.
                    const int own_lo = (int)cluster_ctarank() * (R / (int)cluster_nctarank());
                    // (measured worse with two systems in lock step: warps 1-7 validating while warp 0 still integrates and
                    // publishes the other system - 1.31 s against 1.27 s for the b1024 solve on one GPU)
                    const bool patched = validate_stage(pos, grec, R, st, tid, hsel, &sh.abort, status, &n_stale, own_lo,
                                                        own_lo + R / (int)cluster_nctarank(), &sh.stale_own[t]);
                    // generic-proxy writes to a buffer the async proxy (TMA) overwrites two steps later
                    if (patched) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    compute_bar();
                    if (adapt_up > 0 && tid == 0) {
                        // closed loop on the copy delay: stale records in the slice this block's producer copied = it copied
                        // too early (raise the delay by adapt_up); a clean step lowers it by adapt_down.  The slowest
                        // block never sees stale records, so ITS delay - the one on the critical path - decays to the floor.
                        int dcur = sh.delay[t];
                        if (sh.stale_own[t]) {
                            dcur = min(dcur + adapt_up, 1600);
                            sh.stale_own[t] = 0;
                        } else {
                            dcur = max(dcur - adapt_down, 0);
                        }
                        sh.delay[t] = dcur;
                    }
                }
                tick(5);
                // (1) forces on the warp's four bodies (nbody.cc:56-74) from j-part `jp` of the records
                auto pairs_part = [&](int jp) {
#pragma unroll
                    for (int i = 0; i < BPW; i++) ax[i] = ay[i] = az[i] = 0.0;
                    if (!last) {
                        double xi[BPW], yi[BPW], zi[BPW];
#pragma unroll
                        for (int i = 0; i < BPW; i++) {
                            const double* p = pos + 4 * (body0 + i);
                            xi[i] = p[0], yi[i] = p[1], zi[i] = p[2];
                        }
#pragma unroll PAIR_UNROLL
                        for (int r = 32 * jp + lane; r < RS; r += RQ) {
                            // conflict-free LDS.128 pair: lanes with bit 2 set read the record's second half first
                            const double2 A = *reinterpret_cast<const double2*>(pos + 4 * r + 2 * hsel);
                            const double2 B = *reinterpret_cast<const double2*>(pos + 4 * r + 2 * (hsel ^ 1));
                            const double jx = hsel ? B.x : A.x, jy = hsel ? B.y : A.y, jz = hsel ? A.x : B.x;
                            const double jg = cg[r];
#pragma unroll
                            for (int i = 0; i < BPW; i++) pair<MATH_FAST>(xi[i], yi[i], zi[i], jx, jy, jz, jg, ax[i], ay[i], az[i]);
                        }
                    }
                };
                // (3) transposing butterfly: 12 sums -> lanes 0/8/16/24 hold body 0/1/2/3; into the slot of (body group, j-part)
                auto butterfly_store = [&](int jp) {
                    const bool h16 = lane & 16, h8 = lane & 8;
                    double k[6];
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        // lanes with bit 4 clear keep bodies 0,1 and give away 2,3
                        const double sx = h16 ? ax[i] : ax[i + 2], sy = h16 ? ay[i] : ay[i + 2], sz = h16 ? az[i] : az[i + 2];
                        k[3 * i + 0] = (h16 ? ax[i + 2] : ax[i]) + __shfl_xor_sync(0xffffffffu, sx, 16);
                        k[3 * i + 1] = (h16 ? ay[i + 2] : ay[i]) + __shfl_xor_sync(0xffffffffu, sy, 16);
                        k[3 * i + 2] = (h16 ? az[i + 2] : az[i]) + __shfl_xor_sync(0xffffffffu, sz, 16);
                    }
                    double m0, m1, m2;
                    {
                        const double s0 = h8 ? k[0] : k[3], s1 = h8 ? k[1] : k[4], s2 = h8 ? k[2] : k[5];
                        m0 = (h8 ? k[3] : k[0]) + __shfl_xor_sync(0xffffffffu, s0, 8);
                        m1 = (h8 ? k[4] : k[1]) + __shfl_xor_sync(0xffffffffu, s1, 8);
                        m2 = (h8 ? k[5] : k[2]) + __shfl_xor_sync(0xffffffffu, s2, 8);
                    }
#pragma unroll
                    for (int o = 4; o > 0; o >>= 1) {
                        m0 += __shfl_xor_sync(0xffffffffu, m0, o);
                        m1 += __shfl_xor_sync(0xffffffffu, m1, o);
                        m2 += __shfl_xor_sync(0xffffffffu, m2, o);
                    }
                    if ((lane & 7) == 0) {
                        double* dstp = &sh.part[t][stage][bg * NJ + jp][3 * (lane >> 3)];
                        dstp[0] = m0, dstp[1] = m1, dstp[2] = m2;
                    }
                };
                for (int attempt = 0; attempt < 2; attempt++) {
                    pairs_part(part0);
                    tick(1);
                    // (2) the observer's verdict on the positions of step st
                    flags = wait_bar(&sh.obs[t][stage], (uint32_t)((st - cbegin[t]) >> 1) & 1u) ? sh.flags[t][stage] : 0;
                    if (!(flags & FLAG_REDO)) break;  // else: the device was destroyed at this very step, once per trajectory
                }
                tick(2);
                if (flags & FLAG_STOP) {
                    cact[t] = false;
                    if (tid == 0) {  // releases the producer, which waits for the trigger of step st + 1
                        sh.stop[t] = 1;
                        __threadfence_block();
                        mbar_arrive(&sh.trig[t][(st + 1) & 1]);
                    }
                    continue;
                }
                butterfly_store(part0);
                tick(3);
                if (USE_INT)  // the integrator warp takes it from here
                    asm volatile("bar.arrive %0, %1;" ::"r"(BAR_INT + t), "n"(32 * (NCW + 1)) : "memory");
                else
                    compute_bar();
                if (sh.abort) {  // an exchange wait timed out somewhere in this block
                    aborted = true;
                    break;
                }
                // (4) warp 0: a = sum of the j-parts; v += a*dt; q += v*dt (nbody.cc:77-88); publish the body as one
                //     tagged sector {x, y, z, step}, unfenced
                if (!USE_INT && warp == 0) {
                    if (lane == 0) mbar_arrive(&sh.trig[t][(st + 1) & 1]);  // producer trigger: everybody publishes within ~150 clk
                    if (integ) {
                        const double* p = &sh.part[t][stage][(ib >> 2) * NJ][3 * (ib & 3) + ik];
                        double a = p[0];
#pragma unroll
                        for (int j = 1; j < NJ; j++) a += p[j * 3 * BPW];  // fixed order: deterministic
                        if (my_body < n) kick_drift(a, iv, iq);
                    }
                    const double qy = __shfl_down_sync(0xffffffffu, iq, 1);
                    const double qz = __shfl_down_sync(0xffffffffu, iq, 2);
                    if (integ && ik == 0) st_sector(g_rec(t, st + 1) + 4 * (size_t)my_body, iq, qy, qz, make_tag(st + 1, iq, qy, qz));
                }
                cstep[t] = st + 1;
                tick(4);
            }
            any = false;
#pragma unroll
            for (int t = 0; t < T; t++) any |= cact[t];
        }
        if (aborted && tid == 0) {
#pragma unroll
            for (int t = 0; t < T; t++) sh.stop[t] = 1;
        }

        if (PROFILE) {
            if (tid == 0 && c == 0) {
                long long g1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
                for (int k = 0; k < 5; k++) prof[k] = pacc[k];
                prof[6] = pacc[5];
                prof[7] = (clock64() - c0) * 1000 / (g1 - g0 > 0 ? g1 - g0 : 1);  // SM MHz over the step loop
            }
        }
        if (PROFILE && n_stale) atomicAdd((unsigned long long*)&prof[5], n_stale);
        // write back (several systems: the integrator warp)
        if (!USE_INT && integ && my_body < n) {
            descs[0].q[ik * n + my_body] = iq;
            descs[0].v[ik * n + my_body] = iv;
        }
    }
    if (PROFILE && tid == 0) {  // globaltimer at the end of this block's work: prof[10] = min, prof[11] = max
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        atomicMin((unsigned long long*)&prof[10], g);
        atomicMax((unsigned long long*)&prof[11], g);
    }
    // nobody leaves while a cluster peer may still multicast into its shared memory
    __syncthreads();
    cluster_sync_all();
}

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

int blocks_for(int n) { return (n + GB - 1) / GB; }
int padded_blocks(int n, int cs) { return (blocks_for(n) + cs - 1) / cs * cs; }
size_t smem_for(int n, int T, int cs) {
    const size_t R = (size_t)padded_blocks(n, cs) * GB;
    return (size_t)T * 10 * ((R + RPAD - 1) / RPAD * RPAD) * sizeof(double);
}

struct WsLayout {
    size_t gbuf_bytes, total;
};
WsLayout ws_layout(int n, int T) {
    WsLayout w;
    const size_t R = (size_t)padded_blocks(n, MAX_CS) * GB;
    w.gbuf_bytes = 2 * (size_t)T * R * 4 * sizeof(double);  // [parity][T][R] sectors {x, y, z, step tag}
    w.total = w.gbuf_bytes + 64 + NPROF * sizeof(long long);
    return w;
}

template <int T>
int launch_t(int n, int cs, const TrajDesc* descs, const double* fst, void* ws, cudaStream_t stream) {
    const int C = padded_blocks(n, cs);
    const size_t smem = smem_for(n, T, cs);
    const WsLayout w = ws_layout(n, MAX_T);  // one layout for every T: the status word has a fixed place
    double* gbuf = (double*)ws;
    int* status = (int*)((char*)ws + w.gbuf_bytes);
    long long* prof = (long long*)((char*)ws + w.gbuf_bytes + 64);
    static const bool profile = env_int("NB_GRID_PROFILE", 0) != 0;
    // copy delay after the trigger (SM clocks): one system per launch waits for every copy, so it wants the shortest
    // delay that keeps the polling rare (measured on one box: 3.25 us/step at 600 clk, 3.17 at 700-800, 3.21 at 900, 3.31 at
    // 1100; on another box 750 gave 3.9 and 900 gave 3.2, so 900 it is); with two systems in lock step the copy of one hides
    // behind the pair loop of the other and a longer delay (fewer stale records, fewer polls) wins (measured: b1024
    // four-trajectory solve on one GPU 2.33 s at 900, 2.00 s at 2600)
    static const int delay_clk_env = T == 1 ? env_int("NB_GRID_DELAY", 900) : env_int("NB_GRID_DELAY2", 3000);
    static const int delay_single_env = env_int("NB_GRID_DELAY", 900);
    auto kern = profile ? grid_traj_kernel<T, true> : grid_traj_kernel<T, false>;
    NB_CUDA(cudaMemsetAsync(ws, 0, w.gbuf_bytes, stream));  // tag 0 = no step
    if (profile) NB_CUDA(cudaMemsetAsync(prof, 0, NPROF * sizeof(long long), stream));

    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    if (profile) {
        const unsigned long long big = ~0ULL;
        NB_CUDA(cudaMemcpyAsync(prof + 8, &big, 8, cudaMemcpyHostToDevice, stream));
        NB_CUDA(cudaMemcpyAsync(prof + 10, &big, 8, cudaMemcpyHostToDevice, stream));
        NB_CUDA(cudaEventCreate(&pe0));
        NB_CUDA(cudaEventCreate(&pe1));
        NB_CUDA(cudaEventRecord(pe0, stream));
    }
    int R = C * GB, delay_clk = delay_clk_env, delay_single = delay_single_env;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C), cfg.blockDim = dim3(NTHREADS), cfg.dynamicSmemBytes = smem, cfg.stream = stream;
    cudaLaunchAttribute attrs[2];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = cs, attrs[0].val.clusterDim.y = 1, attrs[0].val.clusterDim.z = 1;
    attrs[1].id = cudaLaunchAttributeCooperative;
    attrs[1].val.cooperative = 1;
    cfg.attrs = attrs, cfg.numAttrs = 2;
    {   // function attributes and the co-residency check: once per (device, kernel, shape) - the chain plan of
        // nb_solve launches this kernel every NB_SOLVE_CHUNK steps.  The dynamic shared-memory limit is an attribute of
        // the kernel FUNCTION (every call overwrites it), so it is only ever raised: a per-(device, kernel) running
        // maximum, else b1024 -> b512 -> b1024 in one process would launch 160 KB against a limit lowered to 80 KB.
        static std::mutex mu;
        static std::set<std::tuple<int, const void*, size_t, int, int>> checked;
        static std::map<std::pair<int, const void*>, size_t> smem_limit;
        int dev = 0;
        NB_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lk(mu);
        size_t& limit = smem_limit[std::make_pair(dev, (const void*)kern)];
        if (smem > limit) {
            NB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            limit = smem;
        }
        const auto key = std::make_tuple(dev, (const void*)kern, smem, cs, C);
        if (!checked.count(key)) {
            if (cs > 8) NB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
            int max_clusters = 0;
            NB_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));
            static const bool force_unsupported = env_int("NB_GRID_FORCE_UNSUPPORTED", 0) != 0;  // tests: the fallback path
            if (force_unsupported) max_clusters = 0;
            if (max_clusters < C / cs) {
                set_error_detail("grid trajectory kernel: " + std::to_string(C / cs) + " clusters of " + std::to_string(cs) +
                                 " blocks are not co-resident on this GPU (max " + std::to_string(max_clusters) + ")");
                return NB_ERR_UNSUPPORTED;  // nothing has been launched: the caller may try a smaller cluster or another kernel
            }
            checked.insert(key);
        }
    }
    const auto h0 = std::chrono::steady_clock::now();
    // NB_GRID_ADAPT="up,down" (clk): closed loop on the copy delay, default 128,8; "0,0" = the constant NB_GRID_DELAY.
    // Measured on B200, b1024, us per step (profiles/r02_grid_exchange.md): constant 900 -> 3.51, constant 400 -> 4.14;
    // adaptive 128,8 -> 3.47 from either start value (64,8: 3.49; 32,4: 3.53; 200,2: 3.59; 64,32: 3.71): the constant that
    // had to be tuned per box (round 1: "on another box 750 gave 3.9") is gone, the gain itself is 1 %.
    static int adapt_up = 128, adapt_down = 8;
    static const bool adapt_read = [] {
        const char* e = getenv("NB_GRID_ADAPT");
        if (e) sscanf(e, "%d,%d", &adapt_up, &adapt_down);
        return true;
    }();
    (void)adapt_read;
    // two systems in lock step: the copy of one system hides behind the other's step, so the delay is a constant in the
    // middle of that window (NB_GRID_DELAY2) - measured on B200, b1024 three-query solve on one GPU: adaptive (capped at
    // 1600 clk) 1.45 s with 36 000 stale records per step, constant 2600: 1.33 - 1.40 s, 3400: 1.32 s with 170, 5000: 1.39 s,
    // 7000: 1.78 s
    const int a_up = T == 1 ? adapt_up : 0;
    NB_CUDA(cudaLaunchKernelEx(&cfg, kern, descs, fst, gbuf, prof, status, R, delay_clk, delay_single, a_up, adapt_down));
    count_launch();
    {
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
        static const bool verbose = getenv("NB_VERBOSE") != nullptr;
        if (verbose && ms > 2.0) fprintf(stderr, "nbody_b200:   cudaLaunchKernelEx took %.1f ms on the host\n", ms);
    }
    // asynchronous: the caller synchronises the stream and then reads the sticky status word (grid_traj_status)
    if (profile) {
        NB_CUDA(cudaEventRecord(pe1, stream));
        NB_CUDA(cudaStreamSynchronize(stream));
        long long h[12];
        NB_CUDA(cudaMemcpy(h, prof, sizeof h, cudaMemcpyDeviceToHost));
        float kms = 0;
        NB_CUDA(cudaEventElapsedTime(&kms, pe0, pe1));
        cudaEventDestroy(pe0), cudaEventDestroy(pe1);
        fprintf(stderr, "grid kernel %.3f ms by events | block entry spread %.1f us | first entry -> last block done %.3f ms | block done spread %.1f us\n",
                kms, (h[9] - h[8]) * 1e-3, (h[11] - h[8]) * 1e-6, (h[11] - h[10]) * 1e-3);
        fprintf(stderr,
                "grid profile T=%d NJ=%d CS=%d delay=%d (clk, block 0 thread 0): wait copy %lld | validate %lld | pairs %lld | wait observer %lld | "
                "butterfly %lld | barrier+integrate+publish %lld | stale records polled (all blocks) %lld | SM clock %lld MHz\n",
                T, NJ, cs, delay_clk, h[0], h[6], h[1], h[2], h[3], h[4], h[5], h[7]);
    }
    return NB_OK;
}

// cluster size: NB_GRID_CS (1, 2, 4, 8), default 4; every cluster must be co-resident
int cluster_size_for(int n) {
    static const int want = env_int("NB_GRID_CS", 4);
    int cs = want;
    if (cs != 1 && cs != 2 && cs != 4 && cs != 8) cs = 4;
    while (cs > 1 && padded_blocks(n, cs) > 144) cs >>= 1;
    return cs;
}

}  // namespace

// the largest group of trajectories one launch takes for this n (shared-memory bound)
static int group_size(int n, int cs) {
    int T = MAX_T;
    while (T > 1 && smem_for(n, T, cs) > 200 * 1024) T--;
    static const int cap = env_int("NB_GRID_T", MAX_T);
    return T < cap ? T : (cap < 1 ? 1 : cap);
}

bool grid_traj_supported(int gpu, int n) {
    static const int enabled = env_int("NB_GRID", 1);
    static const int min_n = env_int("NB_GRID_MIN_N", 128);
    if (!enabled || n < min_n || n > NB_MAX_SMALL_N) return false;
    // three attributes, cached per device: this runs before every launch and cudaGetDeviceProperties costs 2-200 ms
    // a call on the B200 boxes (it was the whole "slow launch" of the chunked chain plan)
    struct Caps {
        int coop = -1, sms = 0, smem_optin = 0;
    };
    static std::mutex mu;
    static Caps caps[64];
    if (gpu < 0 || gpu >= 64) return false;
    Caps c;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (caps[gpu].coop < 0) {
            Caps q;
            if (cudaDeviceGetAttribute(&q.coop, cudaDevAttrCooperativeLaunch, gpu) != cudaSuccess ||
                cudaDeviceGetAttribute(&q.sms, cudaDevAttrMultiProcessorCount, gpu) != cudaSuccess ||
                cudaDeviceGetAttribute(&q.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, gpu) != cudaSuccess)
                return false;
            caps[gpu] = q;
        }
        c = caps[gpu];
    }
    if (!c.coop) return false;
    if (padded_blocks(n, cluster_size_for(n)) > c.sms) return false;
    if (smem_for(n, 1, cluster_size_for(n)) > (size_t)c.smem_optin) return false;
    return true;
}

void grid_traj_warm() {
    cudaFuncAttributes fa;
    (void)cudaFuncGetAttributes(&fa, grid_traj_kernel<1, false>);
    (void)cudaFuncGetAttributes(&fa, grid_traj_kernel<2, false>);  // two systems in lock step
}

// device address of the status word of a workspace: 0 = ok, 1 = an exchange spin timed out (read after the stream is idle)
const int* grid_traj_status(const void* ws, int n) { return (const int*)((const char*)ws + ws_layout(n, MAX_T).gbuf_bytes); }

size_t grid_traj_workspace_bytes(int n) { return ws_layout(n, MAX_T).total; }

int launch_grid_traj(int math, int n, int n_traj, const TrajDesc* descs, const double* fst, int gpu, void* ws,
                     size_t ws_bytes, cudaStream_t stream) {
    if (ws_bytes < ws_layout(n, MAX_T).total) return NB_ERR_ARG;
    // STRICT never comes here: its ascending-j sum is the single-block kernel's (nb_host.cu)
    if (math != NB_MATH_FAST) return NB_ERR_UNSUPPORTED;
    NB_CUDA(cudaMemsetAsync((char*)ws + ws_layout(n, MAX_T).gbuf_bytes, 0, 64, stream));  // status word, sticky over the groups
    // clusters that are not co-resident (MIG / MPS / a shared GPU): halve the cluster size; NB_ERR_UNSUPPORTED comes back
    // before anything has been launched, and with clusters of 1 it goes up to the caller, who has the single-block kernel
    for (int cs = cluster_size_for(n);; cs >>= 1) {
        const int G = group_size(n, cs);
        int rc = NB_OK;
        // Groups of up to G trajectories: two systems per launch run in lock step, one set of 8 compute warps steps both in
        // turn (the exchange of one system hides behind the other's step).  A warp set per system, each at its own pace, was
        // measured slower (b1024 three-query solve on one GPU 1.35 - 1.46 s against 1.27 s): one compute warp per scheduler
        // keeps the FP64 pipe only 33 % busy, two warps of the same system 76 % (profiles/r02_grid_exchange.md, section 5).
        for (int t0 = 0; t0 < n_traj && rc == NB_OK; t0 += G) {
            const int T = n_traj - t0 < G ? n_traj - t0 : G;
            rc = T == 1 ? launch_t<1>(n, cs, descs + t0, fst, ws, stream) : launch_t<2>(n, cs, descs + t0, fst, ws, stream);
            if (rc == NB_ERR_UNSUPPORTED && t0 > 0) return NB_ERR_CUDA;  // cannot happen: the first group decides
        }
        if (rc != NB_ERR_UNSUPPORTED || cs == 1) return rc;
    }
    return NB_OK;
}

}  // namespace nb
