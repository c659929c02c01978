// Symmetric large-N step (FAST math): every UNORDERED pair {i, j} is evaluated once and feeds both a_i and a_j,
// so an ordered pair interaction costs 10 FP64-pipe instructions instead of 16 (nb_large.cu) or the reference's
// 29 + 3 atomics (hw5.cu:159-215).  Arithmetic: nbody.cc:56-88; every ordered pair of run_step still contributes.
//
//   * A block owns a ROW of SB = 1536 consecutive bodies, 6 per lane, in registers {x, y, z, G*m, ax, ay, az}.
//   * j bodies stream through shared memory in tiles of TJ records (1-D TMA bulk copies, mbarrier ring).  A warp
//     takes 32 of them, one per lane, and ROTATES them through its lanes with warp shuffles: after 32 rotations
//     every lane has met every j body, and the j body has collected its own acceleration {ajx, ajy, ajz} in
//     registers that travel with it.  No shared-memory traffic and no FP64 work besides the pair terms.
//   * The eight warps' a_j of a tile meet in shared memory and leave as one coalesced partial row PJ[row][3][j]
//     in the memory of the rank that OWNS body j (a peer-mapped pointer: the reduce-scatter of the accelerations is
//     these stores); a_i leaves once per row run as PI[slot][3][SB].  sym_integrate_kernel sums the partials of a
//     body in a fixed order (deterministic, no atomics), integrates and publishes the new pos4 record to every rank.
//   * The work (upper triangle of the row x j-group matrix) is cut into equal-cost pieces on the host
//     (build_plan): a static schedule, one piece per resident block, granularity 1536 x 32 pairs.
//   * Multi-GPU: rank p holds shard p and evaluates the block pairs (p, p), (p, p+1) .. (p, p+P/2) (the last one
//     split in half for even P), local work first, so that the peers' positions arrive behind it.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "nb_async.cuh"
#include "nb_internal.h"
#include "nb_math.cuh"
#include "nb_sym.cuh"

namespace nb {
namespace sym {

// ================================================================================================ planner (host)
namespace {
struct Span {
    int i0, icount;  // the row: local bodies [i0, i0 + icount) of the rank (at most SB; aligned rows start at a multiple of SB)
    int j0, j1;      // global j range
    bool onesided;
    int src;         // rank that owns [j0, j1)
};

// The bodies of a shard are spread EVENLY over the fewest rows that hold them: a row always occupies all SB register slots
// of its block (a short row leaves lanes idle but takes as long per j body), so rows of equal length keep the cost of a
// (row, j) unit uniform.  stride = bodies per row.
int stride_of(int shard, int sb) {
    const int rows = (shard + sb - 1) / sb;
    return (shard + rows - 1) / rows;
}
int rows_of(int shard, int sb) { return (shard + stride_of(shard, sb) - 1) / stride_of(shard, sb); }

// the spans of rank p, phase by phase (phase 0 = local, phase 1 = remote)
void spans_of_rank(int n, int world, int p, int sb, std::vector<std::vector<Span>>& phases) {
    const int S = n / world, R = rows_of(S, sb), base = p * S, RS = stride_of(S, sb);
    auto cnt = [&](int r) { return std::min(S, (r + 1) * RS) - r * RS; };
    phases.assign(2, {});
    for (int r = 0; r < R; r++) {
        const int r1 = std::min(S, (r + 1) * RS);
        if (r1 < S) phases[0].push_back({r * RS, cnt(r), base + r1, base + S, false, p});  // the rows behind it, symmetric
        phases[0].push_back({r * RS, cnt(r), base + r * RS, base + r1, true, p});           // its own bodies, one-sided
    }
    if (world == 1) return;
    const int full = (world - 1) / 2;  // partners evaluated entirely by this rank
    for (int k = 1; k <= full; k++) {
        const int q = (p + k) % world;
        for (int r = 0; r < R; r++) phases[1].push_back({r * RS, cnt(r), q * S, q * S + S, false, q});
    }
    if (world % 2 == 0) {
        // The block pair (lo, hi = lo + P/2) is shared half and half IN TIME (a row costs the same per j body whatever its
        // length): hi takes its rows behind rb against all of lo, lo takes all its rows against the bodies of hi's rows
        // before rb; with an odd number of rows, hi's row rb is split down the middle of lo: hi takes it against lo's
        // rows from cr on, lo takes its rows before cr against it.  Every cut lies on a row boundary of the owner of the
        // a_j partials, so a PJ row is written entirely or not at all for each row of its owner.
        const int q = (p + world / 2) % world;
        const int rb = R / 2, cr = (R % 2) ? (R + 1) / 2 : 0;
        const int hb = std::min(S, rb * RS), hb1 = std::min(S, (rb + 1) * RS), cb = std::min(S, cr * RS);
        if (p < q) {  // this rank is lo
            if (hb > 0)
                for (int r = 0; r < R; r++) phases[1].push_back({r * RS, cnt(r), q * S, q * S + hb, false, q});
            for (int r = 0; r < cr; r++) phases[1].push_back({r * RS, cnt(r), q * S + hb, q * S + hb1, false, q});
        } else {      // this rank is hi
            if (R % 2) phases[1].push_back({rb * RS, cnt(rb), q * S + cb, q * S + S, false, q});
            for (int r = rb + (R % 2); r < R; r++) phases[1].push_back({r * RS, cnt(r), q * S, q * S + S, false, q});
        }
    }
}
}  // namespace

// i-bodies per lane for this shard size: fewest register slots x relative cost of the loop (measured, n = 65536: 2.93 ms
// with 6 per lane, 3.00 ms with 8)
int choose_ipl(int n, int world) {
    if (n < 1 || world < 1 || n % world) return IPL_A;
    const int S = n / world;
    const double ca = (double)rows_of(S, sb_of(IPL_A)) * sb_of(IPL_A) * 1.0, cb = (double)rows_of(S, sb_of(IPL_B)) * sb_of(IPL_B) * 1.025;
    return cb < ca ? IPL_B : IPL_A;
}

int build_plan(int n, int world, int rank, int blocks, int ipl, Plan& P) {
    if (n < 1 || world < 1 || world > MAX_PEERS || rank < 0 || rank >= world || n % world != 0 || blocks < 1) return NB_ERR_ARG;
    if (ipl != IPL_A && ipl != IPL_B) return NB_ERR_ARG;
    P = Plan{};
    P.ipl = ipl, P.sb = sb_of(ipl);
    const int SB = P.sb;
    P.n = n, P.world = world, P.rank = rank, P.blocks = blocks;
    P.shard = n / world;
    P.rows_local = rows_of(P.shard, SB);
    P.row_stride = stride_of(P.shard, SB);
    P.rows_global = world * P.rows_local;
    const int S = P.shard, base = rank * S;
    std::vector<std::vector<Span>> phases;
    spans_of_rank(n, world, rank, SB, phases);
    std::vector<std::vector<Seg>> per_block(blocks);
    std::vector<double> got(blocks, 0.0);  // cost given to each block so far
    double ideal_before = 0;               // what an exact split of the earlier phases would have given it
    for (const auto& spans : phases) {
        // cost of one SUB-wide unit of a span: a row occupies all SB register slots of the block however many bodies it
        // has, so the time per j body is the same for every row (one-sided: 16 instr per ordered pair, no rotation,
        // against 20 per unordered pair)
        auto unit_cost = [&](const Span& s) { return SB * (s.onesided ? 0.8 : 1.0) + 0.0 * s.icount; };
        double total = 0;
        for (const auto& s : spans) total += unit_cost(s) * ((s.j1 - s.j0 + SUB - 1) / SUB);
        if (total <= 0) continue;
        // block k's share of this phase = an equal part, corrected by what the rounding of the earlier phases gave it
        // too much or too little; bound[k] = end of its window in cumulative cost
        std::vector<double> bound(blocks);
        {
            double acc = 0;
            for (int b = 0; b < blocks; b++) {
                acc += std::max(0.0, total / blocks + (ideal_before - got[b]));
                bound[b] = acc;
            }
            for (int b = 0; b < blocks; b++) bound[b] *= total / acc;  // the corrections sum to ~0; keep the windows exact
        }
        double cum = 0;
        int k = 0;
        for (const auto& s : spans) {
            const int units = (s.j1 - s.j0 + SUB - 1) / SUB;
            const double w = unit_cost(s);
            int u0 = 0;
            while (u0 < units) {
                int take;
                if (k >= blocks - 1) {
                    k = blocks - 1;
                    take = units - u0;
                } else {
                    const double room = bound[k] - cum;
                    take = (int)(room / w + 0.5);
                    if (take > units - u0) take = units - u0;
                    if (take <= 0) {
                        k++;
                        continue;
                    }
                }
                Seg g{};
                g.row_body0 = base + s.i0;
                g.row_count = s.icount;
                g.j0 = s.j0 + u0 * SUB;
                g.j1 = std::min(s.j1, s.j0 + (u0 + take) * SUB);
                g.flags = s.onesided ? SEG_ONESIDED : 0;
                g.pi_slot = -1;
                g.pj_row = rank * P.rows_local + s.i0 / P.row_stride;  // a virtual row takes the number of the aligned row around it
                g.src_rank = s.src;
                per_block[k].push_back(g);
                if (s.onesided)
                    P.onesided_pairs += (long long)g.row_count * (g.j1 - g.j0);
                else
                    P.sym_pairs += (long long)g.row_count * (g.j1 - g.j0);
                cum += take * w;
                got[k] += take * w;
                u0 += take;
                if (k < blocks - 1 && cum >= bound[k] - 0.5 * w) k++;
            }
        }
        ideal_before += total / blocks;
    }
    // merge adjacent pieces of one span, mark row runs, number the PI slots row by row
    struct Flush {
        int row, block, idx;
    };
    std::vector<Flush> flushes;
    auto same_row = [](const Seg& a, const Seg& b) { return a.row_body0 == b.row_body0 && a.row_count == b.row_count; };
    for (int b = 0; b < blocks; b++) {
        auto& v = per_block[b];
        std::vector<Seg> m;
        for (const Seg& g : v) {
            if (!m.empty() && same_row(m.back(), g) && m.back().flags == g.flags && m.back().j1 == g.j0 && m.back().src_rank == g.src_rank)
                m.back().j1 = g.j1;
            else
                m.push_back(g);
        }
        v.swap(m);
        for (size_t i = 0; i < v.size(); i++) {
            if (i == 0 || !same_row(v[i - 1], v[i])) v[i].flags |= SEG_LOAD;
            if (i + 1 == v.size() || !same_row(v[i + 1], v[i])) {
                v[i].flags |= SEG_FLUSH;
                flushes.push_back({(v[i].row_body0 - base) / P.row_stride, b, (int)i});
            }
        }
    }
    std::stable_sort(flushes.begin(), flushes.end(), [](const Flush& a, const Flush& b) { return a.row < b.row; });
    P.pi_ptr.assign(P.rows_local + 1, 0);
    for (size_t s = 0; s < flushes.size(); s++) {
        Seg& g = per_block[flushes[s].block][flushes[s].idx];
        g.pi_slot = (int)s;
        P.pi_ptr[flushes[s].row + 1]++;
        // per slot: {slot, first local body, bodies}: a virtual row covers only part of the aligned row it lies in
        P.pi_list.push_back((int)s);
        P.pi_list.push_back(g.row_body0 - base);
        P.pi_list.push_back(g.row_count);
    }
    for (int r = 0; r < P.rows_local; r++) P.pi_ptr[r + 1] += P.pi_ptr[r];
    P.pi_slots = (int)flushes.size();
    P.block_seg_begin.assign(blocks + 1, 0);
    for (int b = 0; b < blocks; b++) {
        P.block_seg_begin[b + 1] = P.block_seg_begin[b] + (int)per_block[b].size();
        P.segs.insert(P.segs.end(), per_block[b].begin(), per_block[b].end());
    }
    // which PJ rows hold contributions to the bodies of local row c: every rank's symmetric spans that touch it (the
    // part of such a PJ row that nobody writes stays zero)
    std::vector<std::vector<int>> contrib(P.rows_local);
    for (int p = 0; p < world; p++) {
        std::vector<std::vector<Span>> ph;
        spans_of_rank(n, world, p, SB, ph);
        for (const auto& spans : ph)
            for (const auto& s : spans) {
                if (s.onesided || s.src != rank) continue;
                for (int c = 0; c < P.rows_local; c++) {
                    const int c0 = base + c * P.row_stride, c1 = base + std::min(S, (c + 1) * P.row_stride);
                    if (s.j0 < c1 && s.j1 > c0) contrib[c].push_back(p * P.rows_local + s.i0 / P.row_stride);
                }
            }
    }
    P.pj_ptr.assign(P.rows_local + 1, 0);
    for (int c = 0; c < P.rows_local; c++) {
        std::sort(contrib[c].begin(), contrib[c].end());
        contrib[c].erase(std::unique(contrib[c].begin(), contrib[c].end()), contrib[c].end());
        P.pj_ptr[c + 1] = P.pj_ptr[c] + (int)contrib[c].size();
        P.pj_list.insert(P.pj_list.end(), contrib[c].begin(), contrib[c].end());
    }
    return NB_OK;
}

// ================================================================================================ kernels
namespace {

constexpr int NT = 32 * WARPS;  // threads per block
constexpr int ROT_UNROLL = 2;  // unrolled 1 / 4: 2.99 / 2.95 ms per step against 2.93 (profiles/r02_sym_accel.md)
constexpr int TILE_BYTES = TJ * 32;
constexpr int STG_DOUBLES = WARPS * 3 * TJ;  // one staging buffer
constexpr size_t SMEM_BYTES = (size_t)STAGES * TILE_BYTES + 2 * (size_t)STG_DOUBLES * sizeof(double);
// counter block of a rank (unsigned long long): [kind: 0 = pos4 rows arrived, 1 = partial accelerations arrived][parity][source rank]
constexpr int CTR_WORDS = 2 * 2 * MAX_PEERS;

struct Peers {
    double* pj[MAX_PEERS];                    // PJ of every rank: [rows_global][3][shard]
    double4* pos4_next[MAX_PEERS];            // next-step pos4 of every rank: [n]
    unsigned long long* counters[MAX_PEERS];  // counter block of every rank
    int world, my_rank;
};

struct AccelArgs {
    const double4* pos4;  // all bodies, current step
    const Seg* segs;
    const int* block_seg_begin;
    double* pi;  // [pi_slots][3][SB]
    int shard;
    int parity_read;                  // parity of the step whose rows are being read (their arrival counters)
    unsigned long long pos_target;    // 0 = nothing to wait for
    int parity_acc;                   // parity of this step (partial-arrival counters)
    int* status;
};

__device__ __forceinline__ double rot(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

template <int I_PER_LANE>
__global__ void __launch_bounds__(NT, MIN_BLOCKS) sym_accel_kernel(AccelArgs A, Peers peers) {
    constexpr int WARP_I = 32 * I_PER_LANE, SB = WARPS * WARP_I;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double4* tile = reinterpret_cast<double4*>(smem_raw);                         // [STAGES][TJ]
    double* stg = reinterpret_cast<double*>(smem_raw + STAGES * TILE_BYTES);      // [2][WARPS][3][TJ]
    __shared__ alignas(8) uint64_t full[STAGES];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sb = A.block_seg_begin[blockIdx.x], se = A.block_seg_begin[blockIdx.x + 1];
    const Seg* segs = A.segs;

    // ---- producer (thread 0): walks the block's tiles ahead of the consumers
    int p_si = sb, p_j = sb < se ? segs[sb].j0 : 0, p_t = 0;
    unsigned seen = 1u << peers.my_rank;
    auto issue = [&]() {  // next tile into stage p_t % STAGES; false when the list is exhausted
        while (p_si < se && p_j >= segs[p_si].j1) {
            p_si++;
            if (p_si < se) p_j = segs[p_si].j0;
        }
        if (p_si >= se) return false;
        const int src = segs[p_si].src_rank;
        if (A.pos_target && !(seen >> src & 1u)) {
            // rows of another rank: valid once every block of its integrate kernel has stored them here and released
            wait_counter(peers.counters[peers.my_rank] + (0 * 2 + A.parity_read) * MAX_PEERS + src, A.pos_target, A.status, 1);
            asm volatile("fence.proxy.async;" ::: "memory");  // the TMA (async proxy) reads what was just acquired
            seen |= 1u << src;
        }
        const int cnt = min(TJ, segs[p_si].j1 - p_j);
        const int st = p_t % STAGES;
        mbar_expect_tx(&full[st], (uint32_t)cnt * 32u);
        tma_load_1d(tile + st * TJ, A.pos4 + p_j, (uint32_t)cnt * 32u, &full[st]);
        p_j += cnt;
        p_t++;
        return true;
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; s++) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0)
        for (int s = 0; s < STAGES; s++)
            if (!issue()) break;

    // ---- consumers
    double xi[I_PER_LANE], yi[I_PER_LANE], zi[I_PER_LANE], gi[I_PER_LANE];
    double ax[I_PER_LANE], ay[I_PER_LANE], az[I_PER_LANE];
#pragma unroll
    for (int k = 0; k < I_PER_LANE; k++) xi[k] = yi[k] = zi[k] = gi[k] = ax[k] = ay[k] = az[k] = 0.0;
    const int src_lane = (lane + 1) & 31;
    int t = 0;
    for (int si = sb; si < se; si++) {
        const Seg sg = segs[si];
        if (sg.flags & SEG_LOAD) {
#pragma unroll
            for (int k = 0; k < I_PER_LANE; k++) {
                const int off = warp * WARP_I + k * 32 + lane;
                const double4 p = A.pos4[sg.row_body0 + min(off, sg.row_count - 1)];
                xi[k] = p.x, yi[k] = p.y, zi[k] = p.z;
                gi[k] = off < sg.row_count ? p.w : 0.0;  // a padding lane must not pull on anybody
                ax[k] = ay[k] = az[k] = 0.0;
            }
        }
        for (int jb = sg.j0; jb < sg.j1; jb += TJ, t++) {
            const int cnt = min(TJ, sg.j1 - jb);
            const int st = t % STAGES;
            mbar_wait(&full[st], (t / STAGES) & 1);
            const double4* tj = tile + st * TJ;
            if (sg.flags & SEG_ONESIDED) {
                // the row against itself: ordered pairs, every lane reads the same j record (broadcast); the self term is
                // exactly zero (d = 0, eps > 0)
#pragma unroll 2
                for (int j = 0; j < cnt; j++) {
                    const double4 b = tj[j];
                    double c[I_PER_LANE], dx[I_PER_LANE], dy[I_PER_LANE], dz[I_PER_LANE];
#pragma unroll
                    for (int k = 0; k < I_PER_LANE; k++) pair_coeff_fast(xi[k], yi[k], zi[k], b.x, b.y, b.z, b.w, c[k], dx[k], dy[k], dz[k]);
#pragma unroll
                    for (int k = 0; k < I_PER_LANE; k++) pair_accum_fast(c[k], dx[k], dy[k], dz[k], ax[k], ay[k], az[k]);
                }
            } else {
                double* my_stg = stg + (t & 1) * STG_DOUBLES + warp * 3 * TJ;
                for (int s0 = 0; s0 < cnt; s0 += 32) {
                    const int jl = s0 + lane;
                    const double4 b = tj[min(jl, cnt - 1)];
                    double jx = b.x, jy = b.y, jz = b.z, jg = jl < cnt ? b.w : 0.0;
                    double ajx = 0.0, ajy = 0.0, ajz = 0.0;
#pragma unroll ROT_UNROLL
                    for (int r = 0; r < 32; r++) {
                        // The j body moves on to the next lane with what it has collected; after 32 moves it is home
                        // again.  Its position does not depend on this rotation's arithmetic: fetch it first.
                        const double nx = rot(jx, src_lane), ny = rot(jy, src_lane), nz = rot(jz, src_lane), ng = rot(jg, src_lane);
#pragma unroll
                        for (int k = 0; k < I_PER_LANE; k++)
                            pair_sym(xi[k], yi[k], zi[k], gi[k], jx, jy, jz, jg, ax[k], ay[k], az[k], ajx, ajy, ajz);
                        ajx = rot(ajx, src_lane), ajy = rot(ajy, src_lane), ajz = rot(ajz, src_lane);
                        jx = nx, jy = ny, jz = nz, jg = ng;
                    }
                    if (jl < cnt) my_stg[jl] = ajx, my_stg[TJ + jl] = ajy, my_stg[2 * TJ + jl] = ajz;
                }
            }
            __syncthreads();  // everyone is done with stage st (refill it) and the tile's a_j are staged
            if (tid == 0) issue();
            if (!(sg.flags & SEG_ONESIDED)) {
                // the eight warps' a_j -> one partial row in the memory of the rank that owns these bodies
                const double* sbuf = stg + (t & 1) * STG_DOUBLES;
                double* dst = peers.pj[sg.src_rank] + (size_t)sg.pj_row * 3 * A.shard + (jb - sg.src_rank * A.shard);
                for (int idx = tid; idx < 3 * TJ; idx += NT) {
                    const int c = idx / TJ, jl = idx - c * TJ;
                    if (jl < cnt) {
                        double s = sbuf[c * TJ + jl];
#pragma unroll
                        for (int w = 1; w < WARPS; w++) s += sbuf[(w * 3 + c) * TJ + jl];
                        dst[(size_t)c * A.shard + jl] = s;
                    }
                }
            }
        }
        if (sg.flags & SEG_FLUSH) {
            double* out = A.pi + (size_t)sg.pi_slot * 3 * SB;
#pragma unroll
            for (int k = 0; k < I_PER_LANE; k++) {
                const int off = warp * WARP_I + k * 32 + lane;
                out[off] = ax[k], out[SB + off] = ay[k], out[2 * SB + off] = az[k];
            }
        }
    }
    if (peers.world > 1) {
        // this block's partial rows are in their owners' memory: tell every rank (system-scope release)
        __threadfence_system();
        __syncthreads();
        if (tid < peers.world) red_release_sys(peers.counters[tid] + (1 * 2 + A.parity_acc) * MAX_PEERS + peers.my_rank);
    }
}

struct IntegrateArgs {
    const double4* pos4;  // current step, all bodies
    double* vel;          // [3][shard]
    const double* m0;
    const unsigned char* is_device;
    const double* pi;
    const double* pj;  // own PJ
    const int *pi_ptr, *pi_list, *pj_ptr, *pj_list;
    int shard, i_begin, row_stride, sb;
    double fst_next;
    int parity;                     // of this step: partial counters waited on, position counters raised
    unsigned long long acc_target;  // 0 = nothing to wait for (one rank)
    int* status;
};

// a = sum of the partials in a fixed order; v += a*dt; q += v*dt (nbody.cc:77-88); new pos4 record to every rank.
// A block takes IB consecutive bodies; the partial rows of a body (PI slots of its row, then the PJ rows the plan lists:
// up to ~80 at 8 ranks) are dealt round-robin to IP threads, which sum their share in ascending order; the IP shares
// meet in shared memory and are added in part order - deterministic, and IP times the memory parallelism of one thread
// per body.
constexpr int IB = 32, IP = 8;
__global__ void __launch_bounds__(IB * IP) sym_integrate_kernel(IntegrateArgs A, Peers peers) {
    __shared__ double part[IP][3][IB];
    if (A.acc_target) {
        if (threadIdx.x < peers.world)
            wait_counter(peers.counters[peers.my_rank] + (1 * 2 + A.parity) * MAX_PEERS + threadIdx.x, A.acc_target, A.status, 2);
        __syncthreads();
    }
    const int bx = threadIdx.x % IB, pt = threadIdx.x / IB;
    const int il = blockIdx.x * IB + bx;
    double a[3] = {0.0, 0.0, 0.0};
    if (il < A.shard) {
        const int row = il / A.row_stride;
        const int p0 = A.pi_ptr[row], npi = A.pi_ptr[row + 1] - p0, j0 = A.pj_ptr[row], npj = A.pj_ptr[row + 1] - j0;
#pragma unroll 2
        for (int k = pt; k < npi + npj; k += IP) {
            if (k < npi) {
                // {slot, first local body, bodies} of a row run that covers (part of) this row
                const int s = p0 + k, idx = il - A.pi_list[3 * s + 1];
                if (idx >= 0 && idx < A.pi_list[3 * s + 2]) {
                    const double* p = A.pi + (size_t)A.pi_list[3 * s] * 3 * A.sb + idx;
                    a[0] += p[0], a[1] += p[A.sb], a[2] += p[2 * A.sb];
                }
            } else {
                const double* p = A.pj + (size_t)A.pj_list[j0 + k - npi] * 3 * A.shard + il;
                a[0] += p[0], a[1] += p[A.shard], a[2] += p[2 * (size_t)A.shard];
            }
        }
    }
    part[pt][0][bx] = a[0], part[pt][1][bx] = a[1], part[pt][2][bx] = a[2];
    __syncthreads();
    if (pt == 0 && il < A.shard) {
#pragma unroll
        for (int c = 0; c < 3; c++) {
            double t = part[0][c][bx];
#pragma unroll
            for (int q = 1; q < IP; q++) t += part[q][c][bx];
            a[c] = t;
        }
        const int i = A.i_begin + il;
        const double4 p = A.pos4[i];
        double x = p.x, y = p.y, z = p.z;
        double vx = A.vel[il], vy = A.vel[il + A.shard], vz = A.vel[il + 2 * A.shard];
        kick_drift(a[0], vx, x);
        kick_drift(a[1], vy, y);
        kick_drift(a[2], vz, z);
        A.vel[il] = vx, A.vel[il + A.shard] = vy, A.vel[il + 2 * A.shard] = vz;
        const double4 rec = make_double4(x, y, z, gm_eff(A.m0[i], A.is_device[i] != 0, A.fst_next));
        for (int pr = 0; pr < peers.world; pr++) peers.pos4_next[pr][i] = rec;
    }
    if (peers.world > 1) {
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x < peers.world)
            red_release_sys(peers.counters[threadIdx.x] + (0 * 2 + A.parity) * MAX_PEERS + peers.my_rank);
    }
}

// run_step with HOST buffers (bench e2e): the caller's positions of this rank's bodies (planar, just copied host ->
// device) become pos4 records in EVERY rank's current buffer, signalled like the integrate kernel's stores
__global__ void __launch_bounds__(128) sym_publish_kernel(const double* __restrict__ q_own, const double* __restrict__ m0,
                                                          const unsigned char* __restrict__ is_device, int shard, int i_begin,
                                                          double fst, int parity, Peers peers) {
    const int il = blockIdx.x * blockDim.x + threadIdx.x;
    if (il < shard) {
        const int i = i_begin + il;
        const double4 rec = make_double4(q_own[il], q_own[il + shard], q_own[il + 2 * shard], gm_eff(m0[i], is_device[i] != 0, fst));
        for (int pr = 0; pr < peers.world; pr++) peers.pos4_next[pr][i] = rec;
    }
    if (peers.world > 1) {
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x < peers.world)
            red_release_sys(peers.counters[threadIdx.x] + (0 * 2 + parity) * MAX_PEERS + peers.my_rank);
    }
}

__global__ void sym_unpack_rows_kernel(const double4* __restrict__ pos4, int shard, int i_begin, double* __restrict__ q_own) {
    const int il = blockIdx.x * blockDim.x + threadIdx.x;
    if (il >= shard) return;
    const double4 p = pos4[i_begin + il];
    q_own[il] = p.x, q_own[il + shard] = p.y, q_own[il + 2 * shard] = p.z;
}

}  // namespace
}  // namespace sym
}  // namespace nb

using namespace nb;
using namespace nb::sym;

struct nb_sym {
    Plan plan;
    int gpu = -1, integrate_blocks = 0;
    Seg* d_segs = nullptr;
    int *d_bsb = nullptr, *d_tables = nullptr;  // tables: pi_ptr | pi_list | pj_ptr | pj_list
    int off_pi_list = 0, off_pj_ptr = 0, off_pj_list = 0;
    double* d_pi = nullptr;
    long long steps_done[2] = {0, 0};  // steps executed per parity
    long long pos_pubs[2] = {0, 0};    // publications of this rank's rows per parity (integrate kernels + nb_sym_publish_rows)
    int first_step = -1, last_step = -1, accel_step = -1;
};

// One rank has no arrival counters: the step bookkeeping only enforces consecutive steps, and a restart may forget it.
// With world > 1 the counters of every rank count the steps, so there is no restart.
int nb::sym_restart(nb_sym* h) {
    if (!h || h->plan.world != 1) return NB_ERR_ARG;
    h->steps_done[0] = h->steps_done[1] = 0;
    h->pos_pubs[0] = h->pos_pubs[1] = 0;
    h->first_step = h->last_step = h->accel_step = -1;
    return NB_OK;
}

static int sym_default_blocks(int* out) {
    static std::mutex mu;
    static std::map<int, int> cache;
    int dev = 0;
    NB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(dev);
    if (it == cache.end()) {
        int sms = 0, per_sm = 0;
        NB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        int per_sm_b = 0;
        NB_CUDA(cudaFuncSetAttribute(sym_accel_kernel<IPL_A>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        NB_CUDA(cudaFuncSetAttribute(sym_accel_kernel<IPL_B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        NB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sym_accel_kernel<IPL_A>, NT, SMEM_BYTES));
        NB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_b, sym_accel_kernel<IPL_B>, NT, SMEM_BYTES));
        if (per_sm_b < per_sm) per_sm = per_sm_b;
        if (per_sm < 1) {
            set_error_detail("symmetric kernel does not fit on this GPU");
            return NB_ERR_UNSUPPORTED;
        }
        it = cache.emplace(dev, sms * per_sm).first;
    }
    *out = it->second;
    return NB_OK;
}

extern "C" {

int nb_sym_plan_describe(int n, int world, int rank, int blocks, int max_segs, int* segs_out, int* n_segs,
                         int* block_seg_begin, int* pj_ptr, int* pj_list, int max_pj, long long* sym_pairs,
                         long long* onesided_pairs) {
    Plan P;
    int rc = build_plan(n, world, rank, blocks, choose_ipl(n, world), P);
    if (rc) return rc;
    if (n_segs) *n_segs = (int)P.segs.size();
    if (sym_pairs) *sym_pairs = P.sym_pairs;
    if (onesided_pairs) *onesided_pairs = P.onesided_pairs;
    if (segs_out) {
        if ((int)P.segs.size() > max_segs) return NB_ERR_ARG;
        static_assert(sizeof(Seg) == 8 * sizeof(int), "Seg is eight ints");
        memcpy(segs_out, P.segs.data(), P.segs.size() * sizeof(Seg));
    }
    if (block_seg_begin) memcpy(block_seg_begin, P.block_seg_begin.data(), (blocks + 1) * sizeof(int));
    if (pj_ptr) memcpy(pj_ptr, P.pj_ptr.data(), (P.rows_local + 1) * sizeof(int));
    if (pj_list) {
        if ((int)P.pj_list.size() > max_pj) return NB_ERR_ARG;
        memcpy(pj_list, P.pj_list.data(), P.pj_list.size() * sizeof(int));
    }
    return NB_OK;
}

int nb_sym_row_size(void) { return MAX_SB; }
int nb_sym_rows(int n, int world) { return (n < 1 || world < 1 || n % world) ? 0 : rows_of(n / world, sb_of(choose_ipl(n, world))); }
int nb_sym_row_stride(int n, int world) {
    return (n < 1 || world < 1 || n % world) ? 0 : stride_of(n / world, sb_of(choose_ipl(n, world)));
}

int nb_sym_create(int n, int world, int rank, nb_sym** out) {
    if (!out || n < 1 || world < 1 || world > MAX_PEERS || rank < 0 || rank >= world || n % world != 0) return NB_ERR_ARG;
    int blocks = 0;
    int rc = sym_default_blocks(&blocks);
    if (rc) return rc;
    nb_sym* h = new nb_sym();
    rc = build_plan(n, world, rank, blocks, choose_ipl(n, world), h->plan);
    if (rc) {
        delete h;
        return rc;
    }
    const Plan& P = h->plan;
    cudaGetDevice(&h->gpu);
    h->integrate_blocks = (P.shard + IB - 1) / IB;
    std::vector<int> tables;
    tables.insert(tables.end(), P.pi_ptr.begin(), P.pi_ptr.end());
    h->off_pi_list = (int)tables.size();
    tables.insert(tables.end(), P.pi_list.begin(), P.pi_list.end());
    h->off_pj_ptr = (int)tables.size();
    tables.insert(tables.end(), P.pj_ptr.begin(), P.pj_ptr.end());
    h->off_pj_list = (int)tables.size();
    tables.insert(tables.end(), P.pj_list.begin(), P.pj_list.end());
    tables.push_back(0);
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t x) {
        if (e == cudaSuccess) e = x;
    };
    ok(cudaMalloc(&h->d_segs, std::max<size_t>(1, P.segs.size()) * sizeof(Seg)));
    ok(cudaMalloc(&h->d_bsb, (blocks + 1) * sizeof(int)));
    ok(cudaMalloc(&h->d_tables, tables.size() * sizeof(int)));
    ok(cudaMalloc(&h->d_pi, std::max<size_t>(1, (size_t)P.pi_slots) * 3 * P.sb * sizeof(double)));
    if (e == cudaSuccess && !P.segs.empty())
        ok(cudaMemcpy(h->d_segs, P.segs.data(), P.segs.size() * sizeof(Seg), cudaMemcpyHostToDevice));
    if (e == cudaSuccess) ok(cudaMemcpy(h->d_bsb, P.block_seg_begin.data(), (blocks + 1) * sizeof(int), cudaMemcpyHostToDevice));
    if (e == cudaSuccess) ok(cudaMemcpy(h->d_tables, tables.data(), tables.size() * sizeof(int), cudaMemcpyHostToDevice));
    if (e != cudaSuccess) {
        rc = cuda_fail(e, "nb_sym_create", __FILE__, __LINE__);
        nb_sym_destroy(h);
        return rc;
    }
    *out = h;
    return NB_OK;
}

int nb_sym_destroy(nb_sym* h) {
    if (!h) return NB_ERR_ARG;
    cudaFree(h->d_segs), cudaFree(h->d_bsb), cudaFree(h->d_tables), cudaFree(h->d_pi);
    delete h;
    return NB_OK;
}

long long nb_sym_pj_bytes(const nb_sym* h) {
    return h ? (long long)h->plan.rows_global * 3 * h->plan.shard * (long long)sizeof(double) : 0;
}
int nb_sym_counter_bytes(void) { return CTR_WORDS * (int)sizeof(unsigned long long); }
int nb_sym_blocks(const nb_sym* h) { return h ? h->plan.blocks : 0; }

long long nb_sym_remote_partial_bytes(const nb_sym* h) {
    if (!h) return 0;
    long long b = 0;
    for (const Seg& g : h->plan.segs)
        if (!(g.flags & SEG_ONESIDED) && g.src_rank != h->plan.rank) b += (long long)(g.j1 - g.j0) * 3 * sizeof(double);
    return b;
}

long long nb_sym_pairs(const nb_sym* h, long long* sym_pairs, long long* onesided_pairs) {
    if (!h) return 0;
    if (sym_pairs) *sym_pairs = h->plan.sym_pairs;
    if (onesided_pairs) *onesided_pairs = h->plan.onesided_pairs;
    return 2 * h->plan.sym_pairs + h->plan.onesided_pairs;
}

int nb_sym_wait_positions(nb_sym* h, const unsigned long long* my_counters, int* status_dev, void* stream) {
    if (!h || !my_counters || !status_dev) return NB_ERR_ARG;
    if (h->plan.world == 1 || h->last_step < 0) return NB_OK;
    // in stream order, until every rank's rows of the last step have arrived (before the host reads the buffer)
    const int par = h->last_step & 1;
    return launch_counter_wait(my_counters + (0 * 2 + par) * MAX_PEERS, h->plan.world,
                               (unsigned long long)h->integrate_blocks * h->pos_pubs[par], status_dev, 3, (cudaStream_t)stream);
}

int nb_sym_step_phase(nb_sym* h, int step, int phases, const double* pos4_cur, double* const* peer_pos4_next,
                      double* const* peer_pj, unsigned long long* const* peer_counters, int* status_dev, double* vel_dev,
                      const double* m0_dev, const unsigned char* is_device_dev, void* stream) {
    if (!h || step < 1 || phases < 1 || phases > 3 || !pos4_cur || !peer_pos4_next || !peer_pj || !vel_dev || !m0_dev || !is_device_dev) return NB_ERR_ARG;
    const Plan& P = h->plan;
    if (P.world > 1 && (!peer_counters || !status_dev)) return NB_ERR_ARG;
    // the arrival counters count consecutive steps; phase 1 (acceleration) of a step comes before its phase 2 (integrate)
    const bool accel_done = h->accel_step == step;
    if (h->last_step >= 0 && step != h->last_step + 1) return NB_ERR_ARG;
    if ((phases & 1) && accel_done) return NB_ERR_ARG;
    if ((phases & 2) && !(phases & 1) && !accel_done) return NB_ERR_ARG;
    Peers peers{};
    peers.world = P.world, peers.my_rank = P.rank;
    for (int p = 0; p < P.world; p++) {
        if (!peer_pos4_next[p] || !peer_pj[p] || (P.world > 1 && !peer_counters[p])) return NB_ERR_ARG;
        peers.pj[p] = peer_pj[p];
        peers.pos4_next[p] = (double4*)peer_pos4_next[p];
        peers.counters[p] = P.world > 1 ? peer_counters[p] : nullptr;
    }
    cudaStream_t st = (cudaStream_t)stream;
    AccelArgs A{};
    A.pos4 = (const double4*)pos4_cur;
    A.segs = h->d_segs, A.block_seg_begin = h->d_bsb, A.pi = h->d_pi, A.shard = P.shard;
    A.parity_read = (step - 1) & 1;
    // rows of step-1 were published by the integrate kernels of step-1 (none before the first step: packed locally)
    A.pos_target = P.world > 1 ? (unsigned long long)h->integrate_blocks * h->pos_pubs[(step - 1) & 1] : 0;
    A.parity_acc = step & 1;
    A.status = status_dev;
    if (phases & 1) {
        cudaEvent_t pe0 = nullptr, pe1 = nullptr;
        const bool prof = profile_on();
        if (prof) {
            NB_CUDA(cudaEventCreate(&pe0));
            NB_CUDA(cudaEventCreate(&pe1));
            NB_CUDA(cudaEventRecord(pe0, st));
        }
        if (P.ipl == IPL_B)
            sym_accel_kernel<IPL_B><<<P.blocks, NT, SMEM_BYTES, st>>>(A, peers);
        else
            sym_accel_kernel<IPL_A><<<P.blocks, NT, SMEM_BYTES, st>>>(A, peers);
        count_launch();
        NB_CUDA(cudaGetLastError());
        if (prof) {
            NB_CUDA(cudaEventRecord(pe1, st));
            profile_push(pe0, pe1);
        }
        h->accel_step = step;
    }
    if (!(phases & 2)) return NB_OK;
    IntegrateArgs I{};
    I.pos4 = (const double4*)pos4_cur, I.vel = vel_dev, I.m0 = m0_dev, I.is_device = is_device_dev;
    I.pi = h->d_pi, I.pj = peer_pj[P.rank];
    I.pi_ptr = h->d_tables, I.pi_list = h->d_tables + h->off_pi_list;
    I.pj_ptr = h->d_tables + h->off_pj_ptr, I.pj_list = h->d_tables + h->off_pj_list;
    I.shard = P.shard, I.i_begin = P.rank * P.shard, I.row_stride = P.row_stride, I.sb = P.sb;
    I.fst_next = fst_value(step + 1);
    I.parity = step & 1;
    I.acc_target = P.world > 1 ? (unsigned long long)P.blocks * (h->steps_done[step & 1] + 1) : 0;
    I.status = status_dev;
    sym_integrate_kernel<<<h->integrate_blocks, IB * IP, 0, st>>>(I, peers);
    count_launch();
    NB_CUDA(cudaGetLastError());
    h->steps_done[step & 1]++;
    h->pos_pubs[step & 1]++;
    if (h->first_step < 0) h->first_step = step;
    h->last_step = step;
    return NB_OK;
}

int nb_sym_publish_rows(nb_sym* h, int step_next, const double* q_own_planar_dev, double* const* peer_pos4_cur,
                        unsigned long long* const* peer_counters, const double* m0_dev, const unsigned char* is_device_dev,
                        void* stream) {
    if (!h || step_next < 1 || !q_own_planar_dev || !peer_pos4_cur || !m0_dev || !is_device_dev) return NB_ERR_ARG;
    const Plan& P = h->plan;
    if (P.world > 1 && !peer_counters) return NB_ERR_ARG;
    if (h->last_step >= 0 && step_next != h->last_step + 1) return NB_ERR_ARG;
    Peers peers{};
    peers.world = P.world, peers.my_rank = P.rank;
    for (int p = 0; p < P.world; p++) {
        if (!peer_pos4_cur[p] || (P.world > 1 && !peer_counters[p])) return NB_ERR_ARG;
        peers.pos4_next[p] = (double4*)peer_pos4_cur[p];  // "next" = the buffer the coming step reads
        peers.counters[p] = P.world > 1 ? peer_counters[p] : nullptr;
    }
    const int par = (step_next - 1) & 1;  // the parity the coming step's acceleration kernel waits on
    sym_publish_kernel<<<h->integrate_blocks, IB, 0, (cudaStream_t)stream>>>(q_own_planar_dev, m0_dev, is_device_dev, P.shard,
                                                                            P.rank * P.shard, fst_value(step_next), par, peers);
    count_launch();
    NB_CUDA(cudaGetLastError());
    h->pos_pubs[par]++;
    return NB_OK;
}

int nb_sym_unpack_rows(nb_sym* h, const double* pos4_dev, double* q_own_planar_dev, void* stream) {
    if (!h || !pos4_dev || !q_own_planar_dev) return NB_ERR_ARG;
    const Plan& P = h->plan;
    sym_unpack_rows_kernel<<<(P.shard + 255) / 256, 256, 0, (cudaStream_t)stream>>>((const double4*)pos4_dev, P.shard,
                                                                                  P.rank * P.shard, q_own_planar_dev);
    count_launch();
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

// run_step with HOST buffers in one call (bench e2e, nbody.cc:51-54 signature, sharded): this rank's positions and
// velocities (pinned host memory, planar [3][n/world]) go host -> device, are published to every rank, the step's two
// kernels run, the new rows are extracted and copied device -> host; returns when they are there.
int nb_sym_step_host(nb_sym* h, int step, double* q_own_host, double* v_own_host, double* q_own_stage_dev,
                     const double* pos4_cur, double* const* peer_pos4_cur, double* const* peer_pos4_next,
                     double* const* peer_pj, unsigned long long* const* peer_counters, int* status_dev, double* vel_dev,
                     const double* m0_dev, const unsigned char* is_device_dev, void* stream) {
    if (!h || !q_own_host || !v_own_host || !q_own_stage_dev || !peer_pos4_cur || !peer_pos4_next) return NB_ERR_ARG;
    const size_t bytes = 3 * (size_t)h->plan.shard * sizeof(double);
    cudaStream_t st = (cudaStream_t)stream;
    NB_CUDA(cudaMemcpyAsync(q_own_stage_dev, q_own_host, bytes, cudaMemcpyHostToDevice, st));
    NB_CUDA(cudaMemcpyAsync(vel_dev, v_own_host, bytes, cudaMemcpyHostToDevice, st));
    int rc = nb_sym_publish_rows(h, step, q_own_stage_dev, peer_pos4_cur, peer_counters, m0_dev, is_device_dev, stream);
    if (rc) return rc;
    rc = nb_sym_step_phase(h, step, 3, pos4_cur, peer_pos4_next, peer_pj, peer_counters, status_dev, vel_dev, m0_dev, is_device_dev,
                           stream);
    if (rc) return rc;
    // the rank's own rows of the next buffer were written by its own integrate kernel: stream order suffices
    rc = nb_sym_unpack_rows(h, peer_pos4_next[h->plan.rank], q_own_stage_dev, stream);
    if (rc) return rc;
    NB_CUDA(cudaMemcpyAsync(q_own_host, q_own_stage_dev, bytes, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaMemcpyAsync(v_own_host, vel_dev, bytes, cudaMemcpyDeviceToHost, st));
    NB_CUDA(cudaStreamSynchronize(st));
    return NB_OK;
}

int nb_sym_step(nb_sym* h, int step, const double* pos4_cur, double* const* peer_pos4_next, double* const* peer_pj,
                unsigned long long* const* peer_counters, int* status_dev, double* vel_dev, const double* m0_dev,
                const unsigned char* is_device_dev, void* stream) {
    return nb_sym_step_phase(h, step, 3, pos4_cur, peer_pos4_next, peer_pj, peer_counters, status_dev, vel_dev, m0_dev,
                             is_device_dev, stream);
}

}  // extern "C"
