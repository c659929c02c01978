// Shared declarations of the symmetric large-N stepper (nb_sym.cu = kernels + C ABI, nb_sym_plan.cc-free:
// the planner is plain host C++ inside nb_sym.cu so that it builds with the same toolchain).
#pragma once
#include <cstdint>
#include <vector>

namespace nb {
namespace sym {

// Measured on B200 at n = 65536 (profiles/r02_sym_accel.md, variants): 6 i-bodies per lane, 8 warps, ONE block per SM (254
// registers: the six pair chains of a rotation interleave instruction by instruction) 2.93 ms/step; 4 per lane at 128
// registers, 16 warps/SM (chains serialised by the register budget, 8-cycle dependent stalls) 3.28 ms; 12 warps x 168
// registers 3.12 ms.
constexpr int WARPS = 8;       // warps per block
constexpr int MIN_BLOCKS = 1;  // resident blocks per SM the register budget is set for
// i-bodies per lane: two instantiations of the kernel.  6 (rows of up to 1536 bodies) is the faster loop; 8 (2048) wastes no
// register slots when the shard is a power of two (8192 bodies per rank at 8 ranks = 4 rows of 2048, against 6 rows of
// 1366 in 1536 slots).  choose_ipl() takes the one with the smaller slots x cost product.
constexpr int IPL_A = 6, IPL_B = 8;
constexpr int sb_of(int ipl) { return WARPS * 32 * ipl; }  // bodies per row (superblock) = i-bodies per block
constexpr int MAX_SB = sb_of(IPL_B);
constexpr int TJ = 128;                  // j bodies per shared-memory tile (64 / 256: 3.01 / 2.96 ms per step against 2.93)
constexpr int STAGES = 3;                // TMA ring depth
constexpr int SUB = 32;                  // scheduling granularity along j (one warp rotation group)
constexpr int MAX_PEERS = 16;

constexpr int SEG_ONESIDED = 1;  // j range = the row's own bodies: ordered pairs, only a_i accumulated
constexpr int SEG_LOAD = 2;      // first segment of a row run in this block: load the i bodies, zero a_i
constexpr int SEG_FLUSH = 4;     // last segment of a row run: write a_i to PI[pi_slot]

// One unit of a block's work list: the block's row (SB consecutive bodies of the local shard, I_PER_LANE per lane)
// against the j bodies [j0, j1).  Symmetric segments (the default) evaluate every unordered pair {i, j} once and
// accumulate both a_i (registers, flushed to PI) and a_j (rotating registers -> shared memory -> PJ of the
// owner of j); they never contain a body of the row itself.
struct Seg {
    int row_body0;  // global index of the row's first body
    int row_count;  // bodies in the row (<= SB)
    int j0, j1;     // global body range, j0 a multiple of SUB relative to the owner's shard start
    int flags;      // SEG_*
    int pi_slot;    // SEG_FLUSH: slot of the PI buffer
    int pj_row;     // symmetric: row index in the owner's PJ buffer (= global row number)
    int src_rank;   // rank that owns (and publishes) bodies [j0, j1)
};

// Host-side plan of one rank.
struct Plan {
    int n = 0, world = 1, rank = 0, blocks = 0;
    int shard = 0;       // bodies per rank (n / world)
    int ipl = IPL_A, sb = sb_of(IPL_A);  // i-bodies per lane of the kernel instantiation, register slots per row
    int rows_local = 0;  // rows of this rank's shard
    int row_stride = 0;  // bodies per row (the last one may be shorter): the shard spread evenly over the fewest rows, <= SB
    int rows_global = 0; // rows of all ranks (world * rows_local)
    std::vector<Seg> segs;
    std::vector<int> block_seg_begin;  // [blocks + 1]
    int pi_slots = 0;
    // integrate tables, per local row r: PI slots pi_list[pi_ptr[r] .. pi_ptr[r+1]) and PJ rows
    // pj_list[pj_ptr[r] .. pj_ptr[r+1]) (global row numbers, ascending) that hold contributions to its bodies
    std::vector<int> pi_ptr, pi_list, pj_ptr, pj_list;
    long long sym_pairs = 0, onesided_pairs = 0;  // unordered pairs evaluated symmetrically / ordered pairs one-sided
};

// Builds the plan of `rank`.  n % world == 0.  Pure host code (no CUDA): tests call it through nb_sym_plan_describe.
int build_plan(int n, int world, int rank, int blocks, int ipl, Plan& out);
int choose_ipl(int n, int world);

}  // namespace sym
}  // namespace nb
