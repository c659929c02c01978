/*
 * nbody_b200 — C ABI of the B200 (sm_100a) N-body hot path.
 *
 * Drop-in boundary for the one hot path of dasbd72/NTHU_IPC_Nbody-Simulation: the all-pairs FP64
 * softened-gravity step with sin-modulated gravity-device masses + explicit v/q update, iterated
 * 200 000 times, and the three queries built on it.  Every entry point names the reference
 * interface it replaces (file:line into the reference tree).
 *
 * Conventions (SURVEY.md §8b):
 *   - extern "C", POD structs, plain pointers and sizes; no exceptions cross the boundary;
 *   - every function returns NB_OK (0) or a negative NB_ERR_* code; nb_strerror() explains it and
 *     nb_last_error_detail() holds the CUDA error text of the calling thread's last failure;
 *   - host arrays are owned by the caller; device memory is owned by the library behind opaque
 *     handles; one handle = one GPU = one stream; handles may be used from different host threads
 *     concurrently (no global mutable state besides per-GPU lazily built constant tables);
 *   - planar layout of hw5.cu:93-97: q[3*n] = x block, y block, z block (same for v);
 *   - there is NO CPU fallback: without a usable GPU every compute call returns NB_ERR_NO_GPU.
 */
#ifndef NBODY_B200_H
#define NBODY_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define NB_OK 0
#define NB_ERR_ARG (-1)         /* bad argument (null pointer, n <= 0, index out of range, ...) */
#define NB_ERR_CUDA (-2)        /* a CUDA runtime call or kernel failed; see nb_last_error_detail() */
#define NB_ERR_NO_GPU (-3)      /* no CUDA device / requested ordinal does not exist              */
#define NB_ERR_UNSUPPORTED (-4) /* size or mode outside what this build supports                  */
#define NB_ERR_IO (-5)          /* file could not be read / written / parsed                      */

/* arithmetic of the pair term (nbody.cc:65-72) */
#define NB_MATH_FAST 0   /* FMA r^2, rsqrt seed + cubic correction (<= 2^-52 rel.), FMA accumulate, j split over lanes */
#define NB_SOLVE_ALL_DEVICES 0x100 /* OR into `math` of nb_solve / nb_solve_partial: simulate every device's query-3 trajectory from step 0 (diagnostics for all devices) instead of stopping at the cheapest saviour */
#define NB_MATH_STRICT 1 /* IEEE only: sqrt(r2*r2*r2), ((G*mj)*d)/dist3, no FMA, ascending j (== hw5.cu:200-203 form of nbody.cc) */

/* trajectory kinds = the observers that run after every step */
#define NB_KIND_PLAIN 0 /* min distance only, never stops early                               */
#define NB_KIND_Q1 1    /* nbody.cc:106-122: devices massless, min planet-asteroid distance    */
#define NB_KIND_Q2 2    /* nbody.cc:124-138 + hw5.cu:265-287: first hit step, missile reach steps; stops at the hit */
#define NB_KIND_Q3 3    /* hw5.cu:289-309: hit test, then missile destroys `destroy_device`; stops at the hit */

#define NB_MAX_DEVICES 64
#define NB_MAX_SMALL_N 1024 /* largest system the persistent (shared-memory resident) kernels take */

/* physics constants of nbody.cc:9-20 (read-only; exported for callers that need them) */
#define NB_N_STEPS 200000
#define NB_DT 60.0
#define NB_EPS 1e-3
#define NB_G 6.674e-11
#define NB_PLANET_RADIUS 1e7
#define NB_MISSILE_SPEED 1e6

typedef struct nb_system {
    int n;                          /* bodies                                        */
    int planet;                     /* index of the planet   (input header, nbody.cc:27) */
    int asteroid;                   /* index of the asteroid                         */
    const double* q;                /* [3*n] planar positions                        */
    const double* v;                /* [3*n] planar velocities                       */
    const double* m;                /* [n] base masses                               */
    const unsigned char* is_device; /* [n] 1 where type == "device" (nbody.cc:62)    */
} nb_system;

typedef struct nb_events {
    double min_d2;      /* min over observed steps of d^2(planet, asteroid) (hw5.cu:241-252)          */
    int argmin_step;    /* first step attaining it                                                    */
    int hit_step;       /* first step with d^2 < planet_radius^2 (nbody.cc:134), else -2              */
    int destroyed_step; /* Q3: step at which the missile reached the device (hw5.cu:299-307), else -2 */
    double cost;        /* Q3: 1e5 + 1e3*((destroyed_step+1)*dt) (hw5.cu:305), else +inf              */
    int steps_done;     /* step the state is at (== hit step when stopped early); -1 = not yet observed */
    int n_reach;        /* number of devices                                                          */
    int reach_step[NB_MAX_DEVICES]; /* Q2: first step with d^2(planet, device k) < (1e6*60*step)^2, else -2 (hw5.cu:265-287) */
} nb_events;

typedef struct nb_answer {
    double min_dist;       /* output line 1 (nbody.cc:44-48) */
    int hit_time_step;     /* output line 2; -2 = no hit     */
    int gravity_device_id; /* output line 3; -1 = none       */
    double missile_cost;   /* output line 3; 0 when none     */
    /* diagnostics */
    int argmin_step;
    int n_devices;
    int device_index[NB_MAX_DEVICES];
    int reach_step[NB_MAX_DEVICES];
    int q3_hit_step[NB_MAX_DEVICES]; /* -2 = planet saved, -3 = not simulated, else hit step */
    double q3_cost[NB_MAX_DEVICES];
    double gpu_seconds;   /* max over GPUs of the device time spent in trajectory kernels */
    double wall_seconds;  /* host wall time inside nb_solve, context creation included   */
    long long pair_interactions; /* ordered pair interactions evaluated                  */
    int n_trajectories;
    int n_gpus_used;
} nb_answer;

/* ---- library / device ------------------------------------------------------------------- */
const char* nb_version(void);
const char* nb_strerror(int code);
const char* nb_last_error_detail(void); /* thread-local text of the last NB_ERR_CUDA */
int nb_device_count(int* count);        /* NB_ERR_NO_GPU when there is none          */
/* launches of this library's kernels made by the calling process so far (for bench accounting) */
long long nb_kernel_launches(void);
/* Records of the grid kernel's fence-free exchange that passed the step check but failed the full self-check (a torn
 * 32-byte sector) and were fetched again, in this process so far.  Expected: 0 (the hardware reads and writes whole
 * sectors); a non-zero count is harmless for the results and worth reporting. */
long long nb_grid_torn_records(void);

/* ---- the step operator -------------------------------------------------------------------
 * Replaces run_step(step, n, qx,qy,qz, vx,vy,vz, m, type) (nbody.cc:51-89) and the kernel pair
 * compute_accelerations_gpu + update_positions_gpu (hw5.cu:159-215, 231-239): advances the
 * caller's HOST arrays q, v in place by the steps step_begin+1 .. step_end (run_step's `step`
 * argument takes each of those values).  Any n >= 1.  `m` are base masses; device modulation
 * (nbody.cc:14-16) is applied inside.
 */
int nb_run_steps(int gpu, int math, int n, double* q, double* v, const double* m,
                 const unsigned char* is_device, int step_begin, int step_end);

/* ---- trajectories (query drivers' inner loops) --------------------------------------------
 * Replaces the host-driven loops of t_problem_12 / t_problem_3 (hw5.cu:322-436, 438-530): one
 * persistent kernel runs every step and every observer on the GPU.  n <= NB_MAX_SMALL_N.
 */
typedef struct nb_traj nb_traj;
int nb_traj_create(int gpu, const nb_system* sys, int kind, int destroy_device, int math, nb_traj** out);
/* run from the current step up to and including step_end, or until the kind's stop event */
int nb_traj_run(nb_traj* t, int step_end, nb_events* ev);
/* current state (any pointer may be NULL); m = base masses as the trajectory now sees them */
int nb_traj_state(nb_traj* t, double* q, double* v, double* m, int* step);
/* fork: a new trajectory of `kind` starting from t's current state (hw5.cu:275-284 snapshot, :482-483 restore) */
int nb_traj_fork(nb_traj* t, int kind, int destroy_device, nb_traj** out);
/* the same onto another GPU: q, v travel device to device (peer copy), never through the host */
int nb_traj_fork_on(nb_traj* t, int gpu, int kind, int destroy_device, nb_traj** out);
int nb_traj_destroy(nb_traj* t);

/* ---- ensembles ------------------------------------------------------------------------------
 * n_systems independent systems of the same n in one launch, one thread block per system
 * (north-star (c): batches of synthetic systems).  Arrays are system-major: q[s][3*n] ...
 * planet/asteroid/destroy_device are per system.  q, v are updated in place; ev[s] filled.
 */
int nb_ensemble_run(int gpu, int math, int kind, int n_systems, int n, double* q, double* v,
                    const double* m, const unsigned char* is_device, const int* planet,
                    const int* asteroid, const int* destroy_device, int step_begin, int step_end,
                    nb_events* ev, double* gpu_seconds);

/* ---- the three queries ----------------------------------------------------------------------
 * Replaces main() of hw5.cu:532-616 minus file I/O: Q1, Q2 and one Q3 trajectory per device,
 * scheduled over the given GPUs with no collective (hw5.cu:566-567, 587-588 hard-code two).
 * gpus == NULL means ordinals 0..n_gpus-1.  Any n >= 1 (at most NB_MAX_DEVICES gravity devices): n <= NB_MAX_SMALL_N
 * runs on the persistent kernels, larger systems on the large-N steppers with an observer kernel after every step.
 */
int nb_solve(const nb_system* sys, const int* gpus, int n_gpus, int n_steps, int math, nb_answer* ans);
/* The same, split for one-process-per-GPU launches (torchrun): trajectory t (0 = Q1, 1 = Q2,
 * 2+k = Q3 with device k destroyed) belongs to part t % n_parts.  nb_solve_partial runs this
 * part's trajectories on `gpu` and fills evs[t] for them (evs has nb_solve_trajectory_count()
 * entries); after the parts' entries have been gathered, nb_solve_combine applies the selection
 * rule of hw5.cu:509-517, 568-602.  Any n, as nb_solve. */
int nb_solve_trajectory_count(const nb_system* sys, int* count);
int nb_solve_partial(const nb_system* sys, int gpu, int part, int n_parts, int n_steps, int math,
                     nb_events* evs, double* gpu_seconds, long long* pair_interactions);
int nb_solve_combine(const nb_system* sys, const nb_events* evs, nb_answer* ans);

/* ---- file formats (nbody.cc:22-49, hw5.cu:86-141) ------------------------------------------- */
int nb_read_header(const char* path, int* n, int* planet, int* asteroid);
int nb_read_input(const char* path, int max_n, int* n, int* planet, int* asteroid, double* q,
                  double* v, double* m, unsigned char* is_device);
int nb_write_output(const char* path, double min_dist, int hit_time_step, int gravity_device_id,
                    double missile_cost);
/* The input format, written (17 significant digits): generated / advanced systems can go through hw5, nbtool and
 * the reference's samples/nbody.cc alike.  SURVEY.md 8f rank 4. */
int nb_write_input(const char* path, int n, int planet, int asteroid, const double* q, const double* v,
                   const double* m, const unsigned char* is_device);
/* Synthetic system of SURVEY.md 8d config C5 (std::mt19937_64(seed)): body 0 = planet, 1 = asteroid, the last
 * n_devices bodies are gravity devices.  q, v: [3n] planar; m, is_device: [n]. */
int nb_generate_system(int n, unsigned long long seed, int n_devices, double* q, double* v, double* m,
                       unsigned char* is_device, int* planet, int* asteroid);
/* the whole CLI: hw5 <input> <output> (hw5.cu:532-616).  The GPUs (n_gpus, or NB_HW5_GPUS, default 1) are started on
 * helper threads while the input is parsed (hw5.cu:555-567 starts its two GPUs from parallel host threads). */
int nb_hw5_main(const char* input_path, const char* output_path, int n_gpus);
/* process start-up helpers: nb_device_warm = driver initialisation + context + constant tables + kernel module of one
 * GPU (thread-safe; call it early, from a helper thread); nb_hw5_narrow_visible_gpus sets CUDA_VISIBLE_DEVICES to the
 * first `want` GPUs unless the user set it - it changes the PROCESS environment, so only the `hw5` binary's main()
 * calls it, before the first CUDA call, never the library itself.  Returns the number of /dev/nvidiaN nodes, or -1. */
int nb_device_warm(int gpu);
int nb_hw5_narrow_visible_gpus(int want);

/* ---- large systems, body-sharded (north-star (d)) -------------------------------------------
 * DEVICE-pointer interface: the caller (C++ or torch) owns the buffers and the stream, so that a
 * per-step position all-gather (NCCL) can run between calls on the same stream.
 *   pos4     [n][4] doubles  {x, y, z, G*m_eff(step)} of ALL bodies at the current step
 *   pos4_out [n][4] doubles  rows i_begin..i_begin+i_count-1 are written with the state after the
 *                            step and G*m_eff(step+1); other rows untouched (peers fill them)
 *   vel      [3][i_count]    planar velocities of the local bodies, updated in place
 *   m0       [n] base masses, is_device [n]
 *   scratch  nb_large_scratch_bytes() bytes
 */
long long nb_large_scratch_bytes(int n, int i_count);
int nb_large_pack(int math, int n, const double* q_planar_dev, const double* m0_dev,
                  const unsigned char* is_device_dev, int step_next, double* pos4_dev, void* stream);
int nb_large_unpack(int n, const double* pos4_dev, double* q_planar_dev, void* stream);
int nb_large_step(int math, int step, int n, int i_begin, int i_count, const double* pos4_dev,
                  double* pos4_out_dev, double* vel_dev, const double* m0_dev,
                  const unsigned char* is_device_dev, void* scratch_dev, void* stream);

/* The same step with the exchange fused in (north star (d), "P2P stores overlapped with the local tile"):
 * the integrate kernel stores every new pos4 row straight into EVERY rank's pos4_out buffer through
 * peer-mapped pointers (NVLink P2P; entry `rank` is the own buffer); each of its
 * nb_large_blocks_per_step(i_count) blocks then adds 1, with a system-scope release, to counter
 * [step & 1][rank] of every rank (a rank's counter block is nb_large_p2p_counter_bytes() bytes, zeroed).
 * The NEXT step's acceleration kernel waits inside the kernel: blocks whose j range is local start at once
 * (the grid is rotated so that they run first), the others wait until the counter of exactly the source
 * rank they read reaches wait_target = blocks * (steps of that parity executed so far); 0 = no wait
 * (first step).  peer_* are HOST arrays of device pointers (own allocations or nb_ipc_open results);
 * n must be divisible by world and this rank's shard is [rank*n/world, (rank+1)*n/world).
 * nb_large_wait_p2p is the stand-alone wait on all sources (before the host reads the final buffer). */
int nb_large_step_p2p(int math, int step, int n, int i_begin, int i_count, const double* pos4_dev,
                      double* const* peer_pos4_out, unsigned long long* const* peer_counters, int world,
                      int rank, unsigned long long wait_target, int* status_dev, double* vel_dev,
                      const double* m0_dev, const unsigned char* is_device_dev, void* scratch_dev,
                      void* stream);
int nb_large_blocks_per_step(int i_count);
int nb_large_p2p_counter_bytes(void);
int nb_large_wait_p2p(const unsigned long long* my_counters, int parity, int world,
                      unsigned long long target, int* status_dev, void* stream);
/* raw device memory (zero-filled cudaMalloc on the current device) and CUDA IPC handles (64 bytes), so that
 * one process per GPU can map its peers' exchange buffers */
int nb_dev_alloc(long long bytes, void** dev_ptr);
int nb_dev_free(void* dev_ptr);
int nb_dev_copy(void* dst, const void* src, long long bytes, int kind /*0 H2D, 1 D2H, 2 D2D*/, void* stream);
int nb_ipc_export(void* dev_ptr, unsigned char* handle64);
int nb_ipc_open(const unsigned char* handle64, void** dev_ptr);
int nb_ipc_close(void* dev_ptr);

/* ---- large systems, symmetric stepper (FAST math) ---------------------------------------------------
 * The same step as nb_large_step_p2p (run_step, nbody.cc:51-89; replaces hw5.cu:159-215 + 231-239) with every
 * UNORDERED pair evaluated once: both a_i and a_j are accumulated, 10 FP64 instructions per ordered pair.
 * Rank r of `world` holds shard [r*n/world, (r+1)*n/world) and evaluates the block pairs (r, r) .. (r, r + world/2);
 * the partial accelerations of a body are stored straight into the memory of the rank that owns it (PJ, a
 * peer-mapped buffer of nb_sym_pj_bytes() bytes per rank, ZERO-FILLED once: rows nobody writes are summed as zeros)
 * and its integrate kernel sums them in a fixed order,
 * integrates and stores the new pos4 record into EVERY rank's next-step buffer.  Arrival is signalled through
 * per-rank counter blocks (nb_sym_counter_bytes() bytes, zeroed, peer-mapped) with system-scope release/acquire;
 * the kernels wait on them in-kernel, so a step is two launches and no host synchronisation or NCCL call.
 * world == 1: the peer arrays have one entry (own buffers), counters / status may be NULL.
 * Steps must be consecutive (the counters count them).  pos4 layout as above: [n][4] doubles. */
typedef struct nb_sym nb_sym;
int nb_sym_create(int n, int world, int rank, nb_sym** out); /* on the current CUDA device */
int nb_sym_destroy(nb_sym* h);
long long nb_sym_pj_bytes(const nb_sym* h);
int nb_sym_counter_bytes(void);
int nb_sym_blocks(const nb_sym* h);
long long nb_sym_remote_partial_bytes(const nb_sym* h); /* bytes of partial rows this rank stores into peers per step */
/* ordered pair interactions one step of this rank covers (= 2 x symmetric + one-sided) */
long long nb_sym_pairs(const nb_sym* h, long long* sym_pairs, long long* onesided_pairs);
/* stream-ordered wait until every rank's rows of the last step are in this rank's buffer (before the host reads it) */
int nb_sym_wait_positions(nb_sym* h, const unsigned long long* my_counters, int* status_dev, void* stream);
int nb_sym_step(nb_sym* h, int step, const double* pos4_cur_dev, double* const* peer_pos4_next,
                double* const* peer_pj, unsigned long long* const* peer_counters, int* status_dev,
                double* vel_dev, const double* m0_dev, const unsigned char* is_device_dev, void* stream);
/* One step in two calls: phases = 1 launches the acceleration kernel, 2 the integrate kernel, 3 both (= nb_sym_step).
 * With every rank's phase 1 enqueued before any rank's phase 2, several ranks can share ONE GPU and one stream (each
 * in-kernel wait is then already satisfied when it is reached): the multi-rank path is testable on a 1-GPU box. */
int nb_sym_step_phase(nb_sym* h, int step, int phases, const double* pos4_cur_dev, double* const* peer_pos4_next,
                      double* const* peer_pj, unsigned long long* const* peer_counters, int* status_dev,
                      double* vel_dev, const double* m0_dev, const unsigned char* is_device_dev, void* stream);
/* run_step with HOST buffers, sharded (bench "e2e"): nb_sym_publish_rows turns this rank's positions (planar
 * [3][n/world] doubles on the device, just copied from the host) into pos4 records {x, y, z, G*m_eff(step_next)} in EVERY
 * rank's current buffer, signalled like the integrate kernel's stores (every rank must call it before the same step);
 * nb_sym_unpack_rows extracts this rank's rows of a pos4 buffer back into planar form for the copy to the host. */
int nb_sym_publish_rows(nb_sym* h, int step_next, const double* q_own_planar_dev, double* const* peer_pos4_cur,
                        unsigned long long* const* peer_counters, const double* m0_dev,
                        const unsigned char* is_device_dev, void* stream);
int nb_sym_unpack_rows(nb_sym* h, const double* pos4_dev, double* q_own_planar_dev, void* stream);
/* the whole host-buffer step in one call: q_own_host / v_own_host are (pinned) planar [3][n/world] host arrays with this
 * rank's state, in/out; q_own_stage_dev is a device scratch of the same size; peer_pos4_cur / peer_pos4_next are the
 * buffers the step reads / writes.  Returns when the new state is in the host arrays. */
int nb_sym_step_host(nb_sym* h, int step, double* q_own_host, double* v_own_host, double* q_own_stage_dev,
                     const double* pos4_cur_dev, double* const* peer_pos4_cur, double* const* peer_pos4_next,
                     double* const* peer_pj, unsigned long long* const* peer_counters, int* status_dev,
                     double* vel_dev, const double* m0_dev, const unsigned char* is_device_dev, void* stream);
/* The static schedule of one rank (host only, no GPU needed): segments of eight ints
 * {row_body0, row_count, j0, j1, flags, pi_slot, pj_row, src_rank} (flags: 1 = one-sided, 2 = load row, 4 = flush row),
 * block b owns segments [block_seg_begin[b], block_seg_begin[b+1]); pj_ptr / pj_list = per local row the PJ rows
 * that hold contributions to its bodies.  Any output pointer may be NULL. */
int nb_sym_plan_describe(int n, int world, int rank, int blocks, int max_segs, int* segs_out, int* n_segs,
                         int* block_seg_begin, int* pj_ptr, int* pj_list, int max_pj, long long* sym_pairs,
                         long long* onesided_pairs);
int nb_sym_row_size(void);         /* largest row (= i-bodies per thread block) of this build */
int nb_sym_rows(int n, int world); /* rows per rank */
int nb_sym_row_stride(int n, int world); /* bodies per row: the shard spread evenly over the fewest rows */

/* ---- measurement helpers ----------------------------------------------------------------------- */
/* long independent DFMA chains on every SM: measured FP64 peak of this GPU in TFLOP/s */
int nb_fp64_peak(int gpu, double* tflops, double* seconds);
/* the same with register-operand DFMAs: variant 1 = three distinct register pairs per DFMA,
 * variant 2 = one multiplicand shared by consecutive DFMAs (operand-reuse pattern) */
int nb_fp64_peak_variant(int gpu, int variant, double* tflops);
/* When enabled, nb_large_step brackets its acceleration kernel with CUDA events on the caller's
 * stream (calling thread only) and accumulates the durations; nb_profile_read synchronises and
 * returns the total milliseconds and the number of launches since the last enable. */
int nb_profile_enable(int on);
int nb_profile_read(double* accel_ms, long long* accel_launches);

#ifdef __cplusplus
}
#endif
#endif
