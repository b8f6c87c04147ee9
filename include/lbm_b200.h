/*
 * lbm_b200.h -- C ABI of liblbm_b200.so, the B200 (sm_100a) D2Q9 BGK collide-stream engine.
 *
 * This is the drop-in boundary for the per-timestep path of
 * LGMOak/HighPerformanceComputing-LatticeBoltzmannMethod.  The reference has no FFI layer; its
 * boundary is the header-level C++ API that src/main.cpp:11-21 and Solver::run consume.  The
 * C++ headers in this directory (LBMConfig.h, LBMGrid.h, LBMSolver.h, LBMIO.h) keep that API and
 * forward to the entry points below; tests and bench.py bind the same entry points with ctypes.
 * Each entry point names the reference interface it replaces (paths relative to the reference
 * repository root).
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative
 * lbm_status; lbm_last_error() gives the message.  One host thread per handle.  All device
 * work runs on streams owned by the handle.  There is no CPU fallback: without a CUDA device
 * lbm_create* fails with LBM_ERR_CUDA.
 *
 * Host array layouts are the reference's (include/LBMGrid.h:105-111):
 *   populations  padded AoS   [(gy*(lnx+2) + gx)*9 + i], gx in [0,lnx+2), gy in [0,ny+2)
 *   rho/ux/uy    interior     [y*lnx + x]
 *   solid mask   interior     [y*lnx + x], one byte per cell
 * where lnx is the width of this handle's x-slab (== nx for a single-GPU handle).
 */
#ifndef LBM_B200_H
#define LBM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LBM_B200_ABI_VERSION 2

typedef enum lbm_status {
    LBM_OK = 0,
    LBM_ERR_INVALID = -1,  /* bad argument / bad state */
    LBM_ERR_CUDA = -2,     /* CUDA runtime or driver error (incl. "no device") */
    LBM_ERR_NCCL = -3,
    LBM_ERR_NOMEM = -4,
    LBM_ERR_UNSTABLE = -5, /* only from calls documented to return it */
    LBM_ERR_IO = -6
} lbm_status;

/* Extensions beyond the reference (SURVEY.md F11: the reference has no periodic and no
 * body-force mode on this branch).  flags == 0 is exactly the reference's channel. */
enum {
    LBM_FLAG_PERIODIC_X = 1,  /* wrap in x instead of Zou-He inlet/outlet            */
    LBM_FLAG_PERIODIC_Y = 2,  /* wrap in y instead of the wall reflection             */
    LBM_FLAG_NO_CYLINDER = 4, /* obstacle-free domain                                 */
    LBM_FLAG_SHEAR_WAVE_INIT = 8, /* u = (inlet_velocity*sin(2*pi*y/ny), 0) initial field */
    LBM_FLAG_AA = 16 /* in-place AA-pattern variant: ONE population buffer instead of the A-B pair
                        (same populations bit for bit; rho/ux/uy equal to rounding).  Single slab. */
};

/* Mirrors LBM::SimulationParams (include/LBMConfig.h:36-52) field for field, then extensions. */
typedef struct lbm_params {
    double tau;
    double inlet_velocity;
    int32_t nx, ny;
    int32_t num_timesteps;
    int32_t output_frequency;
    double cylinder_x, cylinder_y, cylinder_radius; /* fractions of nx, ny, ny */
    int32_t vtk_start_step;
    int32_t flags;       /* LBM_FLAG_* */
    double body_force_x; /* f_eq + 3 w_i c_i.F form of include/LBMUtils.h:98,117 */
    double body_force_y;
} lbm_params;

typedef struct lbm_info {
    int32_t abi_version;
    int32_t global_nx, global_ny;
    int32_t local_nx, local_ny;
    int32_t x_start, y_start;
    int32_t rank, world;
    int32_t device;
    int32_t cyl_x, cyl_y, cyl_r; /* integer cells, LBMConfig.h:61-65 */
    int32_t solid_cells;         /* in this slab */
    int32_t links;               /* momentum-exchange links owned by this slab */
    int32_t iteration;           /* reference iterations completed so far */
    int64_t bytes_per_buffer;    /* one SoA population buffer on the device */
    int32_t row_pitch;           /* doubles between consecutive x columns in a plane */
    int32_t kernel_variant;
    int32_t halo_p2p;            /* 1: halo columns go by peer stores fused into the edge kernel (CUDA IPC over
                                    NVLink); 0: NCCL send/recv (or a single slab) */
    int32_t pass_depth;          /* reference iterations per launch and per trip through HBM (temporal blocking) */
    int32_t deep_solid_cells;    /* obstacle cells with eight solid neighbours: never loaded, computed or stored */
} lbm_info;

typedef struct lbm_solver* lbm_handle;

/* ---- lifecycle: Solver::Solver + Grid::Grid (include/LBMSolver.h:23, include/LBMGrid.h:57-103) ---- */
int lbm_create(const lbm_params* p, int device, lbm_handle* out);
/* One x-slab of a multi-GPU job, one process per GPU.  Replaces MPI_Cart_create and the
 * neighbour discovery of include/LBMGrid.h:347-364 with contiguous x-slabs (py == 1).
 * nccl_unique_id: the 128 bytes from lbm_nccl_unique_id() on rank 0, broadcast by the caller. */
int lbm_create_slab(const lbm_params* p, int device, int rank, int world, const void* nccl_unique_id,
                    lbm_handle* out);
int lbm_nccl_unique_id(void* out128);
int lbm_destroy(lbm_handle h);
const char* lbm_last_error(lbm_handle h); /* h may be NULL: error of the last failed create */
int lbm_get_info(lbm_handle h, lbm_info* out);

/* Rank discovery for a C++ driver started once per GPU by torchrun / mpirun / srun (used as
 * plain process launchers): replaces MPI_Init + MPI_Comm_rank/size of src/main.cpp:8 and
 * include/LBMGrid.h:58-59.  With world > 1 rank 0 creates the NCCL id and hands it to the other
 * ranks of the same launch through a file in /tmp (single node).  Without a launcher: 0 of 1. */
int lbm_bootstrap_env(int* rank, int* world, int* local_rank, void* nccl_unique_id_out128);
/* Change tau / inlet velocity / cylinder / output_frequency / body force after creation (the
 * reference's Grid is constructed from nx, ny alone and learns the rest in setup_geometry and
 * initialise, include/LBMGrid.h:57,152,185).  nx, ny and periodicity cannot change.
 * On a running handle the new values apply from the next iteration on, as if they had been changed between two
 * iterations of the reference: the observers still show the state the last iteration left, computed with the
 * parameters it ran with (its inlet rule, tau and body force), and the next iteration applies the old inlet rule to
 * the populations it pulls (the reference's boundary pass of the last iteration).  A new obstacle takes effect with
 * lbm_setup_geometry. */
int lbm_set_params(lbm_handle h, const lbm_params* p);

/* ---- set-up: Solver::initialise (include/LBMSolver.h:31-41) ---- */
/* Grid::setup_geometry, LBMGrid.h:152-183.  Rebuilds the mask and every table derived from it.  The populations are
 * those of the old geometry, so the handle is left uninitialised: lbm_step / lbm_run fail with LBM_ERR_INVALID until
 * lbm_initialise (or lbm_upload_f) gives it a state. */
int lbm_setup_geometry(lbm_handle h, int* solid_count);
/* Grid::initialise, LBMGrid.h:185-246: populations eq(1, inlet_u, 0), fluid ux = inlet_u, iteration 0, no stability
 * verdict, no forces rows, caller-written f_next values dropped.  The inlet rule keeps the params' inlet_velocity. */
int lbm_initialise(lbm_handle h, double inlet_u);

/* ---- the hot path: the loop body of Solver::run (include/LBMSolver.h:48-76) ---- */
/* Advance n reference iterations asynchronously: fused pull+boundary+collide kernels, the halo
 * exchange (Grid::exchange_ghost_cells, LBMGrid.h:249-283) and, on iterations t with
 * t % output_frequency == 0, the momentum-exchange reduction (IOManager::record_forces,
 * LBMIO.h:114-168).  Stability flags accumulate on the device (Grid::check_stability,
 * LBMGrid.h:285-317). */
int lbm_step(lbm_handle h, int n_steps);
/* Solver::run for n more iterations with the reference's observable behaviour: forces rows
 * {t, Fx, Fy, C_D, C_L} for every output step (LBMIO.h:171-185), up to max_rows; stops at the
 * first unstable iteration and reports it in *unstable_at (else -1), exactly the t of
 * "Simulation unstable at timestep t" (LBMSolver.h:60-64).  Returns LBM_OK also when unstable. */
int lbm_run(lbm_handle h, int n_steps, double* forces_rows, int max_rows, int* n_rows, int* unstable_at);
int lbm_sync(lbm_handle h);

/* IOManager::record_forces (LBMIO.h:114-168) for the current f_next: slab-local partial sums. */
int lbm_get_forces(lbm_handle h, double* fx, double* fy);
/* How the momentum-exchange sum over the link list is formed (LBMIO.h:123-160 adds the terms to one running sum
 * per component, solid cells in (y, x) order, directions i = 1..8):
 *   LBM_FORCES_ORDERED (default)  the same additions in the same order: the reference's bits, forces.csv byte for
 *                                 byte; one thread per component, ~10 ns per link (81 us at 7904 links);
 *   LBM_FORCES_TREE               a fixed parallel tree (warp shuffles + one shared-memory stage): deterministic from
 *                                 launch to launch, ~3 us whatever the link count, equal to the ordered sum to
 *                                 rounding (<= 1e-14 relative) -- for sampling the forces every (other) step. */
enum { LBM_FORCES_ORDERED = 0, LBM_FORCES_TREE = 1 };
int lbm_set_force_mode(lbm_handle h, int mode);
/* Grid::check_stability (LBMGrid.h:285-317) of the current f_current, plus everything flagged
 * since the last initialise/upload.  *first_bad_step is the reference timestep or -1. */
int lbm_check_stability(lbm_handle h, int* ok, int* first_bad_step);
/* Grid::max_velocity (LBMGrid.h:319-344): slab-local sqrt(max(ux^2+uy^2)). */
int lbm_max_velocity(lbm_handle h, double* out);

/* The reference's scalar reductions over ranks -- MPI_Reduce(SUM) of the force components
 * (LBMIO.h:167-168), MPI_Allreduce(MAX) of the velocity (LBMGrid.h:342), the solid count
 * (LBMGrid.h:175) -- as one in-place NCCL all-reduce of up to LBM_REDUCE_MAX host doubles.
 * Collective: every slab of the job must call it.  No-op for a single slab. */
enum { LBM_SUM = 0, LBM_MIN = 1, LBM_MAX = 2 };
#define LBM_REDUCE_MAX 64
int lbm_allreduce(lbm_handle h, double* values, int n, int op);
/* Solver::write_vtk_frame's gather (LBMSolver.h:269-362) and
 * IOManager::gather_and_reconstruct_field (LBMIO.h:225-300): rho/ux/uy of every slab assembled on
 * rank 0 as global row-major [y*global_nx + x] host arrays (peer slabs arrive over NCCL, then
 * strided D2H copies).  Collective; the pointers are ignored on ranks other than 0. */
int lbm_gather_macros(lbm_handle h, double* rho, double* ux, double* uy);

/* ---- observable state: Grid accessors (include/LBMGrid.h:115-129,145) ---- */
enum { LBM_F_CURRENT = 0, LBM_F_NEXT = 1 };
/* The padded AoS image of this slab.  Interior cells and the ghost ring of a single-slab handle equal the reference's
 * arrays bit for bit.  In a multi-slab job the ghost columns of f_next at a slab INTERFACE hold only the populations
 * the neighbouring GPU stores there (the ones this slab pulls across the face: 6 of 9 in the nearest column with the
 * temporally blocked passes, 3 of 9 with the one-iteration kernels); the reference's exchange copies all nine
 * (LBMGrid.h:395-491), none of the other six is ever read by an iteration. */
int lbm_download_f(lbm_handle h, int which, double* aos_padded);
int lbm_download_macros(lbm_handle h, double* rho, double* ux, double* uy);
int lbm_download_solid(lbm_handle h, unsigned char* mask);
/* Replace the state by a given f_current (padded AoS; ghost entries ignored).  Used for
 * restart and for parity tests on seeded random states.  `iteration` is the reference timestep
 * the next lbm_step will execute.  Allowed at any point of a run, with any kernel variant and pass depth: the run
 * goes on as the reference's would after writing f_current at that iteration boundary.  f_next keeps what the
 * reference's f_next holds there: w in solid cells and the initial equilibrium in the S/N ghost rows, or the values
 * an earlier lbm_upload_f_next wrote.  Until the next iteration the observers derived from f_next describe the
 * uploaded state as right after Grid::initialise: lbm_download_f(LBM_F_NEXT) returns f_current, lbm_get_forces sums
 * its links, rho / u are its moments (1 / 0 / 0 in solid cells), and lbm_check_stability reports no failure. */
int lbm_upload_f(lbm_handle h, const double* f_current_aos_padded, int iteration);

/* Grid::f_next written by the caller (LBMGrid.h:119-121 hands out a mutable reference).  At an iteration boundary of
 * the reference its streaming has already consumed f_next and the next collision overwrites every fluid cell, so
 * only the values of SOLID cells and of the S/N GHOST ROWS (corners included) live on: the next iteration's streaming
 * and every later one pull them.  Exactly those values are taken from the image (fluid cells and the W/E ghost
 * columns, which the exchange rewrites every step, are ignored) and take effect with the next iteration, as in the
 * reference; lbm_download_f shows them after that iteration.  They stay through later lbm_upload_f calls, until
 * lbm_initialise.  From this call on the handle runs the one-iteration kernels: the temporally blocked passes build
 * the default constants in.  Single-rank semantics per slab. */
int lbm_upload_f_next(lbm_handle h, const double* f_next_aos_padded);

/* ---- async output: replaces the MPI gathers of Solver::write_vtk_frame (LBMSolver.h:269-362)
 * and IOManager::gather_and_reconstruct_field (LBMIO.h:225-300).  Snapshots rho/ux/uy of the
 * current state into caller-owned host buffers (pinned via lbm_host_alloc for true overlap) on
 * a copy stream; the compute stream only waits for the on-device macro kernel. */
int lbm_snapshot_begin(lbm_handle h, double* rho, double* ux, double* uy);
int lbm_snapshot_wait(lbm_handle h);
/* The same with one completion event per slot, for a double-buffered writer thread:
 * lbm_snapshot_wait_slot only synchronises on that event and may be called from a second host
 * thread while the owning thread keeps stepping. */
#define LBM_SNAPSHOT_SLOTS 4
int lbm_snapshot_begin_slot(lbm_handle h, int slot, double* rho, double* ux, double* uy);
int lbm_snapshot_wait_slot(lbm_handle h, int slot);
/* ... into an image of the WHOLE channel that the slabs of a job fill side by side (rows of row_pitch doubles;
 * pass the address of this slab's first column): with the image in memory shared by the slab processes and
 * registered with lbm_host_register, every GPU writes its part by itself, asynchronously -- no gather, no collective
 * (the reference funnels every frame through MPI_Gatherv to rank 0, LBMSolver.h:289-337). */
int lbm_snapshot_begin_slot2d(lbm_handle h, int slot, double* rho, double* ux, double* uy, size_t row_pitch);
int lbm_host_register(void* ptr, size_t bytes); /* cudaHostRegister: page-lock memory the caller mapped (e.g. shm) */
int lbm_host_unregister(void* ptr);
int lbm_host_alloc(void** ptr, size_t bytes); /* cudaHostAlloc */
int lbm_host_free(void* ptr);

/* ---- measurement ---- */
/* Run n_steps and time them with CUDA events on the compute stream.  ms_total covers the whole
 * region; ms_bulk is the summed duration of the bulk collide-stream kernel launches only
 * (per_kernel = n > 0: events around the bulk launch of every n-th iteration). */
int lbm_time_steps(lbm_handle h, int n_steps, int per_kernel, float* ms_total, float* ms_bulk, int* launches);
/* Kernel launches issued by this handle since creation; launches and lattice cells of the bulk
 * collide-stream kernel covered by ms_bulk of the last lbm_time_steps(per_kernel=1). */
int lbm_get_counters(lbm_handle h, long long* launches, long long* bulk_launches, long long* bulk_cells);
/* Cell UPDATES of the launches lbm_get_counters reports (cells processed x iterations per pass): a temporally
 * blocked launch of depth T moves each cell through HBM once and updates it T times. */
int lbm_get_bulk_updates(lbm_handle h, long long* updates);
/* CUDA-event marks on the handle's compute stream (after everything its side streams have in
 * flight), so that a caller can time any sequence of entry points -- uploads, runs, downloads --
 * on the device rather than by wall clock. */
#define LBM_EVENT_SLOTS 8
int lbm_event_record(lbm_handle h, int slot);
int lbm_event_elapsed(lbm_handle h, int slot_a, int slot_b, float* ms);
/* Kernel variant of the collide-stream path:
 *   0  one iteration per launch pair (bulk + boundary fix-up), one cell per thread, any ny;
 *   1  the same with two y-adjacent cells per thread and 128-bit loads / stores (even ny, else 0):
 *      at the measured HBM peak for 144 B per update (DESIGN.md section 4);
 *   2  (default) temporal blocking: up to lbm_set_pass_depth() iterations per launch and per trip through
 *      HBM, intermediate states in shared memory, boundary rules inside the kernel (DESIGN.md section 4.2).
 * All three give the same bits.  In a multi-slab job the variant / depth can only change before the first
 * iteration after lbm_initialise / lbm_upload_f. */
int lbm_set_kernel_variant(lbm_handle h, int variant);
int lbm_set_pass_depth(lbm_handle h, int depth); /* 1..3, default 3 (LBM_B200_TB_DEPTH) */
/* The passes lbm_step(n_steps) launches from reference iteration `iteration` on (no device needed: pure host logic).
 * An iteration whose collision is an output step (iteration % output_frequency == 0: record_forces reads ITS
 * populations, LBMSolver.h:52-54) ends its pass; the first iteration after initialise / upload
 * (state_is_f_current != 0) stands alone.  Writes up to max_passes depths, returns the number of passes. */
int lbm_plan_passes(int iteration, int n_steps, int output_frequency, int max_depth, int state_is_f_current, int* depths,
                    int max_passes);
int lbm_device_count(int* n);
/* Self-test: the shared-reciprocal division the kernels use for u = j / rho (csrc/lbm_cell.cuh: div_pair) against the
 * IEEE-754 division on n pseudo-random operand triples (densities near 1 and over the whole exponent range, numerators
 * from +-0 and denormals to overflow, infinities and NaNs); *mismatches = quotients whose bits differ (must be 0). */
int lbm_selftest_division(lbm_handle h, long long n, unsigned long long seed, long long* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* LBM_B200_H */
