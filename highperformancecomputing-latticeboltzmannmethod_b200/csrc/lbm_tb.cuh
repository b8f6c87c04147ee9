// lbm_tb.cuh -- TEMPORAL BLOCKING: T lattice updates per pass over the population buffers.
//
// The A-B kernels of lbm_kernels.cu run at the HBM roofline of 144 B per update (9 fp64 loads + 9 fp64
// stores); the only way past it is to do more than one update per trip through HBM.  One thread block
// owns a strip of rows and marches along x through a chunk of columns.  At march step s (the SKEWED march,
// the default)
//   stage 1   updates column s            from the source buffer in HBM          (reference iteration t)
//   stage k   updates column s-2(k-1)     from stage k-1's ring in SHARED MEMORY (iteration t+k-1)
//   stage T   stores column s-2(T-1)      to the destination buffer in HBM
// so each population is read once and written once per T updates: 144/T B per update.  A stage's ring
// holds each population of a column until the next stage has pulled it (a pull needs the three columns c-1, c, c+1):
// two, three or four columns, depending on the population (see "the ring" below).  Because stage k lags TWO
// columns behind stage k-1, everything it reads was written in earlier steps: the stages of a step are
// independent, stage 1's loads fly while the later stages compute, and one __syncthreads ends the step.
// (The one-column-lag march -- stage k on column s-(k-1), a barrier between the stages, stage 1's loads
// issued a step ahead into a second cell of registers -- is kept for A/B runs: LBM_B200_TB_SKEW=0.)
// Every stage is the complete reference iteration for its
// cells -- pull (include/LBMSolver.h:128-145), boundary rules in the reference's serial order
// (:147-236), stability check (include/LBMGrid.h:285-317), BGK collision (:84-126) -- with the quirks
// of SURVEY.md F3/F4 reproduced as VALUES of the intermediate state: solid cells are w, ghost rows are
// eq(1,u_in,0), ghost columns at the physical inlet/outlet are 0, ghost columns at a slab interface
// are computed from a halo of width T that the neighbouring GPU stored into this slab's memory.
// The per-cell arithmetic is lbm_cell.cuh, so a pass of depth T is bit-identical to T single steps
// (tests/test_tb_emulation.py runs THIS code on the host, thread for thread, both marches;
// tests/test_gpu_tb.py on the GPU).
//
// Redundant work: a strip of B threads yields B-4 rows (each stage needs one more row on either side
// than the next), a chunk of XC columns costs XC + 2(T-1) stage-1 columns: 3 % + 3-6 % at B = 128, XC = 64.
//
// Two bodies run the march.  tb_step_skew is the GENERAL step: it decides per cell and per step what the cell is
// (ghost column, inlet, outlet, ghost row, obstacle, outside the stage's range) and is the only place where the
// boundary columns, the obstacle and the slab-edge chunks of a multi-GPU job are handled.  tb_fast_lane runs every
// stretch of steps whose columns are plain interior columns outside the obstacle (97 % of the steps of a 4096 x 8192
// slab): everything is decided once per thread, pointers advance by a column per step.  Same per-cell functions in the
// same order, so both give the same bits (the emulation runs both).
//
// Depth 3 is the default (lbm_engine.cu): at depth 2 the pass runs at 0.88 of the HBM peak, at depth 3 the fp64 pipe
// is the limit.  Depth 1 is the plain fused step (pull + rules + collide in ONE launch, no fix-up kernel); it is what
// multi-slab jobs use for the single steps between passes because it stores the same wide halo.
#pragma once

#include "lbm_cell.cuh"
#include "lbm_kernels.cuh"
#include "lbm_layout.h"

namespace lbm {

enum TbEdge {
    TB_EDGE_CONST = 0,  // physical inlet / outlet: the ghost column holds 0.0 (SURVEY.md F4)
    TB_EDGE_HALO = 1,   // slab interface: ghost columns hold the neighbour's populations
    TB_EDGE_WRAP = 2    // periodic in x inside one slab: column indices wrap
};

constexpr int TB_MAX_DEPTH = 3;   // == Layout::XO + 1 ghost columns are addressable

// ---- the ring ------------------------------------------------------------------------------------
// Stage k < T keeps the columns it computed in a ring in shared memory until stage k+1 has pulled them.  How long
// depends on the population.  In the skewed march stage k+1 pulls populations 3, 6, 7 (from x+1) of a column one
// step after it was stored, 0, 2, 4 (from x) two steps after and 1, 5, 8 (from x-1) three steps after; a column
// stored in step s is therefore dead after step s+1, s+2, s+3, and since a step has no barrier inside, it must not
// share a slot with the column stored in that last step either.  So the ring is three GROUPS, g = 0 (3, 6, 7),
// 1 (0, 2, 4), 2 (1, 5, 8), with g + 2 slots each, and the column stored in step s goes to slot s mod (g + 2) of
// every group: 27 planes of B doubles per stage instead of 4 x 9 (four depth-3 blocks of 128 rows fit an SM).  The
// one-column-lag march pulls one step earlier, after a barrier, and fits the same slots (tb_slots; both marches are
// replayed by tests/cpp/tb_ring_schedule.cpp).
// A slot is three planes of B doubles (one row per thread), in the order (row offset of the pull) +1, 0, -1:
//   group 0: 7, 3, 6   group 1: 4, 0, 2   group 2: 8, 1, 5
// so that the +-1-row reads of the first and last thread of a block (dead rows, computed by the fused lane) stay
// inside the slot and the ring needs no guard at its end.
constexpr int TB_RING_PLANES = 27;  // per stage

LBM_HD constexpr int tb_ring_slots(int g) { return g + 2; }

// Offset in doubles of the slot of group g in stage k's ring (1 <= k < T) that holds the column stored in march
// step s, row 0 (add the thread's row).
template <int B>
LBM_HD constexpr int tb_ring_at(int k, int g, int s) {
    const int n = tb_ring_slots(g);
    int slot = s % n;
    if (slot < 0) slot += n;
    return ((k - 1) * TB_RING_PLANES + 3 * (g * (g + 3) / 2 + slot)) * B;
}

// The slot term of tb_ring_at: offset of the slot that holds the column stored in step s from slot 0 of its group.
template <int B>
LBM_HD int tb_ring_slot(int g, int s) {
    return tb_ring_at<B>(1, g, s) - tb_ring_at<B>(1, g, 0);
}

// Stage k+1's pull of one cell (column c) out of stage k's ring / stage k's store of one cell into it.  o0, o1, o2:
// the slot offsets (tb_ring_slot) of group 0 / 1 / 2, i.e. of columns c+1, c, c-1 for the pull; rt = ring + tid.
template <int B>
LBM_HD void tb_ring_pull(const double* rt, int k, int o0, int o1, int o2, double f[Q]) {
    const double* e = rt + tb_ring_at<B>(k, 0, 0) + o0;
    const double* z = rt + tb_ring_at<B>(k, 1, 0) + o1;
    const double* w = rt + tb_ring_at<B>(k, 2, 0) + o2;
    f[7] = e[1];
    f[3] = e[B];
    f[6] = e[2 * B - 1];
    f[4] = z[1];
    f[0] = z[B];
    f[2] = z[2 * B - 1];
    f[8] = w[1];
    f[1] = w[B];
    f[5] = w[2 * B - 1];
}
template <int B>
LBM_HD void tb_ring_put(double* rt, int k, int o0, int o1, int o2, const double f[Q]) {
    double* e = rt + tb_ring_at<B>(k, 0, 0) + o0;
    double* z = rt + tb_ring_at<B>(k, 1, 0) + o1;
    double* w = rt + tb_ring_at<B>(k, 2, 0) + o2;
    e[0] = f[7];
    e[B] = f[3];
    e[2 * B] = f[6];
    z[0] = f[4];
    z[B] = f[0];
    z[2 * B] = f[2];
    w[0] = f[8];
    w[B] = f[1];
    w[2 * B] = f[5];
}

// One cell's populations into every slot of stage k's ring (steps 0 .. 3 cover the slots of every group).
template <int B>
LBM_HD void tb_ring_fill(double* rt, int k, const double f[Q]) {
#pragma unroll 1
    for (int s = 0; s < tb_ring_slots(2); ++s) tb_ring_put<B>(rt, k, tb_ring_slot<B>(0, s), tb_ring_slot<B>(1, s), tb_ring_slot<B>(2, s), f);
}

struct TbArgs {
    const double* src;
    double* dst;
    Layout L;
    double tau_inv, Fx, Fy;
    int* first_bad;
    int bad_iter;  // reference timestep whose check_stability stage 1's pulled values belong to (stage k: + k-1)
    BcArgs bc;
    const unsigned char* mask;  // padded, Layout indexing: 0 fluid, 1 solid, 2 solid with eight solid neighbours
    int mask_lo, mask_hi;       // slab columns [lo, hi) (ghost columns count) that may hold solid cells
    int mask_ylo, mask_yhi;     // ... and the rows [ylo, yhi) they lie in: strips outside never look at the mask
    int west, east;             // TbEdge
    int periodic_y;
    int pull;   // depth 1 only: 0 = the first iteration after initialise / upload (collide f_current as it is)
    int write;  // 0: check / observe only, no population is stored
    int x_begin, x_end, xc;  // interior chunks tile [x_begin, x_end) in pieces of xc columns ...
    int edge_cols;           // ... after chunk 0 = [0, edge_cols) and chunk 1 = [lnx-edge_cols, lnx) when > 0
    int halo_w;              // ghost columns a slab interface keeps up to date (the deepest pass of the job)
    // rho / ux / uy exactly as the LAST stage's collision stores them (include/LBMSolver.h:112-114), in
    // the slab's native order [x*ny + y]; nullptr: not wanted
    double *m_rho, *m_ux, *m_uy;
    P2pArgs px;  // multi-slab: peer buffers and the hand-shake words (lbm_kernels.cuh)
    // BYTE offsets relative to (plane 0, column c, row y), filled in by tb_fill_offsets: population i is PULLED
    // from ld_off[i] = 8 (i*plane - c_ix*PY - c_iy) and stored at st_off[i] = 8 i*plane; col_bytes = 8 PY.  Kernel
    // parameters, so that an address is one 64-bit add of a constant-bank operand to a per-thread pointer.
    long long ld_off[Q], st_off[Q], col_bytes;
    long long pf_off[Q];  // 8 (i*plane - c_ix*PY): the column segment population i is pulled from, 16-byte aligned
    int pf_dist;          // columns the L2 prefetch runs ahead of the loads (0: off)
    long long plane_mul[5];  // k * 8 * plane bytes, k = 0..4 (the fast lane's pointer chains)
    int fast_lane;        // 1: plain unmasked stretches of the skewed march take tb_fast_lane (0: A/B runs, tests)
};

inline void tb_fill_offsets(TbArgs& a) {
    for (int i = 0; i < Q; ++i) {
        a.ld_off[i] = 8 * ((long long)i * a.L.plane - (long long)cxi(i) * a.L.PY - cyi(i));
        a.st_off[i] = 8 * (long long)i * a.L.plane;
        a.pf_off[i] = 8 * ((long long)i * a.L.plane - (long long)cxi(i) * a.L.PY);
    }
    a.col_bytes = 8 * (long long)a.L.PY;
    for (int k = 0; k < 5; ++k) a.plane_mul[k] = 8 * (long long)k * a.L.plane;
}

// Keeps a per-thread pointer in its registers as ONE 64-bit value (the compiler would otherwise re-derive it from
// base + 8*index at every use: four integer instructions per access instead of two).
template <class P>
LBM_HD P tb_opaque(P p) {
#if defined(__CUDA_ARCH__)
    asm volatile("" : "+l"(p));
#endif
    return p;
}
// The same for a 32-bit value.  Used for the thread / block indices: re-read from the special registers inside the
// march loop (S2R, which the compiler prefers to spending a register) they sit on a scoreboard shared with the
// prefetch loads just issued, and their first use then waits for a whole trip to memory.
// (A warp shuffle of the value with itself: the one thing neither compiler stage re-derives from %tid / %ctaid.)
LBM_HD int tb_opaque_int(int v) {
#if defined(__CUDA_ARCH__)
    v = __shfl_sync(0xffffffffu, v, threadIdx.x & 31);
#endif
    return v;
}

// ---- host / device glue (the host side exists for the thread-for-thread emulation only) ----------
#if defined(__CUDA_ARCH__)
#define TB_SYNC() __syncthreads()
#define TB_LD(p, coherent) ((coherent) ? __ldcg(p) : __ldg(p))
#define TB_FLAG(ptr, v) atomicMin((ptr), (v))
// (the per-thread pointers are opaque 64-bit values, see tb_opaque: say "global" explicitly)
#define TB_ST(ptr, v) asm volatile("st.global.f64 [%0], %1;" ::"l"(ptr), "d"(v) : "memory")
#define TB_COLD __device__ __host__ __noinline__
#define TB_PREFETCH_L2(p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p))
#define TB_COUNT(which, n) ((void)0)
#else
void tb_host_sync();
void tb_host_flag(int* p, int v);
#define TB_SYNC() tb_host_sync()
#define TB_LD(p, coherent) (*(p))
#define TB_FLAG(ptr, v) tb_host_flag((ptr), (v))
#define TB_ST(ptr, v) (*reinterpret_cast<double*>(ptr) = (v))
#define TB_COLD inline
#define TB_PREFETCH_L2(p) ((void)(p))
void tb_host_count(int which, int n);  // march steps a block took on the fast lane (0) / the general step (1)
#define TB_COUNT(which, n) tb_host_count((which), (n))
#endif

LBM_HD int tb_wrap(int v, int n) {
    v %= n;
    return v < 0 ? v + n : v;
}

template <int T, int B>
struct TbShape {
    static constexpr int ROFF = (T == 1) ? 0 : 2;  // thread j works on row strip*H - ROFF + j
    static constexpr int H = B - 2 * ROFF;         // rows a strip stores (a multiple of four: whole 32-byte sectors)
    static constexpr int RING_DOUBLES = tb_ring_at<B>(T, 0, 0);  // the rings of stages 1 .. T-1
    static_assert(T >= 1 && T <= TB_MAX_DEPTH, "depth");
    static_assert(ROFF >= T - 1, "row overlap");
};

// The chunk of columns [x0, x1) block `chunk` stores; edge = it reads ghost columns / feeds a neighbour.
LBM_HD void tb_chunk(const TbArgs& a, int chunk, int& x0, int& x1, bool& edge) {
    const int lnx = a.L.lnx;
    edge = false;
    if (a.edge_cols > 0) {
        if (chunk == 0) { x0 = 0; x1 = a.edge_cols; edge = true; return; }
        if (chunk == 1) { x0 = lnx - a.edge_cols; x1 = lnx; edge = true; return; }
        chunk -= 2;
    }
    x0 = a.x_begin + chunk * a.xc;
    x1 = x0 + a.xc < a.x_end ? x0 + a.xc : a.x_end;
}

// What one thread holds for one cell of one stage.
struct TbCell {
    double f[Q];
    int kind;  // 0: nothing here; 1: pulled populations, still to be ruled / checked / collided;
               // 2: ghost row (eq(1,u_in,0)); 3: ghost column at a physical edge (0.0); 4: obstacle cell whose
               // eight neighbours are solid (w, nothing to check)
    int m;     // mask byte of the cell (kind 1): 0 fluid, 1 solid
    int xr;    // its slab column (wrapped in a periodic slab)
};

// The thread's fixed view of its row and of the block's chunk.
template <int T, int B>
struct TbRow {
    int tid, y, yr, row_kind;  // row kinds: 0 dead, 1 a cell to compute (row yr), 2 ghost row holding eq(1,u_in,0)
    bool wall_b, wall_t, out_row, edge;
    bool strip_walls;          // (uniform over the block) some row of this strip is a wall row
    int x0, x1;
    const char* srow;  // a.src + the offset of row yr inside a column (column gx = -XO)
    char* drow;        // a.dst + the offset of row y
    bool on[T];          // stage k works on this row
    const char* pf_seg;  // (uniform) start of the block's row segment in column gx = -XO of plane 0, 16-byte aligned
    int pf_bytes;        // (uniform) its length; 0: no L2 prefetch
    int pf_last;         // (uniform) last column worth prefetching: the end of this block's own march
};

// Column kind for stage k (uniform over the block): 0 dead, 1 compute cell column xr, 2 ghost column at a physical
// edge (0.0; corners: e).
template <int T>
LBM_HD int tb_col_kind(const TbArgs& a, int x0, int x1, int k, int c, int& xr) {
    const int grow = T - k;  // how far stage k reaches beyond the columns the block stores
    const int lnx = a.L.lnx;
    xr = c;
    if (c < x0 - grow || c >= x1 + grow) return 0;
    if (c >= 0 && c < lnx) return 1;
    const int mode = c < 0 ? a.west : a.east;
    if (mode == TB_EDGE_WRAP) { xr = tb_wrap(c, lnx); return 1; }
    if (mode == TB_EDGE_HALO) return 1;  // (inside the halo by construction of the chunks)
    return (c == -1 || c == lnx) ? 2 : 0;
}

// Classification shared by both halves of a stage.  PLAIN: the caller guarantees an interior column that is
// neither the inlet nor the outlet column and lies inside the stage's range (no column logic at all);
// MASKED = false: ... and no obstacle cell in it (no mask load either).
template <int T, int B, bool PLAIN>
LBM_HD void tb_classify(const TbArgs& a, const TbRow<T, B>& r, int k, int c, bool masked, TbCell& cell) {
    cell.kind = 0;
    cell.m = 0;
    cell.xr = c;
    if (!r.on[k - 1]) return;
    int col_kind = 1;
    if (!PLAIN) {
        col_kind = tb_col_kind<T>(a, r.x0, r.x1, k, c, cell.xr);
        if (col_kind == 0) return;
    }
    if (r.row_kind == 2) { cell.kind = 2; return; }
    if (!PLAIN && col_kind == 2) { cell.kind = 3; return; }
    cell.kind = 1;
    if (masked) {
        const int gx = cell.xr + 1;
        if (gx >= a.mask_lo && gx < a.mask_hi) {
            cell.m = a.mask[a.L.at(gx, r.yr)];
            if (cell.m == 2) cell.kind = 4;
        }
    }
}

// Stage 1, first half: classify the cell (c, row) and ISSUE its nine loads.  Called one march step ahead of
// tb_finish, so that the loads of column s+1 are in flight while columns s, s-1, ... are being computed.
// Periodic edges are addressed naturally: the ghost rows / columns hold wrapped copies (k_wrap after every pass).
template <int T, int B, bool PLAIN>
LBM_HD void tb_issue(const TbArgs& a, const TbRow<T, B>& r, int c, bool masked, TbCell& cell) {
    tb_classify<T, B, PLAIN>(a, r, 1, c, masked, cell);
    if (cell.kind != 1) return;
    const char* p = r.srow + (long long)(cell.xr + 1 + Layout::XO) * a.col_bytes;
    // the lean path never runs in a slab-edge chunk: one flavour of load
    const bool coherent = PLAIN ? false : r.edge;
    if ((T > 1) || a.pull) {
        // population i comes from column xr - c_ix, row yr - c_iy (reference include/LBMSolver.h:138-142)
#pragma unroll
        for (int i = 0; i < Q; ++i) cell.f[i] = TB_LD(reinterpret_cast<const double*>(p + a.ld_off[i]), coherent);
    } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) cell.f[i] = TB_LD(reinterpret_cast<const double*>(p + a.st_off[i]), coherent);
    }
}

// The ring slots a march step uses (uniform): every stage stores into st[g] (tb_ring_slot of the step) and pulls from
// pl[g].  The skewed march pulls from group g the column stored g + 1 steps before, the one-column-lag march
// (a barrier between the stages) the one stored g steps before: slot s+1 resp. s+2 mod (g + 2).
struct TbSlots {
    int st[3], pl[3];
};
template <int B>
LBM_HD TbSlots tb_slots(int s, bool skew) {
    TbSlots o;
#pragma unroll
    for (int g = 0; g < 3; ++g) {
        o.st[g] = tb_ring_slot<B>(g, s);
        o.pl[g] = tb_ring_slot<B>(g, s + (skew ? 1 : 2));
    }
    return o;
}
// ... of the next step of the skewed march: the slots pulled from become the ones stored into
template <int B>
LBM_HD void tb_slots_advance(TbSlots& o) {
#pragma unroll
    for (int g = 0; g < 3; ++g) {
        o.st[g] = o.pl[g];
        o.pl[g] = o.pl[g] + 3 * B == tb_ring_slots(g) * 3 * B ? 0 : o.pl[g] + 3 * B;
    }
}

// Stage k >= 2, first half: the same cell from stage k-1's ring in shared memory.
template <int T, int B, bool PLAIN>
LBM_HD void tb_from_ring(const TbArgs& a, const TbRow<T, B>& r, const double* ring, int k, int c, const TbSlots& o,
                         bool masked, TbCell& cell) {
    tb_classify<T, B, PLAIN>(a, r, k, c, masked, cell);
    if (cell.kind != 1) return;
    tb_ring_pull<B>(ring + r.tid, k - 1, o.pl[0], o.pl[1], o.pl[2], cell.f);
}

// (cold, kept out of line: the hot loop should fit the instruction cache) a constant cell into stage k's ring, slots
// o0, o1, o2.  which: 2 eq(1,u_in,0), 3 zero, 4 w (the kinds of TbCell).  `a` is a __grid_constant__ kernel parameter:
// taking its address costs nothing.
template <int B>
TB_COLD void tb_ring_const(double* rt, int k, int o0, int o1, int o2, const TbArgs& a, int which) {
    double v[Q];
#pragma unroll
    for (int i = 0; i < Q; ++i) v[i] = which == 3 ? 0.0 : (which == 2 ? a.bc.e[i] : a.bc.w[i]);
    tb_ring_put<B>(rt, k, o0, o1, o2, v);
}

// The last stage's populations of an edge column into the neighbours' ghost columns (peer memory over NVLink).
// Column lnx-1-d goes to the east neighbour's ghost column gx = -d.  What it needs of that column, for a pass of
// depth halo_w: the populations moving towards it (1,5,8) always; the ones that stay in the column (0,2,4) where
// it recomputes the column itself (d <= halo_w-2); the ones moving away (3,6,7) where it also recomputes the
// column beyond (d <= halo_w-3).
template <int T, int B>
LBM_HD void tb_push(const TbArgs& a, const TbRow<T, B>& r, int c, const double* f) {
    const Layout& L = a.L;
    const int lnx = L.lnx;
    const int de = lnx - 1 - c, dw = c;
    if (a.px.peer_dst_east && de < a.halo_w) {
        double* q = a.px.peer_dst_east + L.at(-de, r.y);
        q[1 * L.plane] = f[1];
        q[5 * L.plane] = f[5];
        q[8 * L.plane] = f[8];
        if (de <= a.halo_w - 2) {
            q[0 * L.plane] = f[0];
            q[2 * L.plane] = f[2];
            q[4 * L.plane] = f[4];
        }
        if (de <= a.halo_w - 3) {
            q[3 * L.plane] = f[3];
            q[6 * L.plane] = f[6];
            q[7 * L.plane] = f[7];
        }
    }
    if (a.px.peer_dst_west && dw < a.halo_w) {
        double* q = a.px.peer_dst_west + L.at(lnx + 1 + dw, r.y);
        q[3 * L.plane] = f[3];
        q[6 * L.plane] = f[6];
        q[7 * L.plane] = f[7];
        if (dw <= a.halo_w - 2) {
            q[0 * L.plane] = f[0];
            q[2 * L.plane] = f[2];
            q[4 * L.plane] = f[4];
        }
        if (dw <= a.halo_w - 3) {
            q[1 * L.plane] = f[1];
            q[5 * L.plane] = f[5];
            q[8 * L.plane] = f[8];
        }
    }
}

// Second half of every stage: boundary rules, stability check, collision; then the ring (k < T, slots o.st) or HBM and
// the neighbours' ghost columns (k == T).  Returns true when a checked value was unstable.
template <int T, int B, bool FORCED, bool PLAIN>
LBM_HD bool tb_finish(const TbArgs& a, const TbRow<T, B>& r, double* ring, int k, int c, const TbSlots& o, TbCell& cell) {
    const Layout& L = a.L;
    const int lnx = L.lnx, ny = L.ny;
    if (cell.kind == 0) return false;
    if (cell.kind != 1) {
        // ---- cold: constants.  Written from the argument block straight to the ring: nothing is merged into the
        // registers of the hot path.
        if (k < T) {
            tb_ring_const<B>(ring + r.tid, k, o.st[0], o.st[1], o.st[2], a, cell.kind);
        } else if (cell.kind == 4) {
            if (a.m_rho) {  // include/LBMSolver.h:260-261; rho keeps the constructor's 1.0
                const long long g = (long long)c * ny + r.y;
                a.m_rho[g] = 1.0;
                a.m_ux[g] = 0.0;
                a.m_uy[g] = 0.0;
            }
            if (T == 1 && !a.pull && a.write) {
                char* q = r.drow + (long long)(c + 1 + Layout::XO) * a.col_bytes;
#pragma unroll
                for (int i = 0; i < Q; ++i) TB_ST(q + a.st_off[i], a.bc.w[i]);
            }
            if (!PLAIN && r.edge && a.write) tb_push<T, B>(a, r, c, a.bc.w);  // the neighbour pulls w from here
        }
        return false;
    }
    bool bad = false;
    double* f = cell.f;
    const bool rules = (T > 1) || a.pull;  // the first iteration has no boundary pass before it
    if (rules && cell.m == 0) {
        // the reference's serial order: bottom, top, inlet, outlet (SURVEY.md F5)
        if (r.strip_walls) {
            if (r.wall_b) wall_bottom(f);
            if (r.wall_t) wall_top(f);
        }
        if (!PLAIN) {
            if (a.bc.inlet && cell.xr == 0) (void)zou_he_inlet(f, a.bc.u_in);
            if (a.bc.outlet && cell.xr == lnx - 1) (void)zou_he_outlet(f);
        }
    }
    if (rules) {
#pragma unroll
        for (int i = 0; i < Q; ++i) bad |= unstable_value(f[i]);
    }
    if (cell.m != 0) {
        // ---- cold: an obstacle cell with a fluid neighbour: checked (the reference's check sees what streams into
        // it), then w for ever (SURVEY.md F3)
        if (k < T) {
            tb_ring_const<B>(ring + r.tid, k, o.st[0], o.st[1], o.st[2], a, 4);
        } else {
            if (a.m_rho) {
                const long long g = (long long)c * ny + r.y;
                a.m_rho[g] = 1.0;
                a.m_ux[g] = 0.0;
                a.m_uy[g] = 0.0;
            }
            if (a.write) {
                // never stored -- except by the first iteration after an upload, whose destination may hold anything
                char* q = r.drow + (long long)(c + 1 + Layout::XO) * a.col_bytes;
                if (T == 1 && !a.pull) {
#pragma unroll
                    for (int i = 0; i < Q; ++i) TB_ST(q + a.st_off[i], a.bc.w[i]);
                }
                if (!PLAIN && r.edge) tb_push<T, B>(a, r, c, a.bc.w);
            }
        }
        return bad;
    } else {
        const Moments mo = moments(f);
        if (k == T && a.m_rho) {
            const long long g = (long long)c * ny + r.y;
            a.m_rho[g] = mo.rho;
            a.m_ux[g] = mo.ux;
            a.m_uy[g] = mo.uy;
        }
        if (FORCED)
            bgk_forced(f, mo, a.tau_inv, a.Fx, a.Fy, f);
        else
            bgk(f, mo, a.tau_inv, f);
        if (k < T) {
            tb_ring_put<B>(ring + r.tid, k, o.st[0], o.st[1], o.st[2], f);
            return bad;
        }
        if (!a.write) return bad;
        // ---- the last stage: HBM ...
        char* q = r.drow + (long long)(c + 1 + Layout::XO) * a.col_bytes;
#pragma unroll
        for (int i = 0; i < Q; ++i) TB_ST(q + a.st_off[i], f[i]);
    }
    if (!PLAIN && r.edge) tb_push<T, B>(a, r, c, f);  // ... and the neighbours' ghost columns over NVLink
    return bad;
}

// L2 prefetch, by the bulk-copy engine: ONE thread of the block asks for the nine column segments the block's loads
// of march step `col` will touch (cp.async.bulk.prefetch.L2: a 2 KB segment per instruction, no register, no
// scoreboard).  The register prefetch of tb_step covers one step; a step is shorter than a trip to HBM, so the lines
// are pulled into L2 pf_dist steps earlier.
template <int T, int B>
LBM_HD void tb_prefetch_l2(const TbArgs& a, const char* seg, int bytes, int col) {
#if defined(__CUDA_ARCH__)
    if (col > a.L.lnx) return;
    const char* p = seg + (long long)(col + 1 + Layout::XO) * a.col_bytes;
#pragma unroll
    for (int i = 0; i < Q; ++i)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p + a.pf_off[i]), "r"(bytes) : "memory");
#else
    (void)a; (void)seg; (void)bytes; (void)col;
#endif
}

// One march step: stage 1 on column s (`cur`: its loads were issued a step ago), stages 2..T behind it, and the
// loads of column s+1 into `nxt`.  PLAIN: see tb_classify; masked (uniform): the columns this step touches may hold
// obstacle cells.
template <int T, int B, bool FORCED, bool PLAIN>
LBM_HD void tb_step(const TbArgs& a, const TbRow<T, B>& r, double* ring, int s, bool issue_next, bool masked, TbCell& cur,
                    TbCell& nxt, bool bad[T]) {
    if (r.tid == 0 && r.pf_bytes > 0 && s + 1 + a.pf_dist <= r.pf_last) tb_prefetch_l2<T, B>(a, r.pf_seg, r.pf_bytes, s + 1 + a.pf_dist);
    if (issue_next) tb_issue<T, B, PLAIN>(a, r, s + 1, masked, nxt);
    const TbSlots o = tb_slots<B>(s, false);
    bad[0] |= tb_finish<T, B, FORCED, PLAIN>(a, r, ring, 1, s, o, cur);
#pragma unroll
    for (int k = 2; k <= T; ++k) {
        TB_SYNC();  // stage k-1's column of this step is in its ring
        tb_from_ring<T, B, PLAIN>(a, r, ring, k, s - (k - 1), o, masked, cur);
        bad[k - 1] |= tb_finish<T, B, FORCED, PLAIN>(a, r, ring, k, s - (k - 1), o, cur);
    }
}

// The SKEWED march step (the default): stage k works on column s - 2(k-1), TWO columns behind stage k-1 instead of
// one.  Everything stage k reads was then written in EARLIER steps, so the T stages of a step are independent of one
// another: the loads of stage 1's column are issued first, the later stages (whose inputs are already in shared
// memory) compute while those loads fly, stage 1 finishes last, and ONE barrier ends the step.  No second cell of
// prefetched registers, no loop unrolled by two, and the instruction streams of the stages can overlap.
template <int T, int B, bool FORCED, bool PLAIN>
LBM_HD void tb_step_skew(const TbArgs& a, const TbRow<T, B>& r, double* ring, int s, bool masked, bool bad[T]) {
    if (r.tid == 0 && r.pf_bytes > 0 && s + a.pf_dist <= r.pf_last) tb_prefetch_l2<T, B>(a, r.pf_seg, r.pf_bytes, s + a.pf_dist);
    TbCell first;
    tb_issue<T, B, PLAIN>(a, r, s, masked, first);
    const TbSlots o = tb_slots<B>(s, true);
#pragma unroll
    for (int k = T; k >= 2; --k) {
        TbCell cell;
        tb_from_ring<T, B, PLAIN>(a, r, ring, k, s - 2 * (k - 1), o, masked, cell);
        bad[k - 1] |= tb_finish<T, B, FORCED, PLAIN>(a, r, ring, k, s - 2 * (k - 1), o, cell);
    }
    bad[0] |= tb_finish<T, B, FORCED, PLAIN>(a, r, ring, 1, s, o, first);
    if (T > 1) TB_SYNC();
}

// The FAST LANE of the skewed march: march steps [s, s_end) whose T columns are all plain interior columns (see
// tb_classify's PLAIN) without an obstacle cell, in a pass that stores populations and nothing else (no macro
// emission) -- on the 4096 x 8192 slab that is 95 % of all steps.  Everything the general step decides per cell is
// decided once per thread here: a thread either computes its row at stage k (act[k-1]) or does nothing (ghost rows
// hold eq(1,u_in,0) in every ring slot from tb_thread's prologue on).  The per-thread pointers advance by one column
// per step, so an access costs one 64-bit add of a constant-bank operand.  Same per-cell arithmetic, same order
// (walls, stability check, moments, collision) as tb_finish: bit-identical by construction, and checked thread for
// thread by the host emulation.
// The populations of one cell of the fast lane, loaded / stored along a CHAIN of per-thread pointers: plane i+1 is
// plane i plus ONE constant (8*plane bytes), so the loop needs two 64-bit constants instead of eighteen (which the
// compiler would keep in uniform registers, run out of them and spill).  The pulled column x - c_ix is one of three
// column pointers, the row shift -c_iy is the load's immediate offset.
LBM_HD void tb_chain_load(const char* pl, long long col_bytes, const long long* pm, double f[Q]) {
    const char* p0 = pl;                                 // c_ix =  0: populations 0, 2, 4
    const char* pw = tb_opaque(pl - col_bytes);          // c_ix = +1: populations 1, 5, 8 come from column x - 1
    const char* pe = tb_opaque(pl + col_bytes);          // c_ix = -1: populations 3, 6, 7 come from column x + 1
    f[0] = TB_LD(reinterpret_cast<const double*>(p0), false);
    pw = tb_opaque(pw + pm[1]);
    f[1] = TB_LD(reinterpret_cast<const double*>(pw), false);
    p0 = tb_opaque(p0 + pm[2]);
    f[2] = TB_LD(reinterpret_cast<const double*>(p0) - 1, false);
    pe = tb_opaque(pe + pm[3]);
    f[3] = TB_LD(reinterpret_cast<const double*>(pe), false);
    p0 = tb_opaque(p0 + pm[2]);
    f[4] = TB_LD(reinterpret_cast<const double*>(p0) + 1, false);
    pw = tb_opaque(pw + pm[4]);
    f[5] = TB_LD(reinterpret_cast<const double*>(pw) - 1, false);
    pe = tb_opaque(pe + pm[3]);
    f[6] = TB_LD(reinterpret_cast<const double*>(pe) - 1, false);
    pe = tb_opaque(pe + pm[1]);
    f[7] = TB_LD(reinterpret_cast<const double*>(pe) + 1, false);
    pw = tb_opaque(pw + pm[3]);
    f[8] = TB_LD(reinterpret_cast<const double*>(pw) + 1, false);
}
LBM_HD void tb_chain_store(char* ps, long long plane_bytes, const double f[Q]) {
    char* q = ps;
#pragma unroll
    for (int i = 0; i < Q; ++i) {
        TB_ST(q, f[i]);
        if (i + 1 < Q) q = tb_opaque(q + plane_bytes);
    }
}

// The per-cell work of the fast lane: walls, stability check, moments, collision -- tb_finish's sequence for a
// fluid cell of a plain column.
template <bool FORCED>
LBM_HD bool tb_fast_cell(const TbArgs& a, bool strip_walls, bool wall_b, bool wall_t, double f[Q], Moments& mo) {
    if (strip_walls) {  // (uniform over the block: two strips of the slab)
        if (wall_b) wall_bottom(f);
        if (wall_t) wall_top(f);
    }
    bool u = false;
#pragma unroll
    for (int i = 0; i < Q; ++i) u |= unstable_value(f[i]);
    mo = moments(f);
    if (FORCED)
        bgk_forced(f, mo, a.tau_inv, a.Fx, a.Fy, f);
    else
        bgk(f, mo, a.tau_inv, f);
    return u;
}

template <int T, int B, bool FORCED>
LBM_HD void tb_fast_lane(const TbArgs& a, const TbRow<T, B>& r, double* ring, int s, const int s_end, bool bad[T]) {
    bool act[T];
#pragma unroll
    for (int k = 0; k < T; ++k) act[k] = r.on[k] && r.row_kind == 1;
    const long long plane_bytes = a.st_off[1];
    // L2 prefetch, one 128-byte line per thread: thread j asks for line j % PF_LINES of population j / PF_LINES of the
    // column the block pulls pf_dist steps from now (the nine segments of ~1 KB the bulk prefetch of the other steps
    // covers with nine instructions of ONE thread -- here the work is one instruction in three of the four warps
    // instead of fifty in the first one, which every barrier would wait for).
    constexpr int PF_LINES = (B * 8 + 32 + 2 * 127) / 128;  // lines a segment of up to B + 4 rows can touch
    static_assert(Q * PF_LINES <= B || B < 128, "one prefetch line per thread (the emulation's small blocks: a hint only)");
    const char* pfp = nullptr;
    if (r.pf_bytes > 0 && r.tid < Q * PF_LINES) {
        const int pop = r.tid / PF_LINES, line = r.tid - pop * PF_LINES;
        const int skew = (int)(reinterpret_cast<unsigned long long>(r.pf_seg) & 127);  // the segment starts mid-line
        if (line * 128 < r.pf_bytes + skew)
            pfp = tb_opaque(r.pf_seg - skew + a.pf_off[pop] + line * 128 + (long long)(s + a.pf_dist + 1 + Layout::XO) * a.col_bytes);
    }
    // stage 1 pulls column s; the last stage stores column s - 2(T-1)
    const char* pl = tb_opaque(r.srow + (long long)(s + 1 + Layout::XO) * a.col_bytes);
    char* ps = tb_opaque(r.drow + (long long)(s - 2 * (T - 1) + 1 + Layout::XO) * a.col_bytes);
    double* const rt = ring + r.tid;
    TbSlots o = tb_slots<B>(s, true);  // (uniform, advanced by one slot per step)
    for (; s < s_end; ++s) {
        if (pfp && s + a.pf_dist <= r.pf_last) TB_PREFETCH_L2(pfp);
        // stage k works on column s - 2(k-1) while that lies in its range [x0 - (T-k), x1 + (T-k)) (uniform)
        bool now[T];
#pragma unroll
        for (int k = 1; k <= T; ++k) {
            const int c = s - 2 * (k - 1);
            now[k - 1] = act[k - 1] && c >= r.x0 - (T - k) && c < r.x1 + (T - k);
        }
        double f1[Q];
        if (now[0]) tb_chain_load(pl, a.col_bytes, a.plane_mul, f1);
#pragma unroll
        for (int k = T; k >= 2; --k) {
            if (!now[k - 1]) continue;
            const int c = s - 2 * (k - 1);
            double f[Q];
            tb_ring_pull<B>(rt, k - 1, o.pl[0], o.pl[1], o.pl[2], f);
            Moments mo;
            bad[k - 1] |= tb_fast_cell<FORCED>(a, r.strip_walls, r.wall_b, r.wall_t, f, mo);
            if (k < T) {
                tb_ring_put<B>(rt, k, o.st[0], o.st[1], o.st[2], f);
            } else {
                if (a.m_rho) {  // (uniform; the last pass before an output only)
                    const long long g = (long long)c * a.L.ny + r.y;
                    a.m_rho[g] = mo.rho;
                    a.m_ux[g] = mo.ux;
                    a.m_uy[g] = mo.uy;
                }
                tb_chain_store(ps, plane_bytes, f);
            }
        }
        if (now[0]) {
            Moments mo;
            bad[0] |= tb_fast_cell<FORCED>(a, r.strip_walls, r.wall_b, r.wall_t, f1, mo);
            if (T > 1) {
                tb_ring_put<B>(rt, 1, o.st[0], o.st[1], o.st[2], f1);
            } else {
                if (a.m_rho) {
                    const long long g = (long long)s * a.L.ny + r.y;
                    a.m_rho[g] = mo.rho;
                    a.m_ux[g] = mo.ux;
                    a.m_uy[g] = mo.uy;
                }
                tb_chain_store(ps, plane_bytes, f1);
            }
        }
        pl = tb_opaque(pl + a.col_bytes);
        ps = tb_opaque(ps + a.col_bytes);
        if (pfp) pfp = tb_opaque(pfp + a.col_bytes);
        tb_slots_advance<B>(o);
        if (T > 1) TB_SYNC();
    }
}

// The fast lane with the stages T..2 FUSED (experimental, k_tb<..., FUSED = true>): their cells come from shared
// memory, so all of them are available at once; their arithmetic is written side by side -- the moment sums of all
// cells, ONE branch for all divisions, the collisions -- so that the double-precision dependency chains of T-1
// independent cells interleave in one basic block (the kernel is bound by exactly those chains: ncu's stall_wait and
// the fp64 pipe at 62 %).  Every thread computes (rows that are off at a stage work on whatever the ring holds,
// nothing of it is stored or flagged), which removes the per-thread branches as well.  Only for steps in which every
// stage lies inside its column range: the caller gives the chunk's first and last steps to tb_fast_lane.
template <int T, int B, bool FORCED>
LBM_HD void tb_fast_lane_fused(const TbArgs& a, const TbRow<T, B>& r, double* ring, int s, const int s_end, bool bad[T]) {
    constexpr int K = T > 1 ? T - 1 : 1;  // fused cells: stage k = j + 2 is cell j
    bool act[T];
#pragma unroll
    for (int k = 0; k < T; ++k) act[k] = r.on[k] && r.row_kind == 1;
    const long long plane_bytes = a.st_off[1];
    constexpr int PF_LINES = (B * 8 + 32 + 2 * 127) / 128;
    const char* pfp = nullptr;
    if (r.pf_bytes > 0 && r.tid < Q * PF_LINES) {
        const int pop = r.tid / PF_LINES, line = r.tid - pop * PF_LINES;
        const int skew = (int)(reinterpret_cast<unsigned long long>(r.pf_seg) & 127);
        if (line * 128 < r.pf_bytes + skew)
            pfp = tb_opaque(r.pf_seg - skew + a.pf_off[pop] + line * 128 + (long long)(s + a.pf_dist + 1 + Layout::XO) * a.col_bytes);
    }
    const char* pl = tb_opaque(r.srow + (long long)(s + 1 + Layout::XO) * a.col_bytes);
    char* ps = tb_opaque(r.drow + (long long)(s - 2 * (T - 1) + 1 + Layout::XO) * a.col_bytes);
    double* const rt = ring + r.tid;
    TbSlots o = tb_slots<B>(s, true);
    for (; s < s_end; ++s) {
        if (pfp && s + a.pf_dist <= r.pf_last) TB_PREFETCH_L2(pfp);
        double f1[Q];
        if (act[0]) tb_chain_load(pl, a.col_bytes, a.plane_mul, f1);
        // ---- stages T..2, side by side ----
        double f[K][Q], rho[K], mx[K], my[K];
        Moments mo[K];
        bool window = true;
#pragma unroll
        for (int j = K - 1; j >= 0; --j) tb_ring_pull<B>(rt, j + 1, o.pl[0], o.pl[1], o.pl[2], f[j]);
        if (r.strip_walls) {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (r.wall_b) wall_bottom(f[j]);
                if (r.wall_t) wall_top(f[j]);
            }
        }
#pragma unroll
        for (int j = K - 1; j >= 0; --j) {
            bool u = false;
#pragma unroll
            for (int i = 0; i < Q; ++i) u |= unstable_value(f[j][i]);
            bad[j + 1] |= u && act[j + 1];
            moment_sums(f[j], rho[j], mx[j], my[j]);
            window = window && div_pair_window(mx[j], my[j], rho[j]);
        }
        if (window) {
#pragma unroll
            for (int j = K - 1; j >= 0; --j) {
                mo[j].rho = rho[j];
                div_pair_core(mx[j], my[j], rho[j], mo[j].ux, mo[j].uy);
            }
        } else {
#pragma unroll
            for (int j = K - 1; j >= 0; --j) {
                mo[j].rho = rho[j];
                div_pair(mx[j], my[j], rho[j], mo[j].ux, mo[j].uy);
            }
        }
#pragma unroll
        for (int j = K - 1; j >= 0; --j) {
            if (FORCED)
                bgk_forced(f[j], mo[j], a.tau_inv, a.Fx, a.Fy, f[j]);
            else
                bgk(f[j], mo[j], a.tau_inv, f[j]);
        }
#pragma unroll
        for (int j = K - 1; j >= 0; --j) {
            if (!act[j + 1]) continue;
            const int c = s - 2 * (j + 1);
            if (j + 2 < T) {
                tb_ring_put<B>(rt, j + 2, o.st[0], o.st[1], o.st[2], f[j]);
            } else {
                if (a.m_rho) {  // (uniform; the last pass before an output only)
                    const long long g = (long long)c * a.L.ny + r.y;
                    a.m_rho[g] = mo[j].rho;
                    a.m_ux[g] = mo[j].ux;
                    a.m_uy[g] = mo[j].uy;
                }
                tb_chain_store(ps, plane_bytes, f[j]);
            }
        }
        // ---- stage 1 (its loads have been flying meanwhile) ----
        if (act[0]) {
            Moments m1;
            bad[0] |= tb_fast_cell<FORCED>(a, r.strip_walls, r.wall_b, r.wall_t, f1, m1);
            tb_ring_put<B>(rt, 1, o.st[0], o.st[1], o.st[2], f1);
        }
        pl = tb_opaque(pl + a.col_bytes);
        ps = tb_opaque(ps + a.col_bytes);
        if (pfp) pfp = tb_opaque(pfp + a.col_bytes);
        tb_slots_advance<B>(o);
        TB_SYNC();
    }
}

// One thread of one block: `tid` in [0, B), rows of strip `strip`, columns of chunk `chunk`.
// `ring` is the block's shared memory (TbShape::RING_DOUBLES doubles).
template <int T, int B, bool FORCED, bool SKEW = true, bool FUSED = false>
LBM_HD void tb_thread(const TbArgs& a, double* ring, int tid_, int strip_, int chunk_) {
    using S = TbShape<T, B>;
    const int tid = tb_opaque_int(tid_), strip = tb_opaque_int(strip_), chunk = tb_opaque_int(chunk_);
    const int ny = a.L.ny, lnx = a.L.lnx;
    TbRow<T, B> r;
    tb_chunk(a, chunk, r.x0, r.x1, r.edge);
    if (r.x0 >= r.x1) return;  // (uniform over the block)

    // ---- this thread's row -------------------------------------------------------------------
    r.tid = tid;
    r.y = strip * S::H - S::ROFF + tid;
    r.yr = r.y;
    if (a.periodic_y) {
        r.row_kind = (r.y >= -(T - 1) && r.y < ny + (T - 1)) ? 1 : 0;
        r.yr = tb_wrap(r.y, ny);
    } else {
        r.row_kind = (r.y >= 0 && r.y < ny) ? 1 : ((r.y == -1 || r.y == ny) ? 2 : 0);
    }
    r.wall_b = a.bc.walls && r.yr == 0;
    r.wall_t = a.bc.walls && r.yr == ny - 1;
    {
        const int lo = strip * S::H - S::ROFF, hi = lo + B;  // rows of this block
        r.strip_walls = a.bc.walls && ((lo <= 0 && hi > 0) || (lo <= ny - 1 && hi > ny - 1) || a.periodic_y);
    }
    r.out_row = (tid >= S::ROFF && tid < S::ROFF + S::H && r.y >= 0 && r.y < ny);  // rows the last stage stores
#pragma unroll
    for (int k = 1; k <= T; ++k) {
        const int grow = T - k;  // how far stage k reaches beyond the rows the block stores
        r.on[k - 1] = r.row_kind != 0 && tid >= S::ROFF - grow && tid < S::ROFF + S::H + grow && (k < T || r.out_row);
    }
    r.srow = tb_opaque(reinterpret_cast<const char*>(a.src + (Layout::YO + r.yr)));
    r.drow = tb_opaque(reinterpret_cast<char*>(a.dst + (Layout::YO + r.y)));
    r.pf_bytes = 0;
    r.pf_seg = nullptr;
    if (a.pf_dist > 0) {
        // the rows the block's pulls touch, [strip*H - ROFF - 1, ... + B + 2), widened to whole 16-byte pairs and
        // clipped to the column
        int first = strip * S::H - S::ROFF - 1;
        int last = first + B + 2;
        if (first < -Layout::YO) first = -Layout::YO;
        if (last > a.L.PY - Layout::YO) last = a.L.PY - Layout::YO;
        first &= ~1;
        last = (last + 1) & ~1;
        if (last > first) {
            r.pf_seg = reinterpret_cast<const char*>(a.src + (Layout::YO + first));
            r.pf_bytes = (last - first) * 8;
        }
    }
    bool bad[T];
#pragma unroll
    for (int k = 0; k < T; ++k) bad[k] = false;

    // ---- the march ---------------------------------------------------------------------------------
    const int c_lo = (a.west == TB_EDGE_CONST && a.bc.inlet) ? 1 : 0;           // first plain column
    const int c_hi = (a.east == TB_EDGE_CONST && a.bc.outlet) ? lnx - 1 : lnx;  // one past the last plain column
    if (SKEW) {
        // Stage k on column s - 2(k-1).  Steps whose T columns are all plain interior columns (not a ghost column, not
        // the inlet or outlet column) with every stage inside its range take the lean path.
        const int s_first = r.x0 - (T - 1), s_last = r.x1 - 1 + 2 * (T - 1);
        int p0 = (r.x0 > c_lo ? r.x0 : c_lo) + 2 * (T - 1);
        int p1 = (r.x1 + (T - 2) < c_hi - 1 ? r.x1 + (T - 2) : c_hi - 1) + 1;  // lean steps: [p0, p1)
        if (r.edge) p1 = p0;  // the few slab-edge columns also feed the neighbour: general path
        r.pf_last = r.x1 + (T - 2) < lnx ? r.x1 + (T - 2) : lnx;  // the last column stage 1 loads
        // the columns s-2(T-1) .. s a step touches may hold obstacle cells iff they meet [mask_lo - 1, mask_hi - 1)
        int m0 = a.mask_lo - 1, m1 = a.mask_hi - 1 + 2 * (T - 1);  // steps s in [m0, m1) are masked
        {
            // ... for the strips whose rows meet the obstacle's rows (uniform over the block)
            const int lo = strip * S::H - S::ROFF;
            if (!a.periodic_y && (lo >= a.mask_yhi || lo + B <= a.mask_ylo)) m1 = m0;
        }
        // ghost rows: eq(1,u_in,0) in every ring slot, once, so that the fast lane never has to look at them (the
        // other steps keep writing the same values); the first step's barrier publishes it
        if (T > 1 && r.row_kind == 2) {
#pragma unroll
            for (int k = 1; k < T; ++k)
                if (r.on[k - 1]) tb_ring_fill<B>(ring + r.tid, k, a.bc.e);
        }
        // The fast lane takes every step whose columns are plain and unmasked: in a chunk that touches neither slab
        // edge that is the whole march (the stages switch themselves on and off at the chunk's ends), otherwise the
        // steps [p0, p1) with every stage inside its range.
        const bool fast = a.write && ((T > 1) || a.pull) && a.fast_lane;
        int q0 = p0, q1 = p1;
        if (!r.edge && r.x0 - (T - 1) >= c_lo && r.x1 + (T - 1) <= c_hi) { q0 = s_first; q1 = s_last + 1; }
        if (!fast) q1 = q0;
        int s = s_first;
        while (s <= s_last) {
            if (s >= q0 && s < q1 && !(s >= m0 && s < m1)) {
                // up to the obstacle columns, or from behind them to the end of the stretch
                const int e = (s < m0 && m0 < q1) ? m0 : q1;
                if (tid == 0) TB_COUNT(0, e - s);
                if constexpr (FUSED && T > 2) {
                    // every stage inside its range for s in [p0, p1): those steps with the stages T..2 fused, the
                    // chunk's first and last steps on the plain fast lane (one call site: the loop is not unrolled)
                    const int f0 = s > p0 ? s : p0, f1 = e < p1 ? e : p1;
                    const bool any = f0 < f1;
#pragma unroll 1
                    for (int seg = 0; seg < 3; ++seg) {
                        const int to = !any ? e : (seg == 0 ? f0 : (seg == 1 ? f1 : e));
                        if (s >= to) continue;
                        if (seg == 1 && any) tb_fast_lane_fused<T, B, FORCED>(a, r, ring, s, to, bad);
                        else tb_fast_lane<T, B, FORCED>(a, r, ring, s, to, bad);
                        s = to;
                    }
                } else {
                    tb_fast_lane<T, B, FORCED>(a, r, ring, s, e, bad);
                }
                s = e;
                continue;
            }
            if (tid == 0) TB_COUNT(1, 1);
            tb_step_skew<T, B, FORCED, false>(a, r, ring, s, true, bad);
            ++s;
        }
    } else {
    // Stage k on column s - (k-1), stage 1's loads issued one step ahead into a second cell of registers.
    // Steps whose T columns s, s-1, ..., s-(T-1) are all plain interior columns with every stage inside its range
    // take the lean path; [p0, p1) also keeps column s+1 plain.
    const int s_first = r.x0 - (T - 1), s_last = r.x1 + (T - 2);
    int p0 = r.x0 + (T - 1), p1 = s_last;  // every stage active for s in [x0+T-1, s_last]; s+1 <= s_last
    if (p0 < c_lo + (T - 1)) p0 = c_lo + (T - 1);
    if (p1 > c_hi - 1) p1 = c_hi - 1;
    if (r.edge) p1 = p0;  // the few slab-edge columns also feed the neighbour: general path
    r.pf_last = s_last < lnx ? s_last : lnx;
    // Two cells take turns: while one is being computed the other one's loads (the next column) are in flight.
    TbCell ca, cb;
    tb_issue<T, B, false>(a, r, s_first, true, ca);
    int s = s_first;
    bool a_is_cur = true;
    // the columns s-(T-1) .. s+1 a step touches may hold obstacle cells iff they meet [mask_lo - 1, mask_hi - 1)
    const int m0 = a.mask_lo - 2, m1 = a.mask_hi - 1 + (T - 1);  // steps s in [m0, m1) are masked
    while (s <= s_last) {
        if (a_is_cur && s >= p0 && s + 1 < p1) {
            // a stretch of lean steps, unrolled by two so that the two cells keep their roles (no register copies)
            for (; s + 1 < p1; s += 2) {
                tb_step<T, B, FORCED, true>(a, r, ring, s, true, s >= m0 && s < m1, ca, cb, bad);
                tb_step<T, B, FORCED, true>(a, r, ring, s + 1, true, s + 1 >= m0 && s + 1 < m1, cb, ca, bad);
            }
            continue;
        }
        if (a_is_cur) tb_step<T, B, FORCED, false>(a, r, ring, s, s < s_last, true, ca, cb, bad);
        else tb_step<T, B, FORCED, false>(a, r, ring, s, s < s_last, true, cb, ca, bad);
        a_is_cur = !a_is_cur;
        ++s;
    }
    }
#pragma unroll
    for (int k = 0; k < T; ++k)
        if (bad[k]) TB_FLAG(a.first_bad, a.bad_iter + k);
}

// ---- launch interface (lbm_tb.cu) -----------------------------------------------------------
// depth 1..TB_MAX_DEPTH.  Fills in the chunking (x_begin / x_end / xc / edge_cols) itself.
cudaError_t launch_tb(int depth, TbArgs a, bool p2p, cudaStream_t s);
// Finish emitted macros: native [x*ny+y] -> the reference's interior row-major [y*lnx+x], with the inlet /
// outlet overrides of the boundary pass that follows the last collision (include/LBMSolver.h:203-205,
// 232-234), which are functions of the newest buffer alone.
cudaError_t launch_macros_finish(const ObserveArgs& o, const double* m_rho, const double* m_ux, const double* m_uy,
                                 double* rho, double* ux, double* uy, cudaStream_t s);
bool tb_worthwhile(const Layout& L);
int tb_rows_per_block(int depth);
size_t tb_shared_bytes(int depth);

}  // namespace lbm
