// lbm_engine.cu -- host side of liblbm_b200.so: the slab object behind an lbm_handle, the step
// scheduler (what Solver::run's loop body becomes, reference include/LBMSolver.h:48-76), the halo
// exchange (Grid::exchange_ghost_cells, include/LBMGrid.h:249-283 -> the three populations that cross
// each slab face, stored into the neighbour GPU's ghost column by the step kernel itself over CUDA-IPC
// peer memory, or sent by NCCL where IPC is unavailable), and the extern "C" entry points of
// include/lbm_b200.h.
//
// State convention (SURVEY.md Appendix A).  After t >= 1 reference iterations buffer f[cur] holds
// the POST-COLLISION populations f_next of iteration t-1 and f[cur^1] still holds the state the
// last launch read.  Every reference observable is derived from those two buffers on demand
// (lbm_kernels.cu: k_macros, k_export_f), so the hot kernels store nothing but populations.
// The ghost ring of both buffers permanently holds what the reference's f_next ghosts hold from
// its first exchange on: 0.0 in the W/E ghost columns at physical domain edges, the initial
// equilibrium in the S/N ghost rows and the four corners (SURVEY.md F4); slab-interface ghost
// columns are refreshed by the exchange every iteration.
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <string>
#include <fcntl.h>
#include <unistd.h>
#include <vector>

#include "../../include/lbm_b200.h"
#include "lbm_cell.cuh"
#include "lbm_kernels.cuh"
#include "lbm_layout.h"
#include "lbm_nccl.h"
#include "lbm_tb.cuh"

using namespace lbm;

namespace {
thread_local std::string g_create_error;
std::string g_id_file;  // rank 0: NCCL id file of lbm_bootstrap_env, removed after the communicator is up
constexpr int FORCE_SLOTS = 1024;
}  // namespace

struct lbm_solver {
    lbm_params p{};
    Layout L{};
    int device = 0, rank = 0, world = 1;
    int cyl_x = 0, cyl_y = 0, cyl_r = 0;
    bool periodic_x = false, periodic_y = false;

    cudaStream_t stream = nullptr, copy_stream = nullptr, comm_stream = nullptr;
    cudaEvent_t ev_macros = nullptr, ev_snapshot = nullptr, ev_edge = nullptr, ev_comm = nullptr;
    bool snapshot_pending = false;
    cudaEvent_t ev_slot[LBM_SNAPSHOT_SLOTS] = {};  // completion of the D2H copies of lbm_snapshot_begin_slot

    double* f[2] = {nullptr, nullptr};
    int cur = 0;
    bool cur_is_next = false, prev_is_next = false, fresh = false, initialised = false;
    int iter = 0;

    std::vector<unsigned char> h_mask;  // padded, Layout indexing
    unsigned char* d_mask = nullptr;
    int2* d_ring = nullptr;
    int n_ring = 0;
    int2* d_solids = nullptr;
    int n_solid = 0;
    int n_ring_edge = 0;  // leading ring entries that lie in columns 0 / lnx-1 (the edge kernels redo those columns)
    // Per-column solid runs (StepArgs::cols): where the solid cells of a column form one run the
    // bulk kernels never store them, so they keep w without any reset.  The solid list is ordered
    // [cells of columns without such a run][layer-1 cells: a non-solid neighbour][the rest]:
    // the A-B fix-up resets only the first group every step, the AA fix-up the first two (fluid
    // cells push into layer-1 cells in O-steps); the first iteration after initialise / upload
    // resets every solid cell.
    int4* d_cols = nullptr;
    int col_lo = 0, col_hi = 0;  // columns whose table entry is not empty
    int n_solid_loose = 0, n_solid_l1 = 0;
    bool col_skip = true;
    Link* d_links = nullptr;
    int n_links = 0;

    double *d_rho = nullptr, *d_ux = nullptr, *d_uy = nullptr;
    bool macros_valid = false;
    // Temporal blocking (variant BULK_TB, lbm_tb.cuh): passes of up to tb_depth iterations.  `lag` is the
    // number of iterations between f[cur ^ 1] and f[cur] (the observers of rho / u want 1); the last stage
    // of a pass can emit the moments its collision read in the slab's native order (d_m*), valid for the
    // state after iteration macros_native_iter - 1.
    int tb_depth = 3;
    int lag = 1;
    double *d_mrho = nullptr, *d_mux = nullptr, *d_muy = nullptr;
    int macros_native_iter = -1;
    long long* d_custom_off = nullptr;  // lbm_upload_f_next: (offset, value) of the solid / ghost-row populations written
    double* d_custom_val = nullptr;
    int n_custom = 0;
    int custom_pending = 0;  // ... to be installed into the destination of each of the next two iterations (lbm_upload_f_next)
    bool custom_state = false;  // the caller wrote f_next (solid / ghost-row values may no longer be the constants the
                                // temporally blocked passes build in): one-iteration kernels from then on
    int force_tree = 0;      // LBM_FORCES_TREE: fixed parallel reduction tree instead of the reference's serial order
    bool emit_last = false;  // lbm_run: the last pass of the call emits (the caller will look at the fields)
    int mask_lo = 0, mask_hi = 0;  // padded columns gx in [lo, hi) hold solid cells
    int mask_ylo = 0, mask_yhi = 0;  // ... in rows [ylo, yhi)
    long long n_deep = 0;          // interior solid cells whose eight neighbours are solid (never touched)
    // lbm_download_f / lbm_upload_f: the padded AoS image crosses PCIe in row chunks through two staging buffers,
    // the copy of one chunk overlapping the transpose kernel of the other (no full-size third buffer)
    double* d_stage[2] = {nullptr, nullptr};
    int stage_rows = 0;  // padded rows per chunk (a multiple of 32)
    cudaEvent_t ev_stage_copied[2] = {nullptr, nullptr}, ev_stage_free[2] = {nullptr, nullptr};
    unsigned long long* d_maxbits = nullptr;

    int* d_first_bad = nullptr;
    double* d_forces = nullptr;  // FORCE_SLOTS x {fx, fy}
    struct Pending { int t, slot; };
    std::vector<Pending> pending;
    struct ForceRow { int t; double fx, fy; };
    std::vector<ForceRow> force_log;

    // in-place AA variant (LBM_FLAG_AA): one buffer f[0]; see lbm_aa.cu
    bool aa = false;
    int aa_phase = 0;  // 0 natural layout, 1 reversed layout
    AaFill* d_fills = nullptr;
    int n_fill = 0;
    Link *d_links_rev = nullptr, *d_links_nat = nullptr;  // link offsets in the reversed / pushed-natural layouts
    double* d_ring_out = nullptr;

    BcArgs bc{};
    // The parameters the last iteration ran with.  lbm_set_params replaces h->p and h->bc at once, but the boundary
    // rules of the last iteration are applied by the NEXT launch (it pulls that iteration's populations), and the
    // observers rebuild that iteration's state: both use these (mark_run copies them when an iteration is launched).
    double run_tau_inv = 0.0, run_Fx = 0.0, run_Fy = 0.0;
    BcArgs run_bc{};
    double init_u = 0.0;
    int variant = BULK_TB;
    bool overlap = true;

    ncclComm_t comm = nullptr;
    // Fused edge + halo kernel over CUDA-IPC peer memory (k_edge_p2p); NCCL send/recv is the fallback.
    bool p2p = false;
    int* d_flags = nullptr;              // [0] from west, [1] from east: last exchange delivered by that neighbour
    unsigned int* d_blocks_done = nullptr;
    double* peer_f[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [side: 0 west, 1 east][buffer]
    int* peer_flags[2] = {nullptr, nullptr};
    void* ipc_opened[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
    int edge_seq = 0;                    // exchanges issued so far (identical on every rank)
    int* d_status = nullptr;             // non-zero: a halo wait timed out (lbm_device.cuh); sticky
    unsigned long long halo_timeout_ns = 30ull * 1000000000ull;
    bool halo_failed = false;
    double* d_red = nullptr;       // small device scratch for lbm_allreduce
    double* d_gather = nullptr;    // rank 0: one slab of rho/ux/uy received from a peer
    int* d_first_bad_all = nullptr;
    int west = -1, east = -1;  // neighbour ranks or -1

    long long launches = 0;
    std::vector<cudaEvent_t> bulk_events;  // pairs, only while per-kernel timing is on
    int time_bulk = 0;  // 0 = off, n = events around the bulk launch of every n-th iteration
    long long bulk_timed_launches = 0, bulk_timed_cells = 0;  // of the last lbm_time_steps(per_kernel)
    long long bulk_timed_updates = 0;                         // cell updates of those launches (cells x pass depth)
    cudaEvent_t marks[LBM_EVENT_SLOTS] = {};                  // lbm_event_record / lbm_event_elapsed

    std::string err;
};

namespace {

int fail(lbm_handle h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}

#define CU(h, expr)                                                                                   \
    do {                                                                                              \
        cudaError_t e__ = (expr);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return fail(h, LBM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));        \
    } while (0)

#define NC(h, expr)                                                                                   \
    do {                                                                                              \
        ncclResult_t r__ = (expr);                                                                    \
        if (r__ != ncclSuccess)                                                                       \
            return fail(h, LBM_ERR_NCCL, std::string(#expr) + ": " + nccl_api().GetErrorString(r__)); \
    } while (0)

#define CHECK_H(h) \
    if (!(h)) return fail(nullptr, LBM_ERR_INVALID, "null handle")

StepArgs step_args(lbm_handle h, const double* src, double* dst, int bad_iter, int write) {
    StepArgs a;
    a.src = src;
    a.dst = dst;
    a.L = h->L;
    a.tau_inv = 1.0 / h->p.tau;  // include/LBMSolver.h:85
    a.Fx = h->p.body_force_x;
    a.Fy = h->p.body_force_y;
    a.forced = (a.Fx != 0.0 || a.Fy != 0.0) ? 1 : 0;
    a.first_bad = h->d_first_bad;
    a.bad_iter = bad_iter;
    a.write = write;
    a.cols = h->d_cols;
    a.col_lo = h->col_lo;
    a.col_hi = h->col_hi;
    return a;
}

// Every launch of an iteration ends with this: from now on its parameters are the ones still owed (see run_bc).
void mark_run(lbm_handle h) {
    h->run_tau_inv = 1.0 / h->p.tau;
    h->run_Fx = h->p.body_force_x;
    h->run_Fy = h->p.body_force_y;
    h->run_bc = h->bc;
}

ObserveArgs observe_args(lbm_handle h) {
    ObserveArgs o;
    o.cur = h->f[h->cur];
    o.prev = h->f[h->cur ^ 1];
    o.L = h->L;
    o.mask = h->d_mask;
    o.bc = h->run_bc;
    o.cur_is_next = h->cur_is_next;
    o.prev_is_next = h->prev_is_next;
    o.fresh = h->fresh;
    o.shear_wave = (h->p.flags & LBM_FLAG_SHEAR_WAVE_INIT) ? 1 : 0;
    o.u0 = h->init_u;
    return o;
}

AaArgs aa_args(lbm_handle h, int first) {
    AaArgs a;
    a.f = h->f[0];
    a.L = h->L;
    a.tau_inv = 1.0 / h->p.tau;
    a.Fx = h->p.body_force_x;
    a.Fy = h->p.body_force_y;
    a.forced = (a.Fx != 0.0 || a.Fy != 0.0) ? 1 : 0;
    a.first_bad = h->d_first_bad;
    a.bad_iter = h->iter - 1;
    a.first = first;
    a.skip_rows = h->bc.walls;
    a.x_begin = h->bc.inlet ? 1 : 0;
    a.x_end = h->bc.outlet ? h->L.lnx - 1 : h->L.lnx;
    a.variant = h->variant;
    a.cols = h->d_cols;
    a.col_lo = h->col_lo;
    a.col_hi = h->col_hi;
    return a;
}

AaObserve aa_observe(lbm_handle h) {
    AaObserve o;
    o.f = h->f[0];
    o.L = h->L;
    o.mask = h->d_mask;
    o.bc = h->run_bc;
    o.phase = h->aa_phase;
    o.cur_is_next = h->cur_is_next;
    o.fresh = h->fresh;
    o.ring_out = h->d_ring_out;
    o.periodic_x = h->periodic_x;
    o.periodic_y = h->periodic_y;
    o.open_w = (h->periodic_x || h->west >= 0) ? 1 : 0;
    o.open_e = (h->periodic_x || h->east >= 0) ? 1 : 0;
    o.west_zero = (h->periodic_x || h->west >= 0) ? 0 : 1;
    o.east_zero = (h->periodic_x || h->east >= 0) ? 0 : 1;
    o.shear_wave = (h->p.flags & LBM_FLAG_SHEAR_WAVE_INIT) ? 1 : 0;
    o.u0 = h->init_u;
    o.tau_inv = h->run_tau_inv;
    o.Fx = h->run_Fx;
    o.Fy = h->run_Fy;
    return o;
}

// Geometry on the host: mask over the padded slab in GLOBAL coordinates (reference
// include/LBMGrid.h:159-172), the solid list, the boundary-ring list and the momentum-exchange
// link list (include/LBMIO.h:123-160; a link is owned by the slab that owns its fluid end, so
// no link is lost at a slab face -- cf. SURVEY.md F8).
int build_geometry(lbm_handle h) {
    const Layout& L = h->L;
    const bool cyl = !(h->p.flags & LBM_FLAG_NO_CYLINDER);
    std::fill(h->h_mask.begin(), h->h_mask.end(), 0);
    auto solid_global = [&](int gxg, int gyg) -> bool {
        if (!cyl) return false;
        if (h->periodic_x) gxg = ((gxg % L.gnx) + L.gnx) % L.gnx;
        if (h->periodic_y) gyg = ((gyg % L.ny) + L.ny) % L.ny;
        if (gxg < 0 || gxg >= L.gnx || gyg < 0 || gyg >= L.ny) return false;
        const double dx = gxg - h->cyl_x;
        const double dy = gyg - h->cyl_y;
        const double dist_sq = dx * dx + dy * dy;
        return dist_sq <= h->cyl_r * h->cyl_r;
    };
    std::vector<int2> solids, ring;
    std::vector<Link> links, links_rev, links_nat;
    h->mask_lo = L.lnx + 2 + Layout::XO;
    h->mask_hi = -Layout::XO;
    h->mask_ylo = L.ny + 1;
    h->mask_yhi = -1;
    for (int gx = -Layout::XO; gx < L.lnx + 2 + Layout::XO; ++gx)  // the wide ghost columns of lbm_tb.cuh included
        for (int y = -1; y <= L.ny; ++y) {
            const bool s = solid_global(L.x_start + gx - 1, y);
            h->h_mask[L.at(gx, y)] = s ? 1 : 0;
            if (s) {
                h->mask_lo = std::min(h->mask_lo, gx);
                h->mask_hi = std::max(h->mask_hi, gx + 1);
                h->mask_ylo = std::min(h->mask_ylo, y);
                h->mask_yhi = std::max(h->mask_yhi, y + 1);
            }
            if (s && gx >= 1 && gx <= L.lnx && y >= 0 && y < L.ny) solids.push_back(make_int2(gx - 1, y));
        }
    // ring: fluid cells that get a boundary rule between pull and collide
    {
        std::vector<int2> cand;
        if (h->bc.walls)
            for (int x = 0; x < L.lnx; ++x) {
                cand.push_back(make_int2(x, 0));
                cand.push_back(make_int2(x, L.ny - 1));
            }
        for (int y = 0; y < L.ny; ++y) {
            if (h->bc.inlet) cand.push_back(make_int2(0, y));
            if (h->bc.outlet) cand.push_back(make_int2(L.lnx - 1, y));
        }
        std::sort(cand.begin(), cand.end(), [](const int2& a, const int2& b) { return a.x != b.x ? a.x < b.x : a.y < b.y; });
        cand.erase(std::unique(cand.begin(), cand.end(), [](const int2& a, const int2& b) { return a.x == b.x && a.y == b.y; }),
                   cand.end());
        for (const int2& c : cand)
            if (!h->h_mask[L.at(c.x + 1, c.y)]) ring.push_back(c);
    }
    // Cells of the two slab-edge columns go first in both lists: with a neighbouring slab they
    // are fixed up before the halo leaves, ahead of the interior (see step_one).
    auto edge_first = [&](std::vector<int2>& v) -> int {
        auto mid = std::stable_partition(v.begin(), v.end(), [&](const int2& c) { return c.x == 0 || c.x == L.lnx - 1; });
        return (int)(mid - v.begin());
    };
    h->n_ring_edge = edge_first(ring);
    std::vector<int4> cols((size_t)L.lnx, make_int4(0, 0, 0, 0));
    {
        auto deep = [&](int x, int y) -> bool {  // solid with eight solid neighbours
            for (int i = 1; i < Q; ++i)
                if (!h->h_mask[L.at(x + 1 - cxi(i), y - cyi(i))]) return false;
            return true;
        };
        std::vector<char> loose_col((size_t)L.lnx, 0);
        for (int x = 0; x < L.lnx; ++x) {
            int ys = -1, ye = -1, n = 0, ds = -1, de = -1, nd = 0;
            for (int y = 0; y < L.ny; ++y) {
                if (!h->h_mask[L.at(x + 1, y)]) continue;
                if (ys < 0) ys = y;
                ye = y + 1;
                ++n;
                if (deep(x, y)) {
                    if (ds < 0) ds = y;
                    de = y + 1;
                    ++nd;
                }
            }
            if (n == 0) continue;
            if (!h->col_skip || ye - ys != n) {  // several runs in this column: the list-driven reset handles it
                loose_col[x] = 1;
                continue;
            }
            cols[x] = (nd > 0 && de - ds == nd) ? make_int4(ys, ye, ds, de) : make_int4(ys, ye, 0, 0);
        }
        auto l1 = [&](const int2& c) { return !deep(c.x, c.y); };
        auto m0 = std::stable_partition(solids.begin(), solids.end(), [&](const int2& c) { return loose_col[c.x] != 0; });
        auto m1 = std::stable_partition(m0, solids.end(), l1);
        h->n_solid_loose = (int)(m0 - solids.begin());
        h->n_solid_l1 = (int)(m1 - m0);
        h->col_lo = L.lnx;
        h->col_hi = 0;
        for (int x = 0; x < L.lnx; ++x)
            if (cols[x].y > cols[x].x) {
                h->col_lo = std::min(h->col_lo, x);
                h->col_hi = std::max(h->col_hi, x + 1);
            }
    }
    // links, in the reference's (y, x, i) order over solid cells
    for (int y = 0; y < L.ny; ++y)
        for (int x = -1; x <= L.lnx; ++x) {
            if (!h->h_mask[L.at(x + 1, y)]) continue;
            for (int i = 1; i < Q; ++i) {
                int fx = x - cxi(i), fy = y - cyi(i);
                if (h->periodic_y) fy = ((fy % L.ny) + L.ny) % L.ny;
                if (fx >= 0 && fx < L.lnx && fy >= 0 && fy < L.ny && !h->h_mask[L.at(fx + 1, fy)]) {
                    Link l;
                    l.off = (long long)i * L.plane + L.at(fx + 1, fy);
                    l.cx2 = 2 * cxi(i);
                    l.cy2 = 2 * cyi(i);
                    links.push_back(l);
                    if (h->aa) {
                        // the same link in the reversed layout (A[fluid][opp(i)]) and in the natural
                        // layout after an O-step, where the population has been pushed into the solid
                        // cell itself (through the reverse wrap if it crossed a periodic edge)
                        l.off = (long long)oppi(i) * L.plane + L.at(fx + 1, fy);
                        links_rev.push_back(l);
                        // (one periodic slab: through the reverse wrap; a slab interface: it sits in MY ghost column)
                        const int sx = (h->periodic_x && h->world == 1) ? ((x % L.lnx) + L.lnx) % L.lnx : x;
                        l.off = (long long)i * L.plane + L.at(sx + 1, y);
                        links_nat.push_back(l);
                    }
                }
            }
        }
    std::vector<AaFill> fills;
    if (h->aa) {
        // slots of fluid cells that no cell pushes into during an O-step
        for (int x = 0; x < L.lnx; ++x)
            for (int y = 0; y < L.ny; ++y) {
                if (h->h_mask[L.at(x + 1, y)]) continue;
                for (int i = 1; i < Q; ++i) {
                    const int nx_ = x - cxi(i), ny_ = y - cyi(i);
                    // (a slab interface is an open edge: the neighbouring GPU's cells push across it)
                    const bool out_x = (nx_ < 0 && !h->periodic_x && h->west < 0) || (nx_ >= L.lnx && !h->periodic_x && h->east < 0);
                    const bool out_y = !h->periodic_y && (ny_ < 0 || ny_ >= L.ny);
                    AaFill e;
                    e.off = (long long)i * L.plane + L.at(x + 1, y);
                    e.i = i;
                    if (out_y) e.kind = 2;                                  // S/N ghost rows and corners: eq(1,u_in,0)
                    else if (out_x) e.kind = 1;                             // W/E ghost columns: 0.0
                    else if (h->h_mask[L.at(nx_ + 1, ny_)]) e.kind = 0;     // solid neighbour: w
                    else continue;
                    fills.push_back(e);
                }
            }
    }
    cudaFree(h->d_ring); cudaFree(h->d_solids); cudaFree(h->d_links);
    cudaFree(h->d_fills); cudaFree(h->d_links_rev); cudaFree(h->d_links_nat);
    h->d_ring = nullptr; h->d_solids = nullptr; h->d_links = nullptr;
    h->d_fills = nullptr; h->d_links_rev = nullptr; h->d_links_nat = nullptr;
    cudaFree(h->d_cols);
    h->d_cols = nullptr;
    CU(h, cudaMalloc(&h->d_cols, sizeof(int4) * cols.size()));
    CU(h, cudaMemcpyAsync(h->d_cols, cols.data(), sizeof(int4) * cols.size(), cudaMemcpyHostToDevice, h->stream));
    if (h->aa && links_rev.size() != links.size())
        return fail(h, LBM_ERR_INVALID, "internal: link lists of the two buffer schemes disagree");
    h->n_fill = (int)fills.size();
    if (!fills.empty()) {
        CU(h, cudaMalloc(&h->d_fills, sizeof(AaFill) * fills.size()));
        CU(h, cudaMemcpyAsync(h->d_fills, fills.data(), sizeof(AaFill) * fills.size(), cudaMemcpyHostToDevice, h->stream));
    }
    if (!links_rev.empty()) {
        CU(h, cudaMalloc(&h->d_links_rev, sizeof(Link) * links_rev.size()));
        CU(h, cudaMalloc(&h->d_links_nat, sizeof(Link) * links_nat.size()));
        CU(h, cudaMemcpyAsync(h->d_links_rev, links_rev.data(), sizeof(Link) * links_rev.size(), cudaMemcpyHostToDevice, h->stream));
        CU(h, cudaMemcpyAsync(h->d_links_nat, links_nat.data(), sizeof(Link) * links_nat.size(), cudaMemcpyHostToDevice, h->stream));
    }
    h->n_ring = (int)ring.size();
    h->n_solid = (int)solids.size();
    h->n_links = (int)links.size();
    {
        // 2 = solid with eight solid neighbours: pulls nothing but w, is never checked, computed or stored
        // (every other kernel only asks "non-zero?")
        std::vector<unsigned char> m2 = h->h_mask;
        h->n_deep = 0;
        for (int gx = -Layout::XO + 1; gx < L.lnx + 1 + Layout::XO; ++gx)
            for (int y = 0; y < L.ny; ++y) {
                if (!h->h_mask[L.at(gx, y)]) continue;
                bool deep = true;
                for (int i = 1; i < Q && deep; ++i) deep = h->h_mask[L.at(gx - cxi(i), y - cyi(i))] != 0;
                if (deep) {
                    m2[L.at(gx, y)] = 2;
                    if (gx >= 1 && gx <= L.lnx) h->n_deep += 1;
                }
            }
        h->h_mask.swap(m2);
    }
    CU(h, cudaMemcpyAsync(h->d_mask, h->h_mask.data(), h->h_mask.size(), cudaMemcpyHostToDevice, h->stream));
    if (h->n_ring) {
        CU(h, cudaMalloc(&h->d_ring, sizeof(int2) * ring.size()));
        CU(h, cudaMemcpyAsync(h->d_ring, ring.data(), sizeof(int2) * ring.size(), cudaMemcpyHostToDevice, h->stream));
    }
    if (h->n_solid) {
        CU(h, cudaMalloc(&h->d_solids, sizeof(int2) * solids.size()));
        CU(h, cudaMemcpyAsync(h->d_solids, solids.data(), sizeof(int2) * solids.size(), cudaMemcpyHostToDevice, h->stream));
    }
    if (h->n_links) {
        CU(h, cudaMalloc(&h->d_links, sizeof(Link) * links.size()));
        CU(h, cudaMemcpyAsync(h->d_links, links.data(), sizeof(Link) * links.size(), cudaMemcpyHostToDevice, h->stream));
    }
    CU(h, cudaStreamSynchronize(h->stream));  // the host vectors die here
    return LBM_OK;
}

int drain_forces(lbm_handle h) {
    if (h->pending.empty()) return LBM_OK;
    std::vector<double> tmp(2 * FORCE_SLOTS);
    CU(h, cudaMemcpyAsync(tmp.data(), h->d_forces, sizeof(double) * 2 * FORCE_SLOTS, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    for (const auto& pd : h->pending) h->force_log.push_back({pd.t, tmp[2 * pd.slot], tmp[2 * pd.slot + 1]});
    h->pending.clear();
    return LBM_OK;
}

P2pArgs p2p_args(lbm_handle h, int dst_index, int seq) {
    P2pArgs x;
    x.peer_dst_west = h->west >= 0 ? h->peer_f[0][dst_index] : nullptr;
    x.peer_dst_east = h->east >= 0 ? h->peer_f[1][dst_index] : nullptr;
    x.my_flags = h->d_flags;
    x.west_flag = h->west >= 0 ? h->peer_flags[0] + 1 : nullptr;  // I am my west neighbour's east side
    x.east_flag = h->east >= 0 ? h->peer_flags[1] + 0 : nullptr;
    x.blocks_done = h->d_blocks_done;
    x.seq = seq;
    x.status = h->d_status;
    x.timeout_ns = h->halo_timeout_ns;
    return x;
}

// Everything in flight between the slabs has landed (peer stores of the neighbours' last edge
// kernels, or the NCCL exchange): observers of ghost columns call this first.
int join_halo(lbm_handle h) {
    if (h->west < 0 && h->east < 0) return LBM_OK;
    if (h->p2p) {
        if (h->edge_seq > 0) CU(h, launch_wait_halo(p2p_args(h, 0, h->edge_seq), h->stream));
    } else {
        CU(h, cudaStreamWaitEvent(h->stream, h->ev_comm, 0));
    }
    return LBM_OK;
}

// All slabs have reached this point and their streams are drained (an NCCL all-reduce as a barrier).
int slab_barrier(lbm_handle h) {
    if (!h->comm) return LBM_OK;
    CU(h, cudaStreamSynchronize(h->comm_stream));
    NC(h, nccl_api().AllReduce(h->d_red, h->d_red, 1, ncclDouble, ncclSum, h->comm, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    return LBM_OK;
}

// Exchange CUDA IPC handles of both population buffers and the flag words with the x-neighbours
// and map theirs.  Any failure on any rank leaves every rank on the NCCL path.
int setup_p2p(lbm_handle h) {
    struct Pack { cudaIpcMemHandle_t f0, f1, flags; char uuid[16]; };
    const NcclApi& N = nccl_api();
    bool ok = true;
    if (const char* v = std::getenv("LBM_B200_P2P")) ok = std::atoi(v) != 0;
    Pack mine{};
    if (cudaMalloc(&h->d_flags, 64 * sizeof(int)) != cudaSuccess || cudaMalloc(&h->d_blocks_done, sizeof(unsigned int)) != cudaSuccess)
        return fail(h, LBM_ERR_NOMEM, "cudaMalloc of the halo flags failed");
    CU(h, cudaMemsetAsync(h->d_flags, 0, 64 * sizeof(int), h->stream));
    CU(h, cudaMemsetAsync(h->d_blocks_done, 0, sizeof(unsigned int), h->stream));
    if (cudaMalloc(&h->d_status, sizeof(int)) != cudaSuccess) return fail(h, LBM_ERR_NOMEM, "cudaMalloc of the halo status word failed");
    CU(h, cudaMemsetAsync(h->d_status, 0, sizeof(int), h->stream));
    {
        cudaDeviceProp prop;
        CU(h, cudaGetDeviceProperties(&prop, h->device));
        std::memcpy(mine.uuid, prop.uuid.bytes, 16);
    }
    // (the in-place variant has ONE population buffer: it stands for both)
    ok = ok && cudaIpcGetMemHandle(&mine.f0, h->f[0]) == cudaSuccess &&
         cudaIpcGetMemHandle(&mine.f1, h->f[1] ? h->f[1] : h->f[0]) == cudaSuccess &&
         cudaIpcGetMemHandle(&mine.flags, h->d_flags) == cudaSuccess;
    cudaGetLastError();
    Pack* d_io = nullptr;  // [0] mine, [1] from west, [2] from east
    CU(h, cudaMalloc(&d_io, 3 * sizeof(Pack)));
    Pack got[3];
    {
        // (a lambda so that every early return below frees d_io)
        auto swap_packs = [&]() -> int {
            CU(h, cudaMemcpyAsync(d_io, &mine, sizeof(Pack), cudaMemcpyHostToDevice, h->stream));
            NC(h, N.GroupStart());
            if (h->east >= 0) {
                NC(h, N.Send(d_io, sizeof(Pack), ncclChar, h->east, h->comm, h->stream));
                NC(h, N.Recv(d_io + 2, sizeof(Pack), ncclChar, h->east, h->comm, h->stream));
            }
            if (h->west >= 0) {
                NC(h, N.Send(d_io, sizeof(Pack), ncclChar, h->west, h->comm, h->stream));
                NC(h, N.Recv(d_io + 1, sizeof(Pack), ncclChar, h->west, h->comm, h->stream));
            }
            NC(h, N.GroupEnd());
            CU(h, cudaMemcpyAsync(got, d_io, 3 * sizeof(Pack), cudaMemcpyDeviceToHost, h->stream));
            CU(h, cudaStreamSynchronize(h->stream));
            return LBM_OK;
        };
        const int rc = swap_packs();
        cudaFree(d_io);
        if (rc) return rc;
    }
    // Two slabs on ONE GPU would have their step kernels wait for each other inside the same device: progress
    // would hang on time-slicing between processes.  Such a job exchanges by NCCL.
    for (int side = 0; side < 2; ++side)
        if ((side == 0 ? h->west : h->east) >= 0 && std::memcmp(got[1 + side].uuid, mine.uuid, 16) == 0) ok = false;
    for (int side = 0; side < 2 && ok; ++side) {
        if ((side == 0 ? h->west : h->east) < 0) continue;
        const Pack& p = got[1 + side];
        const cudaIpcMemHandle_t* hs[3] = {&p.f0, &p.f1, &p.flags};
        for (int k = 0; k < 3 && ok; ++k) {
            if (k == 1 && h->aa) continue;  // the same allocation as k == 0: open it once
            ok = cudaIpcOpenMemHandle(&h->ipc_opened[side][k], *hs[k], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
        }
        if (ok) {
            h->peer_f[side][0] = static_cast<double*>(h->ipc_opened[side][0]);
            h->peer_f[side][1] = static_cast<double*>(h->aa ? h->ipc_opened[side][0] : h->ipc_opened[side][1]);
            h->peer_flags[side] = static_cast<int*>(h->ipc_opened[side][2]);
        }
    }
    cudaGetLastError();
    double agree = ok ? 1.0 : 0.0;  // all or nothing
    CU(h, cudaMemcpyAsync(h->d_red, &agree, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    NC(h, N.AllReduce(h->d_red, h->d_red, 1, ncclDouble, ncclMin, h->comm, h->stream));
    CU(h, cudaMemcpyAsync(&agree, h->d_red, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    h->p2p = agree > 0.5;
    if (h->aa && !h->p2p)
        return fail(h, LBM_ERR_INVALID, "LBM_FLAG_AA over several slabs exchanges through CUDA IPC peer memory, which is unavailable here");
    return LBM_OK;
}

void close_p2p(lbm_handle h) {
    for (int side = 0; side < 2; ++side)
        for (int k = 0; k < 3; ++k)
            if (h->ipc_opened[side][k]) {
                cudaIpcCloseMemHandle(h->ipc_opened[side][k]);
                h->ipc_opened[side][k] = nullptr;
            }
    cudaGetLastError();
}

// Halo exchange of the freshly written buffer: interior column lnx -> east neighbour's W ghost
// (populations 1,5,8 move in +x), interior column 1 -> west neighbour's E ghost (3,6,7).
// Rows 0..ny-1 only: ghost-row/corner entries keep the initial equilibrium as in the 1-rank
// reference.  A column of one population is contiguous, so there is no pack kernel.
int exchange(lbm_handle h, double* buf, cudaStream_t s) {
    if (h->world == 1 || (h->west < 0 && h->east < 0)) return LBM_OK;
    const NcclApi& N = nccl_api();
    const Layout& L = h->L;
    static const int to_east[3] = {1, 5, 8}, to_west[3] = {3, 6, 7};
    NC(h, N.GroupStart());
    // NCCL pairs the sends and receives between two ranks in issue order.  With two slabs and
    // periodic x the east and the west neighbour are the SAME rank: my east-going send has to meet
    // its receive "from the west", so every rank issues send-east, recv-west, send-west, recv-east.
    for (int k = 0; k < 3; ++k) {
        if (h->east >= 0) NC(h, N.Send(buf + to_east[k] * L.plane + L.at(L.lnx, 0), L.ny, ncclDouble, h->east, h->comm, s));
        if (h->west >= 0) NC(h, N.Recv(buf + to_east[k] * L.plane + L.at(0, 0), L.ny, ncclDouble, h->west, h->comm, s));
        if (h->west >= 0) NC(h, N.Send(buf + to_west[k] * L.plane + L.at(1, 0), L.ny, ncclDouble, h->west, h->comm, s));
        if (h->east >= 0) NC(h, N.Recv(buf + to_west[k] * L.plane + L.at(L.lnx + 1, 0), L.ny, ncclDouble, h->east, h->comm, s));
    }
    NC(h, N.GroupEnd());
    return LBM_OK;
}

// Leading entries of the solid list that the per-step fix-up must reset to w (see lbm_solver).
int solids_to_reset(lbm_handle h, bool steady, bool aa) {
    if (!steady) return h->n_solid;  // first iteration after initialise / upload: an uploaded state may hold anything
    return h->n_solid_loose + (aa ? h->n_solid_l1 : 0);
}

const Link* aa_links(lbm_handle h) {
    if (!h->cur_is_next) return h->d_links;  // fresh: f_next == f_current, natural addressing
    return h->aa_phase == 1 ? h->d_links_rev : h->d_links_nat;
}

// One reference iteration in the single-buffer variant: E-step from the natural layout, O-step
// from the reversed one (lbm_aa.cu).
int step_one_aa(lbm_handle h) {
    const Layout& L = h->L;
    const bool odd = h->aa_phase == 1;
    if (odd && (h->west >= 0 || h->east >= 0)) {  // x-slabs: the neighbours' edge columns of the E-step must be in my ghost columns
        int rc = join_halo(h);
        if (rc) return rc;
    }
    AaArgs a = aa_args(h, (!odd && !h->cur_is_next) ? 1 : 0);
    if (h->time_bulk && (h->iter % h->time_bulk) == 0) {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaEventRecord(e0, h->stream);
        CU(h, launch_aa_bulk(odd, a, h->stream));
        cudaEventRecord(e1, h->stream);
        h->bulk_events.push_back(e0);
        h->bulk_events.push_back(e1);
        h->bulk_timed_launches += 1;
        h->bulk_timed_cells += (long long)(a.x_end - a.x_begin) * (L.ny - (a.skip_rows ? 2 : 0)) - h->n_deep;
        h->bulk_timed_updates += (long long)(a.x_end - a.x_begin) * (L.ny - (a.skip_rows ? 2 : 0)) - h->n_deep;
    } else {
        CU(h, launch_aa_bulk(odd, a, h->stream));
    }
    const bool multi = h->west >= 0 || h->east >= 0;
    const bool wrap_x1 = h->periodic_x && h->world == 1;  // the wrap stays inside this GPU
    const int open_x = ((h->periodic_x || h->west >= 0) ? 1 : 0) | ((h->periodic_x || h->east >= 0) ? 2 : 0);
    if (!odd) {
        CU(h, launch_aa_fix_even(a, h->run_bc, h->d_ring, h->n_ring, h->d_solids, solids_to_reset(h, !a.first, true), h->stream));
        h->launches += 2;
        if (wrap_x1) { CU(h, launch_wrap(h->f[0], L, 1, 0, h->stream)); h->launches += 1; }
        if (multi) {
            // forward halo: my edge columns into the neighbours' ghost columns; their O-step waits for it
            h->edge_seq += 1;
            CU(h, launch_aa_halo(h->f[0], L, 0, 0, p2p_args(h, 0, h->edge_seq), h->stream));
            h->launches += 1;
        }
        if (h->periodic_y) {
            if (multi) { int rc = join_halo(h); if (rc) return rc; }  // the corners copy the ghost columns
            CU(h, launch_wrap(h->f[0], L, 0, 1, h->stream));
            h->launches += 1;
        }
    } else {
        // Constant fill last: across an open edge the reverse wrap / halo also carries what solid cells
        // pushed, and the fill must overwrite that.
        const bool wrap = wrap_x1 || h->periodic_y || multi;
        CU(h, launch_aa_fix_odd(a, h->run_bc, h->d_ring, h->n_ring, h->d_fills, wrap ? 0 : h->n_fill, h->d_ring_out, open_x,
                                h->periodic_y ? 1 : 0, h->stream));
        h->launches += 2;
        if (wrap) {
            if (wrap_x1 || h->periodic_y) {
                CU(h, launch_aa_unwrap(h->f[0], L, wrap_x1 ? 1 : 0, h->periodic_y ? 1 : 0, h->stream));
                h->launches += (wrap_x1 ? 1 : 0) + (h->periodic_y ? 1 : 0);
            }
            if (multi) {
                // reverse halo: what my cells pushed across a face goes into the neighbour's edge column; mine arrives
                // from the neighbours before the constants are filled in
                h->edge_seq += 1;
                CU(h, launch_aa_halo(h->f[0], L, 1, h->periodic_y ? 1 : 0, p2p_args(h, 0, h->edge_seq), h->stream));
                h->launches += 1;
                int rc = join_halo(h);
                if (rc) return rc;
            }
            CU(h, launch_aa_fix_odd(a, h->run_bc, h->d_ring, 0, h->d_fills, h->n_fill, h->d_ring_out, 0, 0, h->stream));
            h->launches += (h->n_fill ? 1 : 0);
        }
    }
    mark_run(h);
    h->aa_phase ^= 1;
    h->prev_is_next = h->cur_is_next;
    h->cur_is_next = true;
    h->fresh = false;
    h->macros_valid = false;
    if (h->p.output_frequency > 0 && h->iter % h->p.output_frequency == 0) {
        if ((int)h->pending.size() >= FORCE_SLOTS) {
            int rc = drain_forces(h);
            if (rc) return rc;
        }
        const int slot = (int)h->pending.size();
        CU(h, launch_forces(h->f[0], aa_links(h), h->n_links, h->d_forces + 2 * slot, h->stream, h->force_tree));
        h->launches += 1;
        h->pending.push_back({h->iter, slot});
    }
    h->iter += 1;
    return LBM_OK;
}


// ---- temporal blocking (variant BULK_TB) ---------------------------------------------------------
bool multi_slab(lbm_handle h) { return h->west >= 0 || h->east >= 0; }

// Ghost columns a slab interface keeps current: the deepest pass of the job.
int halo_width(lbm_handle h) { return h->tb_depth < 2 ? 2 : h->tb_depth; }

TbArgs tb_args(lbm_handle h, const double* src, double* dst, int bad_iter, int write) {
    TbArgs a{};
    a.src = src;
    a.dst = dst;
    a.L = h->L;
    a.tau_inv = 1.0 / h->p.tau;  // include/LBMSolver.h:85
    a.Fx = h->p.body_force_x;
    a.Fy = h->p.body_force_y;
    a.first_bad = h->d_first_bad;
    a.bad_iter = bad_iter;
    a.bc = h->run_bc;  // the rules of the iteration the first stage pulls
    a.mask = h->d_mask;
    a.mask_lo = h->mask_lo;
    a.mask_hi = h->mask_hi;
    a.mask_ylo = h->mask_ylo;
    a.mask_yhi = h->mask_yhi;
    a.west = h->west >= 0 ? TB_EDGE_HALO : (h->periodic_x ? TB_EDGE_WRAP : TB_EDGE_CONST);
    a.east = h->east >= 0 ? TB_EDGE_HALO : (h->periodic_x ? TB_EDGE_WRAP : TB_EDGE_CONST);
    a.periodic_y = h->periodic_y ? 1 : 0;
    a.pull = 1;
    a.write = write;
    a.halo_w = halo_width(h);
    return a;
}

int ensure_native_macros(lbm_handle h) {
    if (h->d_mrho) return LBM_OK;
    const size_t n = (size_t)h->L.lnx * h->L.ny * sizeof(double);
    CU(h, cudaMalloc(&h->d_mrho, n));
    CU(h, cudaMalloc(&h->d_mux, n));
    CU(h, cudaMalloc(&h->d_muy, n));
    return LBM_OK;
}

// The wide halo of a pass by NCCL (the fallback where CUDA IPC is unavailable): column lnx-1-d -> the east
// neighbour's ghost column gx = -d and column d -> the west neighbour's gx = lnx+1+d, the same populations the
// fused kernel stores (lbm_tb.cuh).  In stream order, after the kernel; the fallback does not overlap.
int exchange_wide(lbm_handle h, double* buf, cudaStream_t s) {
    if (!multi_slab(h)) return LBM_OK;
    const NcclApi& N = nccl_api();
    const Layout& L = h->L;
    static const int east_going[3] = {1, 5, 8}, still[3] = {0, 2, 4}, west_going[3] = {3, 6, 7};
    const int W = halo_width(h);
    NC(h, N.GroupStart());
    for (int d = 0; d < W; ++d)
        for (int g = 0; g < 3; ++g) {
            if (g == 1 && d > W - 2) continue;
            if (g == 2 && d > W - 3) continue;
            // group 0: the populations moving towards the receiver; 1: staying in the column; 2: moving away
            const int* to_e = g == 0 ? east_going : (g == 1 ? still : west_going);
            const int* to_w = g == 0 ? west_going : (g == 1 ? still : east_going);
            for (int k = 0; k < 3; ++k) {
                // issue order send-east, recv-west, send-west, recv-east: see exchange()
                if (h->east >= 0) NC(h, N.Send(buf + to_e[k] * L.plane + L.at(L.lnx - d, 0), L.ny, ncclDouble, h->east, h->comm, s));
                if (h->west >= 0) NC(h, N.Recv(buf + to_e[k] * L.plane + L.at(-d, 0), L.ny, ncclDouble, h->west, h->comm, s));
                if (h->west >= 0) NC(h, N.Send(buf + to_w[k] * L.plane + L.at(1 + d, 0), L.ny, ncclDouble, h->west, h->comm, s));
                if (h->east >= 0) NC(h, N.Recv(buf + to_w[k] * L.plane + L.at(L.lnx + 1 + d, 0), L.ny, ncclDouble, h->east, h->comm, s));
            }
        }
    NC(h, N.GroupEnd());
    return LBM_OK;
}

void record_bulk(lbm_handle h, cudaEvent_t e0, cudaEvent_t e1, long long cells, int depth) {
    h->bulk_events.push_back(e0);
    h->bulk_events.push_back(e1);
    h->bulk_timed_launches += 1;
    h->bulk_timed_cells += cells;
    h->bulk_timed_updates += cells * depth;
}

// `depth` reference iterations (include/LBMSolver.h:49-58) in ONE launch and one pass over HBM.
int step_tb(lbm_handle h, int depth, bool emit) {
    const Layout& L = h->L;
    const bool pull = h->cur_is_next;
    if (!pull && depth != 1) return fail(h, LBM_ERR_INVALID, "internal: the first iteration is a pass of depth 1");
    double* dst = h->f[h->cur ^ 1];
    TbArgs a = tb_args(h, h->f[h->cur], dst, h->iter - 1, 1);
    a.pull = pull ? 1 : 0;
    if (emit) {
        int rc = ensure_native_macros(h);
        if (rc) return rc;
        a.m_rho = h->d_mrho;
        a.m_ux = h->d_mux;
        a.m_uy = h->d_muy;
    }
    const bool multi = multi_slab(h);
    const bool fused = multi && h->p2p;
    if (fused) {
        h->edge_seq += 1;
        a.px = p2p_args(h, h->cur ^ 1, h->edge_seq);
    }
    if (h->time_bulk && (h->iter % h->time_bulk) < depth) {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaEventRecord(e0, h->stream);
        CU(h, launch_tb(depth, a, fused, h->stream));
        cudaEventRecord(e1, h->stream);
        record_bulk(h, e0, e1, (long long)L.lnx * L.ny - h->n_deep, depth);
    } else {
        CU(h, launch_tb(depth, a, fused, h->stream));
    }
    h->launches += 1;
    if (multi && !fused) {
        int rc = exchange_wide(h, dst, h->stream);
        if (rc) return rc;
    }
    if (!pull && h->n_solid) {
        // The buffer just read may hold anything in its solid cells (an uploaded f_current); it is the
        // next destination and solid cells are never stored: give them w once, now.
        StepArgs back = step_args(h, h->f[h->cur], h->f[h->cur], h->iter - 1, 1);
        CU(h, launch_fixup(false, back, h->bc, nullptr, 0, h->d_solids, h->n_solid, h->stream));
        h->launches += 1;
    }
    // The passes themselves address periodic edges by wrapped indices; the ghost copies are for the observers.
    if (h->periodic_x && h->world == 1) { CU(h, launch_wrap(dst, L, 1, 0, h->stream)); h->launches += 1; }
    if (h->periodic_y) {
        if (fused) {
            int rc = join_halo(h);
            if (rc) return rc;
        }
        CU(h, launch_wrap(dst, L, 0, 1, h->stream));
        h->launches += 1;
    }
    const int last = h->iter + depth - 1;  // the collision whose populations dst holds
    if (h->p.output_frequency > 0 && last % h->p.output_frequency == 0) {  // IOManager::record_forces, LBMSolver.h:52-54
        if ((int)h->pending.size() >= FORCE_SLOTS) {
            int rc = drain_forces(h);
            if (rc) return rc;
        }
        const int slot = (int)h->pending.size();
        CU(h, launch_forces(dst, h->d_links, h->n_links, h->d_forces + 2 * slot, h->stream, h->force_tree));
        h->launches += 1;
        h->pending.push_back({last, slot});
    }
    mark_run(h);
    h->cur ^= 1;
    h->prev_is_next = depth > 1 ? true : h->cur_is_next;
    h->cur_is_next = true;
    h->lag = depth;
    h->fresh = false;
    h->macros_valid = false;
    h->iter += depth;
    if (emit) h->macros_native_iter = h->iter;
    return LBM_OK;
}

// How many iterations the next pass covers: as deep as the job allows, but an iteration whose collision is an
// output step (forces are taken from ITS populations) must be the last one of its pass, and the first
// iteration after initialise / upload stands alone.  Pure: lbm_plan_passes exposes it to the CPU tests.
int plan_depth(int iter, int remaining, int of, int max_depth, bool cur_is_next) {
    if (!cur_is_next) return 1;
    int d = 1;
    while (d < max_depth && d < remaining && !(of > 0 && (iter + d - 1) % of == 0)) ++d;
    return d;
}

int next_depth(lbm_handle h, int remaining) {
    // A pass applies one set of boundary rules: after lbm_set_params changed u_in, the iteration that still owes the
    // old inlet rule is a pass of its own.
    if (h->run_bc.u_in != h->bc.u_in) return 1;
    return plan_depth(h->iter, remaining, h->p.output_frequency, h->tb_depth, h->cur_is_next);
}

// One reference iteration (include/LBMSolver.h:49-58) as kernel launches.
int step_one(lbm_handle h) {
    if (h->aa) return step_one_aa(h);
    const Layout& L = h->L;
    const bool pull = h->cur_is_next;
    double* dst = h->f[h->cur ^ 1];
    StepArgs a = step_args(h, h->f[h->cur], dst, h->iter - 1, 1);
    const bool multi = (h->west >= 0 || h->east >= 0);
    const bool split = multi && h->overlap && L.lnx >= 4;

    auto bulk = [&](int x0, int x1) -> cudaError_t {
        if (h->time_bulk && (h->iter % h->time_bulk) == 0) {
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0);
            cudaEventCreate(&e1);
            cudaEventRecord(e0, h->stream);
            cudaError_t r = launch_bulk(h->variant, pull, a, h->stream, x0, x1);
            cudaEventRecord(e1, h->stream);
            h->bulk_events.push_back(e0);
            h->bulk_events.push_back(e1);
            h->bulk_timed_launches += 1;
            h->bulk_timed_cells += (long long)(x1 - x0) * L.ny - h->n_deep;  // deep obstacle cells are skipped
            h->bulk_timed_updates += (long long)(x1 - x0) * L.ny - h->n_deep;
            return r;
        }
        return launch_bulk(h->variant, pull, a, h->stream, x0, x1);
    };

    if (split && h->p2p) {
        // Two launches, one stream, no NCCL call and no event -- the single-GPU chain.  The two slab-edge
        // columns are the FIRST blocks of the bulk launch: they wait for the neighbours' previous push (it
        // landed a whole kernel ago), compute, and store their face populations straight into the
        // neighbours' ghost columns over NVLink while the interior blocks run (k_bulk_vec2_p2p).
        // Odd ny / scalar variant: bulk over every column, then the same edge work inside the fix-up.
        h->edge_seq += 1;
        const P2pArgs px = p2p_args(h, h->cur ^ 1, h->edge_seq);
        const bool fused = bulk_p2p_supported(h->variant, a);
        if (!fused) {
            CU(h, bulk(0, L.lnx));
            CU(h, launch_fixup_p2p(pull, a, h->run_bc, h->d_ring + h->n_ring_edge, h->n_ring - h->n_ring_edge,
                                   h->d_solids, solids_to_reset(h, pull, false), h->d_mask,
                                   px, h->stream));
        } else {
            if (h->time_bulk && (h->iter % h->time_bulk) == 0) {
                cudaEvent_t e0, e1;
                cudaEventCreate(&e0);
                cudaEventCreate(&e1);
                cudaEventRecord(e0, h->stream);
                CU(h, launch_bulk_p2p(pull, a, h->run_bc, h->d_mask, px, h->stream));
                cudaEventRecord(e1, h->stream);
                h->bulk_events.push_back(e0);
                h->bulk_events.push_back(e1);
                h->bulk_timed_launches += 1;
                h->bulk_timed_cells += (long long)L.lnx * L.ny - h->n_deep;
                h->bulk_timed_updates += (long long)L.lnx * L.ny - h->n_deep;
            } else {
                CU(h, launch_bulk_p2p(pull, a, h->run_bc, h->d_mask, px, h->stream));
            }
            CU(h, launch_fixup(pull, a, h->run_bc, h->d_ring + h->n_ring_edge, h->n_ring - h->n_ring_edge,
                               h->d_solids, solids_to_reset(h, pull, false), h->stream));
        }
        h->launches += 2;
    } else if (split) {
        // The wire is never on the critical path, and the main stream stays one unbroken chain of
        // dependent launches (bulk -> fix-up -> edge -> bulk ...):
        //   main stream : interior columns of t, interior fix-up, [halo of t-1 landed?] edge columns of t
        //   comm stream : [edge columns of t done] halo exchange of t
        // Only the edge kernel reads ghost columns; it comes last, a whole interior kernel after the
        // exchange it depends on was issued, so its wait is satisfied long before it is reached.
        CU(h, bulk(1, L.lnx - 1));
        CU(h, launch_fixup(pull, a, h->run_bc, h->d_ring + h->n_ring_edge, h->n_ring - h->n_ring_edge,
                           h->d_solids, solids_to_reset(h, pull, false), h->stream));
        CU(h, cudaStreamWaitEvent(h->stream, h->ev_comm, 0));
        CU(h, launch_edge(pull, a, h->run_bc, h->d_mask, h->stream));
        CU(h, cudaEventRecord(h->ev_edge, h->stream));
        CU(h, cudaStreamWaitEvent(h->comm_stream, h->ev_edge, 0));
        int rc = exchange(h, dst, h->comm_stream);
        if (rc) return rc;
        CU(h, cudaEventRecord(h->ev_comm, h->comm_stream));
        h->launches += 3;
    } else {
        CU(h, bulk(0, L.lnx));
        CU(h, launch_fixup(pull, a, h->run_bc, h->d_ring, h->n_ring, h->d_solids, solids_to_reset(h, pull, false), h->stream));
        h->launches += 2;
        if (multi) {
            int rc = exchange(h, dst, h->stream);
            if (rc) return rc;
        }
    }
    if (!pull && h->n_solid) {
        // The buffer just read may hold anything in its solid cells (an uploaded f_current); it is the
        // next destination and the bulk kernels never store solid cells: give them w once, now.
        StepArgs back = a;
        back.dst = h->f[h->cur];
        CU(h, launch_fixup(false, back, h->bc, nullptr, 0, h->d_solids, h->n_solid, h->stream));
        h->launches += 1;
    }
    if (h->periodic_x && h->world == 1) { CU(h, launch_wrap(dst, L, 1, 0, h->stream)); h->launches += 1; }
    if (h->periodic_y) {
        // ghost columns must be final before the rows (corners) are wrapped
        if (split) {
            int rc = join_halo(h);
            if (rc) return rc;
        }
        CU(h, launch_wrap(dst, L, 0, 1, h->stream));
        h->launches += 1;
    }

    // IOManager::record_forces, include/LBMSolver.h:52-54: after collision, on output steps
    if (h->p.output_frequency > 0 && h->iter % h->p.output_frequency == 0) {
        if ((int)h->pending.size() >= FORCE_SLOTS) {
            int rc = drain_forces(h);
            if (rc) return rc;
        }
        const int slot = (int)h->pending.size();
        CU(h, launch_forces(dst, h->d_links, h->n_links, h->d_forces + 2 * slot, h->stream, h->force_tree));
        h->launches += 1;
        h->pending.push_back({h->iter, slot});
    }

    if (h->custom_pending > 0) {
        // into the buffer just written, never into the one just read: the observers of rho / u still rebuild the state
        // the last collision saw from it, and that state was streamed from the OLD values
        CU(h, launch_scatter(h->d_custom_off, h->d_custom_val, h->n_custom, dst, nullptr, h->stream));
        h->launches += 1;
        h->custom_pending -= 1;
    }
    mark_run(h);
    h->cur ^= 1;
    h->prev_is_next = h->cur_is_next;
    h->cur_is_next = true;
    h->lag = 1;
    h->fresh = false;
    h->macros_valid = false;
    h->iter += 1;
    return LBM_OK;
}

int ensure_macros(lbm_handle h) {
    if (h->macros_valid) return LBM_OK;
    const size_t n = (size_t)h->L.lnx * h->L.ny * sizeof(double);
    if (!h->d_rho) {
        CU(h, cudaMalloc(&h->d_rho, n));
        CU(h, cudaMalloc(&h->d_ux, n));
        CU(h, cudaMalloc(&h->d_uy, n));
    }
    if (h->snapshot_pending) CU(h, cudaStreamWaitEvent(h->stream, h->ev_snapshot, 0));
    { int rc_ = join_halo(h); if (rc_) return rc_; }
    if (h->aa) {
        CU(h, launch_aa_macros(aa_observe(h), h->d_rho, h->d_ux, h->d_uy, h->stream));
        h->launches += 1;
        h->macros_valid = true;
        return LBM_OK;
    }
    bool read_prev = false;  // the kernels below pull from the PREVIOUS buffer, ghost columns included
    if (h->macros_native_iter != h->iter && h->cur_is_next && h->lag > 1) {
        // The last pass covered several iterations and did not emit: its source buffer is still intact, so the
        // same pass once more, storing no population, emits the moments its last collision read.
        int rc = ensure_native_macros(h);
        if (rc) return rc;
        TbArgs a = tb_args(h, h->f[h->cur ^ 1], h->f[h->cur], h->iter - h->lag - 1, 0);
        a.tau_inv = h->run_tau_inv;  // (the pass ran with these even if lbm_set_params has replaced them since)
        a.Fx = h->run_Fx;
        a.Fy = h->run_Fy;
        a.first_bad = h->d_first_bad_all;  // (already judged by the pass itself; keep the verdict word untouched)
        a.m_rho = h->d_mrho;
        a.m_ux = h->d_mux;
        a.m_uy = h->d_muy;
        CU(h, launch_tb(h->lag, a, false, h->stream));
        h->launches += 1;
        h->macros_native_iter = h->iter;
        read_prev = true;
    }
    if (h->macros_native_iter == h->iter && h->cur_is_next) {
        CU(h, launch_macros_finish(observe_args(h), h->d_mrho, h->d_mux, h->d_muy, h->d_rho, h->d_ux, h->d_uy, h->stream));
    } else {
        CU(h, launch_macros(observe_args(h), h->d_rho, h->d_ux, h->d_uy, h->stream));
        read_prev = h->cur_is_next && h->prev_is_next;
    }
    h->launches += 1;
    h->macros_valid = true;
    if (read_prev && h->p2p && multi_slab(h)) {
        // A neighbour may start its next pass as soon as it has MY halo of the last one, and that pass stores
        // into the ghost columns of the buffer just read.  Nobody moves on before every slab has observed:
        // in a multi-slab job the observers of rho / u are collective calls (include/lbm_b200.h).
        return slab_barrier(h);
    }
    return LBM_OK;
}

int ensure_stage(lbm_handle h) {
    if (h->d_stage[0]) return LBM_OK;
    const size_t row_bytes = (size_t)(h->L.lnx + 2) * Q * sizeof(double);
    size_t rows = (size_t)(64u << 20) / row_bytes;  // ~64 MB per chunk
    rows = rows < 32 ? 32 : (rows / 32) * 32;
    if (rows > (size_t)((h->L.ny + 2 + 31) / 32) * 32) rows = (size_t)((h->L.ny + 2 + 31) / 32) * 32;
    h->stage_rows = (int)rows;
    for (int b = 0; b < 2; ++b) {
        CU(h, cudaMalloc(&h->d_stage[b], rows * row_bytes));
        CU(h, cudaEventCreateWithFlags(&h->ev_stage_copied[b], cudaEventDisableTiming));
        CU(h, cudaEventCreateWithFlags(&h->ev_stage_free[b], cudaEventDisableTiming));
    }
    return LBM_OK;
}

// Grid::check_stability of the CURRENT f_current (the last iteration's check), which the fused
// kernels would only see one launch later: a store-less pass of the same kernels.
int check_pending(lbm_handle h) {
    if (!h->cur_is_next) return LBM_OK;
    if (h->aa) {
        { int rc_ = join_halo(h); if (rc_) return rc_; }
        CU(h, launch_aa_check(aa_observe(h), h->d_first_bad, h->iter - 1, h->stream));
        h->launches += 1;
        return LBM_OK;
    }
    { int rc_ = join_halo(h); if (rc_) return rc_; }
    if (h->variant == BULK_TB && !h->custom_state) {
        TbArgs t = tb_args(h, h->f[h->cur], h->f[h->cur ^ 1], h->iter - 1, 0);
        t.tau_inv = h->run_tau_inv;
        t.Fx = h->run_Fx;
        t.Fy = h->run_Fy;
        CU(h, launch_tb(1, t, false, h->stream));
        h->launches += 1;
        return LBM_OK;
    }
    StepArgs a = step_args(h, h->f[h->cur], h->f[h->cur ^ 1], h->iter - 1, 0);
    a.tau_inv = h->run_tau_inv;
    a.Fx = h->run_Fx;
    a.Fy = h->run_Fy;
    a.forced = (a.Fx != 0.0 || a.Fy != 0.0) ? 1 : 0;
    CU(h, launch_bulk(BULK_VEC2, true, a, h->stream, 0, h->L.lnx));
    CU(h, launch_fixup(true, a, h->run_bc, h->d_ring, h->n_ring, nullptr, 0, h->stream));
    h->launches += 2;
    return LBM_OK;
}

// A halo wait that ran into its bound (lbm_device.cuh) leaves a mark in the slab's status word: from then on
// the results are void and every synchronising entry point says so instead of hanging.
int halo_status(lbm_handle h) {
    if (!h->d_status) return LBM_OK;
    if (!h->halo_failed) {
        int st = 0;
        CU(h, cudaMemcpyAsync(&st, h->d_status, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
        h->halo_failed = st != 0;
    }
    if (h->halo_failed)
        return fail(h, LBM_ERR_NCCL, "halo exchange timed out: a neighbouring slab stopped delivering (LBM_B200_HALO_TIMEOUT_MS)");
    return LBM_OK;
}

// The verdict of Grid::check_stability is global (MPI_Allreduce MIN, include/LBMGrid.h:315):
// with several slabs every rank gets the smallest failing timestep of any of them.
int read_first_bad(lbm_handle h, int* out) {
    int v = INT_MAX;
    const int* src = h->d_first_bad;
    { int rc_ = join_halo(h); if (rc_) return rc_; }  // edge kernels flag too
    { int rc_ = halo_status(h); if (rc_) return rc_; }  // (before the collective: a lost neighbour would never join it)
    if (h->comm) {
        NC(h, nccl_api().AllReduce(h->d_first_bad, h->d_first_bad_all, 1, ncclInt, ncclMin, h->comm, h->stream));
        src = h->d_first_bad_all;
    }
    CU(h, cudaMemcpyAsync(&v, src, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    *out = v;
    return halo_status(h);
}

int create_common(const lbm_params* p, int device, int rank, int world, const void* uid, lbm_handle* out) {
    if (!p || !out) return fail(nullptr, LBM_ERR_INVALID, "null argument");
    *out = nullptr;
    if (p->nx <= 0 || p->ny <= 0) return fail(nullptr, LBM_ERR_INVALID, "nx and ny must be positive");
    if (!(p->tau > 0.5)) return fail(nullptr, LBM_ERR_INVALID, "tau must exceed 0.5");
    if (world < 1 || rank < 0 || rank >= world) return fail(nullptr, LBM_ERR_INVALID, "bad rank/world");
    if (p->nx % world != 0)  // include/LBMGrid.h:358 requires divisibility too
        return fail(nullptr, LBM_ERR_INVALID, "nx must be divisible by the number of slabs");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, LBM_ERR_CUDA, std::string("no CUDA device: liblbm_b200 has no CPU path (") +
                                               cudaGetErrorString(e) + ")");
    if (device < 0 || device >= ndev) return fail(nullptr, LBM_ERR_INVALID, "device index out of range");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, LBM_ERR_CUDA, cudaGetErrorString(e));

    lbm_handle h = new lbm_solver();
    h->p = *p;
    h->device = device;
    h->rank = rank;
    h->world = world;
    h->periodic_x = (p->flags & LBM_FLAG_PERIODIC_X) != 0;
    h->periodic_y = (p->flags & LBM_FLAG_PERIODIC_Y) != 0;
    h->aa = (p->flags & LBM_FLAG_AA) != 0;
    const int lnx = p->nx / world;
    h->L = Layout::make(lnx, p->ny, p->nx, rank * lnx);
    // include/LBMConfig.h:61-65
    h->cyl_x = static_cast<int>(p->cylinder_x * p->nx);
    h->cyl_y = static_cast<int>(p->cylinder_y * p->ny);
    h->cyl_r = static_cast<int>(p->cylinder_radius * p->ny);
    h->bc.u_in = p->inlet_velocity;
    h->bc.inlet = (!h->periodic_x && rank == 0) ? 1 : 0;
    h->bc.outlet = (!h->periodic_x && rank == world - 1) ? 1 : 0;
    h->bc.walls = h->periodic_y ? 0 : 1;
    equilibrium_init(1.0, 0.0, 0.0, h->bc.w);
    equilibrium_init(1.0, p->inlet_velocity, 0.0, h->bc.e);
    h->init_u = p->inlet_velocity;
    if (const char* v = std::getenv("LBM_B200_VARIANT")) h->variant = std::atoi(v);
    if (const char* v = std::getenv("LBM_B200_OVERLAP")) h->overlap = std::atoi(v) != 0;
    if (const char* v = std::getenv("LBM_B200_COLSKIP")) h->col_skip = std::atoi(v) != 0;
    if (const char* v = std::getenv("LBM_B200_TB_DEPTH")) h->tb_depth = std::min(std::max(std::atoi(v), 1), (int)TB_MAX_DEPTH);
    if (const char* v = std::getenv("LBM_B200_HALO_TIMEOUT_MS")) h->halo_timeout_ns = (unsigned long long)std::atoll(v) * 1000000ull;
    if (h->variant < 0 || h->variant > BULK_TB) h->variant = BULK_TB;
    // default: temporal blocking where the slab is large enough to feed it (every slab of a job has the same shape)
    if (!std::getenv("LBM_B200_VARIANT") && !tb_worthwhile(h->L)) h->variant = BULK_VEC2;
    if (world > 1) {
        h->west = rank > 0 ? rank - 1 : (h->periodic_x ? world - 1 : -1);
        h->east = rank < world - 1 ? rank + 1 : (h->periodic_x ? 0 : -1);
    }

    auto bail = [&](int code, const std::string& m) {
        g_create_error = m;
        lbm_destroy(h);
        return code;
    };
#define CUC(expr)                                                                              \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return bail(e__ == cudaErrorMemoryAllocation ? LBM_ERR_NOMEM : LBM_ERR_CUDA,       \
                        std::string(#expr) + ": " + cudaGetErrorString(e__));                  \
    } while (0)
    int lo = 0, hi = 0;
    CUC(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CUC(cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, lo));
    CUC(cudaStreamCreateWithPriority(&h->copy_stream, cudaStreamNonBlocking, lo));
    CUC(cudaStreamCreateWithPriority(&h->comm_stream, cudaStreamNonBlocking, hi));
    CUC(cudaEventCreateWithFlags(&h->ev_macros, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&h->ev_snapshot, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&h->ev_edge, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&h->ev_comm, cudaEventDisableTiming));
    const size_t fbytes = (size_t)h->L.plane * Q * sizeof(double);
    CUC(cudaMalloc(&h->f[0], fbytes));
    CUC(cudaMemsetAsync(h->f[0], 0, fbytes, h->stream));
    if (h->aa) {
        h->f[1] = nullptr;  // the point of the variant: no second buffer
        const size_t rbytes = (size_t)(2 * h->L.ny + 2 * h->L.lnx) * Q * sizeof(double);
        CUC(cudaMalloc(&h->d_ring_out, rbytes));
        CUC(cudaMemsetAsync(h->d_ring_out, 0, rbytes, h->stream));
    } else {
        CUC(cudaMalloc(&h->f[1], fbytes));
        CUC(cudaMemsetAsync(h->f[1], 0, fbytes, h->stream));
    }
    h->h_mask.assign((size_t)h->L.cells_padded(), 0);
    CUC(cudaMalloc(&h->d_mask, h->h_mask.size()));
    CUC(cudaMemsetAsync(h->d_mask, 0, h->h_mask.size(), h->stream));
    CUC(cudaMalloc(&h->d_first_bad, sizeof(int)));
    CUC(cudaMalloc(&h->d_forces, sizeof(double) * 2 * FORCE_SLOTS));
    CUC(cudaMalloc(&h->d_maxbits, sizeof(unsigned long long)));
    CUC(cudaMalloc(&h->d_red, sizeof(double) * LBM_REDUCE_MAX));
    CUC(cudaMalloc(&h->d_first_bad_all, sizeof(int)));
    const int big = INT_MAX;
    CUC(cudaMemcpyAsync(h->d_first_bad, &big, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CUC(cudaStreamSynchronize(h->stream));
    CUC(cudaEventRecord(h->ev_comm, h->comm_stream));
    CUC(cudaEventRecord(h->ev_edge, h->comm_stream));
#undef CUC
    if (world > 1) {
        const NcclApi& N = nccl_api();
        if (!N.ok) return bail(LBM_ERR_NCCL, std::string("NCCL unavailable: ") + N.why);
        if (!uid) return bail(LBM_ERR_INVALID, "nccl_unique_id is required when world > 1");
        ncclUniqueId id;
        static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
        std::memcpy(&id, uid, sizeof(id));
        ncclResult_t r = N.CommInitRank(&h->comm, world, id, rank);
        if (r != ncclSuccess) return bail(LBM_ERR_NCCL, std::string("ncclCommInitRank: ") + N.GetErrorString(r));
        if (!g_id_file.empty()) {
            std::remove(g_id_file.c_str());
            g_id_file.clear();
        }
        if (h->west >= 0 || h->east >= 0) {
            int rc = setup_p2p(h);
            if (rc) {
                std::string m = h->err;
                return bail(rc, m);
            }
        }
    }
    // ring list etc. for an obstacle-free domain; lbm_setup_geometry adds the cylinder
    {
        const int keep = h->p.flags;
        h->p.flags |= LBM_FLAG_NO_CYLINDER;
        int rc = build_geometry(h);
        h->p.flags = keep;
        if (rc) {
            std::string m = h->err;
            return bail(rc, m);
        }
    }
    *out = h;
    return LBM_OK;
}

}  // namespace

// ============================================================================================
extern "C" {

int lbm_device_count(int* n) {
    if (!n) return LBM_ERR_INVALID;
    cudaError_t e = cudaGetDeviceCount(n);
    if (e != cudaSuccess) {
        *n = 0;
        return fail(nullptr, LBM_ERR_CUDA, cudaGetErrorString(e));
    }
    return LBM_OK;
}

int lbm_create(const lbm_params* p, int device, lbm_handle* out) { return create_common(p, device, 0, 1, nullptr, out); }

int lbm_create_slab(const lbm_params* p, int device, int rank, int world, const void* uid, lbm_handle* out) {
    return create_common(p, device, rank, world, uid, out);
}

int lbm_nccl_unique_id(void* out128) {
    if (!out128) return LBM_ERR_INVALID;
    const NcclApi& N = nccl_api();
    if (!N.ok) return fail(nullptr, LBM_ERR_NCCL, std::string("NCCL unavailable: ") + N.why);
    ncclUniqueId id;
    ncclResult_t r = N.GetUniqueId(&id);
    if (r != ncclSuccess) return fail(nullptr, LBM_ERR_NCCL, N.GetErrorString(r));
    std::memcpy(out128, &id, sizeof(id));
    return LBM_OK;
}

int lbm_destroy(lbm_handle h) {
    if (!h) return LBM_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm_stream) cudaStreamSynchronize(h->comm_stream);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    if (h->comm && h->p2p && !h->halo_failed) slab_barrier(h);  // no neighbour may still be storing into this slab's memory
    close_p2p(h);
    if (h->comm) nccl_api().CommDestroy(h->comm);
    for (cudaEvent_t e : h->bulk_events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->marks)
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_slot)
        if (e) cudaEventDestroy(e);
    for (int b = 0; b < 2; ++b) {
        if (h->ev_stage_copied[b]) cudaEventDestroy(h->ev_stage_copied[b]);
        if (h->ev_stage_free[b]) cudaEventDestroy(h->ev_stage_free[b]);
    }
    cudaFree(h->f[0]); cudaFree(h->f[1]); cudaFree(h->d_mask); cudaFree(h->d_ring); cudaFree(h->d_solids);
    cudaFree(h->d_links); cudaFree(h->d_rho); cudaFree(h->d_ux); cudaFree(h->d_uy); cudaFree(h->d_stage[0]); cudaFree(h->d_stage[1]);
    cudaFree(h->d_first_bad); cudaFree(h->d_forces); cudaFree(h->d_maxbits);
    cudaFree(h->d_red); cudaFree(h->d_gather); cudaFree(h->d_first_bad_all);
    cudaFree(h->d_flags); cudaFree(h->d_blocks_done); cudaFree(h->d_status);
    cudaFree(h->d_mrho); cudaFree(h->d_mux); cudaFree(h->d_muy); cudaFree(h->d_custom_off); cudaFree(h->d_custom_val);
    cudaFree(h->d_cols); cudaFree(h->d_fills); cudaFree(h->d_links_rev); cudaFree(h->d_links_nat); cudaFree(h->d_ring_out);
    if (h->ev_macros) cudaEventDestroy(h->ev_macros);
    if (h->ev_snapshot) cudaEventDestroy(h->ev_snapshot);
    if (h->ev_edge) cudaEventDestroy(h->ev_edge);
    if (h->ev_comm) cudaEventDestroy(h->ev_comm);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->comm_stream) cudaStreamDestroy(h->comm_stream);
    delete h;
    return LBM_OK;
}

const char* lbm_last_error(lbm_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int lbm_get_info(lbm_handle h, lbm_info* o) {
    CHECK_H(h);
    if (!o) return fail(h, LBM_ERR_INVALID, "null info");
    o->abi_version = LBM_B200_ABI_VERSION;
    o->global_nx = h->p.nx; o->global_ny = h->p.ny;
    o->local_nx = h->L.lnx; o->local_ny = h->L.ny;
    o->x_start = h->L.x_start; o->y_start = 0;
    o->rank = h->rank; o->world = h->world; o->device = h->device;
    o->cyl_x = h->cyl_x; o->cyl_y = h->cyl_y; o->cyl_r = h->cyl_r;
    o->solid_cells = h->n_solid; o->links = h->n_links; o->iteration = h->iter;
    o->bytes_per_buffer = (int64_t)h->L.plane * Q * (int64_t)sizeof(double);
    o->row_pitch = h->L.PY;
    o->kernel_variant = h->variant;
    o->halo_p2p = h->p2p ? 1 : 0;
    o->pass_depth = (h->variant == BULK_TB && !h->aa) ? h->tb_depth : 1;
    o->deep_solid_cells = (int32_t)h->n_deep;
    return LBM_OK;
}

int lbm_setup_geometry(lbm_handle h, int* solid_count) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = build_geometry(h);
    if (rc) return rc;
    if (solid_count) *solid_count = h->n_solid;
    // The buffers still hold the old geometry's state (a cell that became solid holds a different value in each):
    // the next step needs lbm_initialise or lbm_upload_f first.
    h->initialised = false;
    return LBM_OK;
}

int lbm_initialise(lbm_handle h, double inlet_u) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaStreamSynchronize(h->comm_stream));  // nothing of an earlier run may still touch the buffers
    CU(h, cudaStreamSynchronize(h->stream));
    if (h->p2p) {  // ... nor a neighbour's edge kernel (it stores into this slab's ghost columns)
        int rc = slab_barrier(h);
        if (rc) return rc;
    }
    h->init_u = inlet_u;
    equilibrium_init(1.0, inlet_u, 0.0, h->bc.e);
    const int wz = (!h->periodic_x && h->rank == 0) ? 1 : 0;
    const int ez = (!h->periodic_x && h->rank == h->world - 1) ? 1 : 0;
    const int sw = (h->p.flags & LBM_FLAG_SHEAR_WAVE_INIT) ? 1 : 0;
    CU(h, launch_init(h->f[0], h->aa ? h->f[0] : h->f[1], h->L, h->d_mask, h->bc, wz, ez, sw, inlet_u, h->stream));
    h->launches += 1;
    if (h->aa) {
        CU(h, launch_aa_ghosts(h->f[0], h->L, h->bc, wz, ez, h->stream));
        h->launches += 1;
        h->aa_phase = 0;
    }
    if (!h->aa && h->variant == BULK_TB) {  // (not in the middle of a run: cudaMalloc synchronises the device)
        int rc = ensure_native_macros(h);
        if (rc) return rc;
    }
    const int big = INT_MAX;
    CU(h, cudaMemcpyAsync(h->d_first_bad, &big, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    h->cur = 0;
    h->cur_is_next = false;
    h->prev_is_next = false;
    h->fresh = true;
    h->initialised = true;
    h->iter = 0;
    h->macros_valid = false;
    h->lag = 1;
    h->macros_native_iter = -1;
    h->custom_state = false;
    h->custom_pending = 0;
    mark_run(h);
    h->pending.clear();
    h->force_log.clear();
    if (h->p2p) return slab_barrier(h);  // every slab initialised before any neighbour pushes a halo into it
    return LBM_OK;
}

int lbm_step(lbm_handle h, int n_steps) {
    CHECK_H(h);
    if (!h->initialised) return fail(h, LBM_ERR_INVALID, "lbm_initialise or lbm_upload_f first");
    if (n_steps < 0) return fail(h, LBM_ERR_INVALID, "n_steps < 0");
    CU(h, cudaSetDevice(h->device));
    if (h->halo_failed) return halo_status(h);
    if (h->aa || h->variant != BULK_TB || h->custom_state) {
        for (int k = 0; k < n_steps; ++k) {
            int rc = step_one(h);
            if (rc) return rc;
        }
        return LBM_OK;
    }
    for (int k = 0; k < n_steps;) {
        const int d = next_depth(h, n_steps - k);
        // The caller of lbm_run looks at rho / u after the call (Solver::run: max_velocity and VTK after every output
        // step, and its chunks END on output steps): the last pass of such a call emits the moments of its last
        // collision (24 B per cell).  Anywhere else an observer re-runs the pass store-less (ensure_macros).
        const bool emit = h->emit_last && k + d == n_steps;
        int rc = step_tb(h, d, emit);
        if (rc) return rc;
        k += d;
    }
    return LBM_OK;
}

int lbm_sync(lbm_handle h) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaStreamSynchronize(h->comm_stream));
    CU(h, cudaStreamSynchronize(h->copy_stream));
    return halo_status(h);
}

int lbm_run(lbm_handle h, int n_steps, double* rows, int max_rows, int* n_rows, int* unstable_at) {
    CHECK_H(h);
    if (unstable_at) *unstable_at = -1;
    if (n_rows) *n_rows = 0;
    const int t0 = h->iter;
    const size_t log0 = h->force_log.size();
    int bad = INT_MAX;
    // Launch in chunks; look at the stability flag between chunks so that a blown-up run stops
    // within one chunk instead of grinding through NaNs for 120 000 steps.
    // Chunks END on output steps (as Solver::run's do), so that a temporally blocked pass never has to be cut
    // short in the middle of a chunk: an output iteration is the last one of its pass anyway.
    const int of = h->p.output_frequency;
    int done = 0;
    while (done < n_steps) {
        int n = 256;
        if (of > 0) {
            int end = ((h->iter + of - 1) / of) * of;  // the next output iteration (possibly this one) ...
            while (end - h->iter + 1 < 64) end += of;  // ... but at least 64 iterations between two looks at the flags
            n = end - h->iter + 1;
        }
        if (n > n_steps - done) n = n_steps - done;
        h->emit_last = (done + n == n_steps);
        int rc = lbm_step(h, n);
        h->emit_last = false;
        if (rc) return rc;
        done += n;
        rc = drain_forces(h);
        if (rc) return rc;
        rc = read_first_bad(h, &bad);
        if (rc) return rc;
        if (bad != INT_MAX) break;
    }
    if (bad == INT_MAX) {  // the last iteration's own check
        int rc = check_pending(h);
        if (rc) return rc;
        rc = read_first_bad(h, &bad);
        if (rc) return rc;
    }
    const int bad_iter = (bad == INT_MAX) ? -1 : bad;
    // rows the reference would have written: output steps t <= failing iteration
    int k = 0;
    const double D_ref = 2.0 * h->cyl_r;                                           // include/LBMIO.h:174
    const double q_ref = 0.5 * 1.0 * h->p.inlet_velocity * h->p.inlet_velocity * D_ref;  // :176
    for (size_t r = log0; r < h->force_log.size(); ++r) {
        const auto& fr = h->force_log[r];
        if (fr.t < t0) continue;
        if (bad_iter >= 0 && fr.t > bad_iter) break;
        if (rows && k < max_rows) {
            double* o = rows + 5 * (size_t)k;
            o[0] = fr.t; o[1] = fr.fx; o[2] = fr.fy;
            o[3] = (q_ref > 1e-12) ? fr.fx / q_ref : 0.0;  // :177-178
            o[4] = (q_ref > 1e-12) ? fr.fy / q_ref : 0.0;
        }
        ++k;
    }
    if (n_rows) *n_rows = k;
    if (unstable_at) *unstable_at = bad_iter;
    return LBM_OK;
}

int lbm_get_forces(lbm_handle h, double* fx, double* fy) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = drain_forces(h);
    if (rc) return rc;
    { int rc_ = join_halo(h); if (rc_) return rc_; }
    if (h->aa)
        CU(h, launch_forces(h->f[0], aa_links(h), h->n_links, h->d_forces, h->stream, h->force_tree));
    else
        CU(h, launch_forces(h->f[h->cur], h->d_links, h->n_links, h->d_forces, h->stream, h->force_tree));
    h->launches += 1;
    double v[2];
    CU(h, cudaMemcpyAsync(v, h->d_forces, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    if (fx) *fx = v[0];
    if (fy) *fy = v[1];
    return LBM_OK;
}

int lbm_check_stability(lbm_handle h, int* ok, int* first_bad_step) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = check_pending(h);
    if (rc) return rc;
    int bad = INT_MAX;
    rc = read_first_bad(h, &bad);
    if (rc) return rc;
    if (ok) *ok = (bad == INT_MAX) ? 1 : 0;
    if (first_bad_step) *first_bad_step = (bad == INT_MAX) ? -1 : bad;
    return LBM_OK;
}

int lbm_max_velocity(lbm_handle h, double* out) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = ensure_macros(h);
    if (rc) return rc;
    CU(h, launch_maxvel(h->d_ux, h->d_uy, (long long)h->L.lnx * h->L.ny, h->d_maxbits, h->stream));
    h->launches += 1;
    unsigned long long bits = 0;
    CU(h, cudaMemcpyAsync(&bits, h->d_maxbits, sizeof(bits), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    double m;
    std::memcpy(&m, &bits, sizeof(m));
    if (out) *out = std::sqrt(m);  // include/LBMGrid.h:343
    return LBM_OK;
}

int lbm_download_f(lbm_handle h, int which, double* aos) {
    CHECK_H(h);
    if (!aos || (which != LBM_F_CURRENT && which != LBM_F_NEXT)) return fail(h, LBM_ERR_INVALID, "bad argument");
    CU(h, cudaSetDevice(h->device));
    int rc = ensure_stage(h);
    if (rc) return rc;
    { int rc_ = join_halo(h); if (rc_) return rc_; }
    // chunk k: export kernel on the compute stream -> D2H on the copy stream, while the kernel of chunk k+1 runs
    const int tny = h->L.ny + 2;
    const size_t row_elems = (size_t)(h->L.lnx + 2) * Q;
    int k = 0;
    for (int row0 = 0; row0 < tny; row0 += h->stage_rows, ++k) {
        const int b = k & 1, rows = std::min(h->stage_rows, tny - row0);
        if (k >= 2) CU(h, cudaStreamWaitEvent(h->stream, h->ev_stage_free[b], 0));  // its last copy has left the buffer
        if (h->aa)
            CU(h, launch_aa_export(aa_observe(h), which, h->d_stage[b], row0, rows, h->stream));
        else
            CU(h, launch_export_f(observe_args(h), which, h->d_stage[b], row0, rows, h->stream));
        h->launches += 1;
        CU(h, cudaEventRecord(h->ev_stage_copied[b], h->stream));
        CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev_stage_copied[b], 0));
        CU(h, cudaMemcpyAsync(aos + (size_t)row0 * row_elems, h->d_stage[b], (size_t)rows * row_elems * sizeof(double),
                              cudaMemcpyDeviceToHost, h->copy_stream));
        CU(h, cudaEventRecord(h->ev_stage_free[b], h->copy_stream));
    }
    CU(h, cudaStreamSynchronize(h->copy_stream));
    CU(h, cudaStreamSynchronize(h->stream));
    return LBM_OK;
}

int lbm_download_macros(lbm_handle h, double* rho, double* ux, double* uy) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = ensure_macros(h);
    if (rc) return rc;
    const size_t n = (size_t)h->L.lnx * h->L.ny * sizeof(double);
    if (rho) CU(h, cudaMemcpyAsync(rho, h->d_rho, n, cudaMemcpyDeviceToHost, h->stream));
    if (ux) CU(h, cudaMemcpyAsync(ux, h->d_ux, n, cudaMemcpyDeviceToHost, h->stream));
    if (uy) CU(h, cudaMemcpyAsync(uy, h->d_uy, n, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    return LBM_OK;
}

int lbm_download_solid(lbm_handle h, unsigned char* mask) {
    CHECK_H(h);
    if (!mask) return fail(h, LBM_ERR_INVALID, "null mask");
    for (int y = 0; y < h->L.ny; ++y)
        for (int x = 0; x < h->L.lnx; ++x) mask[(size_t)y * h->L.lnx + x] = h->h_mask[h->L.at(x + 1, y)] ? 1 : 0;
    return LBM_OK;
}

int lbm_upload_f(lbm_handle h, const double* aos, int iteration) {
    CHECK_H(h);
    if (!aos || iteration < 0) return fail(h, LBM_ERR_INVALID, "bad argument");
    CU(h, cudaSetDevice(h->device));
    int rc = ensure_stage(h);
    if (rc) return rc;
    rc = drain_forces(h);
    if (rc) return rc;
    CU(h, cudaStreamSynchronize(h->comm_stream));
    if (h->p2p) {
        CU(h, cudaStreamSynchronize(h->stream));
        int rc2 = slab_barrier(h);
        if (rc2) return rc2;
    }
    // chunk k: H2D on the copy stream -> transpose kernel on the compute stream, while chunk k+1 is being copied
    h->cur = 0;
    {
        const int tny = h->L.ny + 2;
        const size_t row_elems = (size_t)(h->L.lnx + 2) * Q;
        CU(h, cudaStreamSynchronize(h->stream));
        int k = 0;
        for (int row0 = 0; row0 < tny; row0 += h->stage_rows, ++k) {
            const int b = k & 1, rows = std::min(h->stage_rows, tny - row0);
            if (k >= 2) CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev_stage_free[b], 0));  // its kernel has consumed the buffer
            CU(h, cudaMemcpyAsync(h->d_stage[b], aos + (size_t)row0 * row_elems, (size_t)rows * row_elems * sizeof(double),
                                  cudaMemcpyHostToDevice, h->copy_stream));
            CU(h, cudaEventRecord(h->ev_stage_copied[b], h->copy_stream));
            CU(h, cudaStreamWaitEvent(h->stream, h->ev_stage_copied[b], 0));
            CU(h, launch_import_f(h->d_stage[b], h->f[0], h->L, row0, rows, h->stream));
            CU(h, cudaEventRecord(h->ev_stage_free[b], h->stream));
            h->launches += 1;
        }
    }
    const int wz = (!h->periodic_x && h->rank == 0) ? 1 : 0;
    const int ez = (!h->periodic_x && h->rank == h->world - 1) ? 1 : 0;
    if (h->aa) {
        CU(h, launch_aa_ghosts(h->f[0], h->L, h->bc, wz, ez, h->stream));
        h->aa_phase = 0;
    } else {
        CU(h, launch_reset_ghosts(h->f[0], h->L, h->bc, wz, ez, h->stream));
        CU(h, launch_reset_ghosts(h->f[1], h->L, h->bc, wz, ez, h->stream));
    }
    h->launches += 2;
    const int big = INT_MAX;
    CU(h, cudaMemcpyAsync(h->d_first_bad, &big, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    h->cur_is_next = false;
    h->prev_is_next = false;
    h->fresh = false;
    h->initialised = true;
    h->iter = iteration;
    h->macros_valid = false;
    h->lag = 1;
    h->macros_native_iter = -1;
    // The ghost rows were just reset in both buffers, and the first step resets every solid cell: values the caller
    // wrote into f_next (lbm_upload_f_next) go into the destinations of the next two steps again.
    if (h->custom_state && h->n_custom) h->custom_pending = 2;
    mark_run(h);
    if (h->p2p) return slab_barrier(h);
    return LBM_OK;
}

int lbm_upload_f_next(lbm_handle h, const double* aos) {
    CHECK_H(h);
    if (!aos) return fail(h, LBM_ERR_INVALID, "null argument");
    if (!h->initialised) return fail(h, LBM_ERR_INVALID, "lbm_initialise or lbm_upload_f first");
    if (h->aa) return fail(h, LBM_ERR_INVALID, "the in-place variant keeps no separate f_next to write into");
    CU(h, cudaSetDevice(h->device));
    // What a write to f_next can mean at an iteration boundary of the reference (include/LBMSolver.h:48-64): its
    // streaming has already consumed f_next and the next collision overwrites every FLUID cell, so fluid values are
    // dead; the values of solid cells and of the S/N ghost rows live on -- the NEXT iteration's streaming, and every
    // later one, pulls them.  The engine's fused step still owes the streaming of the iteration just finished (it
    // must pull the OLD values), so the new ones go into the destination buffer of each of the next two steps (solid
    // cells and ghost rows are never stored by the kernels: from then on both buffers keep them).
    const Layout& L = h->L;
    const size_t tnx = (size_t)L.lnx + 2;
    std::vector<long long> off;
    std::vector<double> val;
    auto take = [&](int gx, int y) {
        const double* src = aos + ((size_t)(y + 1) * tnx + gx) * Q;
        for (int i = 0; i < Q; ++i) {
            off.push_back((long long)i * L.plane + L.at(gx, y));
            val.push_back(src[i]);
        }
    };
    for (int y = 0; y < L.ny; ++y)
        for (int gx = 1; gx <= L.lnx; ++gx)
            if (h->h_mask[L.at(gx, y)]) take(gx, y);
    if (!h->periodic_y)
        for (int gx = 0; gx < L.lnx + 2; ++gx) {
            take(gx, -1);
            take(gx, L.ny);
        }
    CU(h, cudaStreamSynchronize(h->stream));
    cudaFree(h->d_custom_off);
    cudaFree(h->d_custom_val);
    h->d_custom_off = nullptr;
    h->d_custom_val = nullptr;
    h->n_custom = (int)off.size();
    if (h->n_custom) {
        CU(h, cudaMalloc(&h->d_custom_off, off.size() * sizeof(long long)));
        CU(h, cudaMalloc(&h->d_custom_val, val.size() * sizeof(double)));
        CU(h, cudaMemcpy(h->d_custom_off, off.data(), off.size() * sizeof(long long), cudaMemcpyHostToDevice));
        CU(h, cudaMemcpy(h->d_custom_val, val.data(), val.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    h->custom_pending = h->n_custom > 0 ? 2 : 0;
    h->custom_state = true;
    return LBM_OK;
}

int lbm_snapshot_begin(lbm_handle h, double* rho, double* ux, double* uy) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = ensure_macros(h);
    if (rc) return rc;
    CU(h, cudaEventRecord(h->ev_macros, h->stream));
    CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev_macros, 0));
    const size_t n = (size_t)h->L.lnx * h->L.ny * sizeof(double);
    if (rho) CU(h, cudaMemcpyAsync(rho, h->d_rho, n, cudaMemcpyDeviceToHost, h->copy_stream));
    if (ux) CU(h, cudaMemcpyAsync(ux, h->d_ux, n, cudaMemcpyDeviceToHost, h->copy_stream));
    if (uy) CU(h, cudaMemcpyAsync(uy, h->d_uy, n, cudaMemcpyDeviceToHost, h->copy_stream));
    CU(h, cudaEventRecord(h->ev_snapshot, h->copy_stream));
    h->snapshot_pending = true;
    return LBM_OK;
}

int lbm_snapshot_begin_slot(lbm_handle h, int slot, double* rho, double* ux, double* uy) {
    CHECK_H(h);
    if (slot < 0 || slot >= LBM_SNAPSHOT_SLOTS) return fail(h, LBM_ERR_INVALID, "snapshot slot out of range");
    CU(h, cudaSetDevice(h->device));
    if (!h->ev_slot[slot]) CU(h, cudaEventCreateWithFlags(&h->ev_slot[slot], cudaEventDisableTiming));
    int rc = lbm_snapshot_begin(h, rho, ux, uy);
    if (rc) return rc;
    CU(h, cudaEventRecord(h->ev_slot[slot], h->copy_stream));
    return LBM_OK;
}

// The same into a wider host image: row y of this slab lands at rho + y*row_pitch (doubles), i.e. the caller passes
// the address of its slab's first column inside an image of the whole channel that several slabs fill side by side.
int lbm_snapshot_begin_slot2d(lbm_handle h, int slot, double* rho, double* ux, double* uy, size_t row_pitch) {
    CHECK_H(h);
    if (slot < 0 || slot >= LBM_SNAPSHOT_SLOTS) return fail(h, LBM_ERR_INVALID, "snapshot slot out of range");
    if (row_pitch < (size_t)h->L.lnx) return fail(h, LBM_ERR_INVALID, "row pitch smaller than the slab width");
    CU(h, cudaSetDevice(h->device));
    if (!h->ev_slot[slot]) CU(h, cudaEventCreateWithFlags(&h->ev_slot[slot], cudaEventDisableTiming));
    int rc = ensure_macros(h);
    if (rc) return rc;
    CU(h, cudaEventRecord(h->ev_macros, h->stream));
    CU(h, cudaStreamWaitEvent(h->copy_stream, h->ev_macros, 0));
    const size_t w = (size_t)h->L.lnx * sizeof(double), dp = row_pitch * sizeof(double);
    double* dst[3] = {rho, ux, uy};
    double* src[3] = {h->d_rho, h->d_ux, h->d_uy};
    for (int k = 0; k < 3; ++k)
        if (dst[k]) CU(h, cudaMemcpy2DAsync(dst[k], dp, src[k], w, w, h->L.ny, cudaMemcpyDeviceToHost, h->copy_stream));
    CU(h, cudaEventRecord(h->ev_snapshot, h->copy_stream));
    h->snapshot_pending = true;
    CU(h, cudaEventRecord(h->ev_slot[slot], h->copy_stream));
    return LBM_OK;
}

// Safe to call from a second host thread (an output writer): touches nothing but the event.
int lbm_snapshot_wait_slot(lbm_handle h, int slot) {
    CHECK_H(h);
    if (slot < 0 || slot >= LBM_SNAPSHOT_SLOTS || !h->ev_slot[slot]) return LBM_ERR_INVALID;
    cudaError_t e = cudaEventSynchronize(h->ev_slot[slot]);
    return e == cudaSuccess ? LBM_OK : LBM_ERR_CUDA;
}

int lbm_snapshot_wait(lbm_handle h) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    if (h->snapshot_pending) {
        CU(h, cudaEventSynchronize(h->ev_snapshot));
        h->snapshot_pending = false;
    }
    return LBM_OK;
}

int lbm_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return LBM_ERR_INVALID;
    cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(nullptr, e == cudaErrorMemoryAllocation ? LBM_ERR_NOMEM : LBM_ERR_CUDA, cudaGetErrorString(e));
    return LBM_OK;
}

int lbm_host_register(void* ptr, size_t bytes) {
    cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) return fail(nullptr, LBM_ERR_CUDA, cudaGetErrorString(e));
    return LBM_OK;
}

int lbm_host_unregister(void* ptr) {
    cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) return fail(nullptr, LBM_ERR_CUDA, cudaGetErrorString(e));
    return LBM_OK;
}

int lbm_host_free(void* ptr) {
    cudaError_t e = cudaFreeHost(ptr);
    if (e != cudaSuccess) return fail(nullptr, LBM_ERR_CUDA, cudaGetErrorString(e));
    return LBM_OK;
}

int lbm_time_steps(lbm_handle h, int n_steps, int per_kernel, float* ms_total, float* ms_bulk, int* launches) {
    CHECK_H(h);
    if (!h->initialised) return fail(h, LBM_ERR_INVALID, "lbm_initialise first");
    CU(h, cudaSetDevice(h->device));
    cudaEvent_t e0, e1;
    CU(h, cudaEventCreate(&e0));
    CU(h, cudaEventCreate(&e1));
    const long long l0 = h->launches;
    h->time_bulk = per_kernel > 0 ? per_kernel : 0;
    if (h->time_bulk) h->bulk_timed_launches = h->bulk_timed_cells = h->bulk_timed_updates = 0;
    CU(h, cudaStreamSynchronize(h->comm_stream));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaEventRecord(e0, h->stream));
    int rc = lbm_step(h, n_steps);
    h->time_bulk = 0;
    if (rc) return rc;
    { int rc_ = join_halo(h); if (rc_) return rc_; }
    CU(h, cudaEventRecord(e1, h->stream));
    CU(h, cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(h, cudaEventElapsedTime(&ms, e0, e1));
    if (ms_total) *ms_total = ms;
    float sum = 0.f;
    for (size_t k = 0; k + 1 < h->bulk_events.size(); k += 2) {
        float m = 0.f;
        cudaEventElapsedTime(&m, h->bulk_events[k], h->bulk_events[k + 1]);
        sum += m;
        cudaEventDestroy(h->bulk_events[k]);
        cudaEventDestroy(h->bulk_events[k + 1]);
    }
    h->bulk_events.clear();
    if (ms_bulk) *ms_bulk = sum;
    if (launches) *launches = (int)(h->launches - l0);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return LBM_OK;
}

int lbm_get_counters(lbm_handle h, long long* launches, long long* bulk_launches, long long* bulk_cells) {
    CHECK_H(h);
    if (launches) *launches = h->launches;
    if (bulk_launches) *bulk_launches = h->bulk_timed_launches;
    if (bulk_cells) *bulk_cells = h->bulk_timed_cells;
    return LBM_OK;
}

int lbm_get_bulk_updates(lbm_handle h, long long* updates) {
    CHECK_H(h);
    if (updates) *updates = h->bulk_timed_updates;
    return LBM_OK;
}

int lbm_plan_passes(int iteration, int n_steps, int output_frequency, int max_depth, int state_is_f_current, int* depths,
                    int max_passes) {
    if (n_steps < 0 || max_depth < 1 || max_depth > TB_MAX_DEPTH || (max_passes > 0 && !depths)) return LBM_ERR_INVALID;
    int n = 0;
    bool cur_is_next = state_is_f_current == 0;
    for (int k = 0; k < n_steps;) {
        const int d = plan_depth(iteration + k, n_steps - k, output_frequency, max_depth, cur_is_next);
        if (n < max_passes) depths[n] = d;
        ++n;
        k += d;
        cur_is_next = true;
    }
    return n;
}

int lbm_selftest_division(lbm_handle h, long long n, unsigned long long seed, long long* mismatches) {
    CHECK_H(h);
    if (!mismatches || n < 0) return fail(h, LBM_ERR_INVALID, "bad argument");
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaMemsetAsync(h->d_maxbits, 0, sizeof(unsigned long long), h->stream));
    CU(h, launch_selftest_div(seed, n, h->d_maxbits, h->stream));
    unsigned long long bad = 0;
    CU(h, cudaMemcpyAsync(&bad, h->d_maxbits, sizeof(bad), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    *mismatches = (long long)bad;
    return LBM_OK;
}

int lbm_set_force_mode(lbm_handle h, int mode) {
    CHECK_H(h);
    if (mode != LBM_FORCES_ORDERED && mode != LBM_FORCES_TREE) return fail(h, LBM_ERR_INVALID, "force mode must be 0 or 1");
    h->force_tree = mode;
    return LBM_OK;
}

int lbm_set_pass_depth(lbm_handle h, int depth) {
    CHECK_H(h);
    if (depth < 1 || depth > TB_MAX_DEPTH) return fail(h, LBM_ERR_INVALID, "pass depth must be 1, 2 or 3");
    if (depth != h->tb_depth && multi_slab(h) && h->initialised && h->cur_is_next)
        return fail(h, LBM_ERR_INVALID, "in a multi-slab job the pass depth can only change before the first iteration");
    h->tb_depth = depth;
    return LBM_OK;
}

int lbm_event_record(lbm_handle h, int slot) {
    CHECK_H(h);
    if (slot < 0 || slot >= LBM_EVENT_SLOTS) return fail(h, LBM_ERR_INVALID, "event slot out of range");
    CU(h, cudaSetDevice(h->device));
    if (!h->marks[slot]) CU(h, cudaEventCreate(&h->marks[slot]));
    // everything the handle has in flight on its side streams is ordered before the mark
    { int rc_ = join_halo(h); if (rc_) return rc_; }
    if (h->snapshot_pending) CU(h, cudaStreamWaitEvent(h->stream, h->ev_snapshot, 0));
    CU(h, cudaEventRecord(h->marks[slot], h->stream));
    return LBM_OK;
}

int lbm_event_elapsed(lbm_handle h, int slot_a, int slot_b, float* ms) {
    CHECK_H(h);
    if (slot_a < 0 || slot_a >= LBM_EVENT_SLOTS || slot_b < 0 || slot_b >= LBM_EVENT_SLOTS || !ms ||
        !h->marks[slot_a] || !h->marks[slot_b])
        return fail(h, LBM_ERR_INVALID, "bad event slots");
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaEventSynchronize(h->marks[slot_b]));
    CU(h, cudaEventElapsedTime(ms, h->marks[slot_a], h->marks[slot_b]));
    return LBM_OK;
}

// ---- multi-slab plumbing -------------------------------------------------------------------
namespace {
const char* env_first(std::initializer_list<const char*> names) {
    for (const char* n : names)
        if (const char* v = std::getenv(n)) return v;
    return nullptr;
}
}  // namespace

int lbm_bootstrap_env(int* rank, int* world, int* local_rank, void* id128) {
    // torchrun: RANK / WORLD_SIZE / LOCAL_RANK.  mpirun or srun used purely as a process launcher:
    // the usual OMPI_ / PMI_ / SLURM_ variables.  No launcher: one slab.
    const char* r = env_first({"LBM_B200_RANK", "RANK", "OMPI_COMM_WORLD_RANK", "PMI_RANK", "SLURM_PROCID"});
    const char* w = env_first({"LBM_B200_WORLD", "WORLD_SIZE", "OMPI_COMM_WORLD_SIZE", "PMI_SIZE", "SLURM_NTASKS"});
    const char* l = env_first({"LBM_B200_LOCAL_RANK", "LOCAL_RANK", "OMPI_COMM_WORLD_LOCAL_RANK", "MPI_LOCALRANKID", "SLURM_LOCALID"});
    const int wr = w ? std::atoi(w) : 1;
    const int rr = (r && wr > 1) ? std::atoi(r) : 0;
    if (wr < 1 || rr < 0 || rr >= wr) return fail(nullptr, LBM_ERR_INVALID, "inconsistent RANK / WORLD_SIZE in the environment");
    if (rank) *rank = rr;
    if (world) *world = wr;
    if (local_rank) *local_rank = (l && wr > 1) ? std::atoi(l) : rr;
    if (wr == 1 || !id128) return LBM_OK;
    // The 128-byte NCCL id travels through a file that only ranks of this launch agree on: all
    // ranks are children of one launcher process, so its pid names the file.
    char path[512];
    if (const char* f = std::getenv("LBM_B200_ID_FILE"))
        std::snprintf(path, sizeof(path), "%s", f);
    else
        std::snprintf(path, sizeof(path), "/tmp/lbm_b200_nccl_%ld_%s.id", (long)getppid(),
                      std::getenv("MASTER_PORT") ? std::getenv("MASTER_PORT") : "0");
    // File format: 8 bytes magic, 8 bytes launch stamp, 128 bytes id.  The stamp is the launcher's start time where
    // the launcher exports one (TORCHELASTIC_RUN_ID / SLURM_JOB_ID / the parent's pid as a last resort), so that a file
    // left behind by an earlier launch with the same parent pid and port is never taken for this launch's.
    unsigned long long stamp = 1469598103934665603ULL;
    for (const char* name : {"TORCHELASTIC_RUN_ID", "SLURM_JOB_ID", "LBM_B200_LAUNCH_ID"})
        if (const char* v = std::getenv(name))
            for (const char* c = v; *c; ++c) stamp = (stamp ^ (unsigned char)*c) * 1099511628211ULL;
    stamp ^= (unsigned long long)getppid() * 0x9E3779B97F4A7C15ULL;
    const unsigned long long magic = 0x4c424d4e43434c49ULL;
    if (rr == 0) {
        int rc = lbm_nccl_unique_id(id128);
        if (rc) return rc;
        // created exclusively, owner-only, under a private temporary name (a pre-created file or symlink at that name
        // makes the open fail instead of being followed), then renamed into place
        std::string tmp = std::string(path) + "." + std::to_string((long)getpid()) + ".tmp";
        unlink(tmp.c_str());
        unlink(path);  // a stale file of an earlier launch
        const int fd = open(tmp.c_str(), O_WRONLY | O_CREAT | O_EXCL | O_NOFOLLOW, 0600);
        bool ok = fd >= 0;
        ok = ok && write(fd, &magic, 8) == 8 && write(fd, &stamp, 8) == 8 && write(fd, id128, 128) == 128;
        if (fd >= 0) close(fd);
        if (!ok) {
            unlink(tmp.c_str());
            return fail(nullptr, LBM_ERR_IO, std::string("cannot write ") + tmp);
        }
        if (std::rename(tmp.c_str(), path) != 0) return fail(nullptr, LBM_ERR_IO, std::string("cannot rename to ") + path);
        g_id_file = path;  // removed once every rank has joined the communicator (create_common)
        return LBM_OK;
    }
    for (int tries = 0; tries < 6000; ++tries) {  // up to 60 s
        const int fd = open(path, O_RDONLY | O_NOFOLLOW);
        if (fd >= 0) {
            unsigned long long head[2] = {0, 0};
            const bool ok = read(fd, head, 16) == 16 && head[0] == magic && head[1] == stamp && read(fd, id128, 128) == 128;
            close(fd);
            if (ok) return LBM_OK;
        }
        usleep(10000);
    }
    return fail(nullptr, LBM_ERR_IO, std::string("timed out waiting for ") + path);
}

int lbm_set_params(lbm_handle h, const lbm_params* p) {
    CHECK_H(h);
    if (!p) return fail(h, LBM_ERR_INVALID, "null params");
    if (p->nx != h->p.nx || p->ny != h->p.ny) return fail(h, LBM_ERR_INVALID, "nx / ny are fixed at creation");
    if (!(p->tau > 0.5)) return fail(h, LBM_ERR_INVALID, "tau must exceed 0.5");
    if (((p->flags ^ h->p.flags) & (LBM_FLAG_PERIODIC_X | LBM_FLAG_PERIODIC_Y | LBM_FLAG_AA)) != 0)
        return fail(h, LBM_ERR_INVALID, "periodicity and the buffer scheme are fixed at creation");
    h->p = *p;
    h->cyl_x = static_cast<int>(p->cylinder_x * p->nx);
    h->cyl_y = static_cast<int>(p->cylinder_y * p->ny);
    h->cyl_r = static_cast<int>(p->cylinder_radius * p->ny);
    h->bc.u_in = p->inlet_velocity;
    return LBM_OK;
}

int lbm_allreduce(lbm_handle h, double* v, int n, int op) {
    CHECK_H(h);
    if (!v || n < 0 || n > LBM_REDUCE_MAX || op < LBM_SUM || op > LBM_MAX) return fail(h, LBM_ERR_INVALID, "bad argument");
    if (!h->comm || n == 0) return LBM_OK;  // one slab: the local value is the global one
    CU(h, cudaSetDevice(h->device));
    const ncclRedOp_t o = op == LBM_SUM ? ncclSum : (op == LBM_MIN ? ncclMin : ncclMax);
    CU(h, cudaMemcpyAsync(h->d_red, v, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    NC(h, nccl_api().AllReduce(h->d_red, h->d_red, n, ncclDouble, o, h->comm, h->stream));
    CU(h, cudaMemcpyAsync(v, h->d_red, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    return LBM_OK;
}

int lbm_gather_macros(lbm_handle h, double* rho, double* ux, double* uy) {
    CHECK_H(h);
    CU(h, cudaSetDevice(h->device));
    int rc = ensure_macros(h);
    if (rc) return rc;
    const Layout& L = h->L;
    const size_t slab = (size_t)L.lnx * L.ny;
    double* host[3] = {rho, ux, uy};
    double* dev[3] = {h->d_rho, h->d_ux, h->d_uy};
    if (h->world == 1) return lbm_download_macros(h, rho, ux, uy);
    const NcclApi& N = nccl_api();
    if (h->rank != 0) {
        for (int k = 0; k < 3; ++k) NC(h, N.Send(dev[k], slab, ncclDouble, 0, h->comm, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
        return LBM_OK;
    }
    if (!rho || !ux || !uy) return fail(h, LBM_ERR_INVALID, "rank 0 needs all three output arrays");
    if (!h->d_gather) CU(h, cudaMalloc(&h->d_gather, slab * sizeof(double)));
    const size_t dpitch = (size_t)L.gnx * sizeof(double), spitch = (size_t)L.lnx * sizeof(double);
    for (int k = 0; k < 3; ++k)  // own slab: rows of lnx doubles into rows of gnx
        CU(h, cudaMemcpy2DAsync(host[k], dpitch, dev[k], spitch, spitch, L.ny, cudaMemcpyDeviceToHost, h->stream));
    for (int r = 1; r < h->world; ++r)
        for (int k = 0; k < 3; ++k) {
            NC(h, N.Recv(h->d_gather, slab, ncclDouble, r, h->comm, h->stream));
            CU(h, cudaMemcpy2DAsync(host[k] + (size_t)r * L.lnx, dpitch, h->d_gather, spitch, spitch, L.ny,
                                    cudaMemcpyDeviceToHost, h->stream));
        }
    CU(h, cudaStreamSynchronize(h->stream));
    return LBM_OK;
}

int lbm_set_kernel_variant(lbm_handle h, int variant) {
    CHECK_H(h);
    if (variant < 0 || variant > BULK_TB) return fail(h, LBM_ERR_INVALID, "variant must be 0, 1 or 2");
    if (variant != h->variant && multi_slab(h) && h->initialised && h->cur_is_next)
        return fail(h, LBM_ERR_INVALID, "in a multi-slab job the kernel variant can only change before the first iteration "
                                        "(the temporally blocked passes keep a wider halo current)");
    h->variant = variant;
    return LBM_OK;
}

}  // extern "C"
