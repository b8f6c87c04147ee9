// oracle/prototypes/tb_emul.cpp -- thread-for-thread HOST emulation of the temporally blocked kernel.
// TEST INFRASTRUCTURE (tests/test_tb_emulation.py); never linked into the product.
//
// The thread program of the sm_100a kernel k_tb (csrc/lbm_tb.cuh: tb_thread<T, B, FORCED>) is a
// __host__ __device__ template.  Here every CUDA thread of every block becomes a std::thread, __syncthreads
// a std::barrier, shared memory a heap array, the SoA slab buffers host arrays in the device Layout, and
// the neighbouring GPUs' ghost columns plain pointers into the other slabs' buffers.  What this pins on
// the CPU, before any GPU time is spent, is the bookkeeping of the scheme: ring slots, row / column
// overlap, the boundary rules inside the stages, ghost constants, solid cells, the wide halo between
// slabs and the chunking -- the result must equal the oracle's single steps bit for bit.
#include <barrier>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "../../highperformancecomputing-latticeboltzmannmethod_b200/csrc/lbm_tb.cuh"

namespace lbm {
namespace {
thread_local std::barrier<>* g_barrier = nullptr;
std::mutex g_flag_mutex;
long long g_steps[2] = {0, 0};
}  // namespace
void tb_host_count(int which, int n) {
    std::lock_guard<std::mutex> lock(g_flag_mutex);
    g_steps[which] += n;
}
void tb_host_sync() { g_barrier->arrive_and_wait(); }
void tb_host_flag(int* p, int v) {
    std::lock_guard<std::mutex> lock(g_flag_mutex);
    if (v < *p) *p = v;
}
}  // namespace lbm

using namespace lbm;

namespace {

bool g_skew = true;  // which march (lbm_tb.cuh) the emulation runs; tb_set_skew
int g_fast = 1;      // ... and whether the skewed march takes its fast lane
bool g_fused = false;  // ... with the stages T..2 fused (k_tb<..., FUSED = true>)
double g_force[2] = {0.0, 0.0};  // tb_set_force: a body force selects the FORCED = true thread program
double* g_sink[3] = {nullptr, nullptr, nullptr};  // tb_set_macro_sink

struct Slab {
    Layout L;
    std::vector<double> f[2];
    std::vector<unsigned char> mask;
    int cur = 0;
};

// The padded columns [lo, hi) that hold solid cells, as the engine's build_geometry hands them to the kernels
// (an empty range when there is none): outside it the march skips the mask and may take its fast lane.
void mask_range(const Slab& s, TbArgs& a) {
    const Layout& L = s.L;
    a.mask_lo = L.lnx + 2 + Layout::XO;
    a.mask_hi = -Layout::XO;
    a.mask_ylo = L.ny + 1;
    a.mask_yhi = -1;
    for (int gx = -Layout::XO; gx < L.lnx + 2 + Layout::XO; ++gx)
        for (int y = -1; y <= L.ny; ++y)
            if (s.mask[L.at(gx, y)]) {
                a.mask_lo = gx < a.mask_lo ? gx : a.mask_lo;
                a.mask_hi = gx + 1 > a.mask_hi ? gx + 1 : a.mask_hi;
                a.mask_ylo = y < a.mask_ylo ? y : a.mask_ylo;
                a.mask_yhi = y + 1 > a.mask_yhi ? y + 1 : a.mask_yhi;
            }
}

// k_wrap of the engine: periodic edges keep wrapped copies in the ghost ring (x first, then y with the ghost
// columns, so that the corners come out right).
void wrap_ghosts(Slab& s, bool wrap_x, bool wrap_y) {
    const Layout& L = s.L;
    double* f = s.f[s.cur].data();
    for (int i = 0; i < Q; ++i) {
        double* p = f + i * L.plane;
        if (wrap_x)
            for (int y = 0; y < L.ny; ++y) {
                p[L.at(0, y)] = p[L.at(L.lnx, y)];
                p[L.at(L.lnx + 1, y)] = p[L.at(1, y)];
            }
        if (wrap_y)
            for (int gx = 0; gx < L.lnx + 2; ++gx) {
                p[L.at(gx, -1)] = p[L.at(gx, L.ny - 1)];
                p[L.at(gx, L.ny)] = p[L.at(gx, 0)];
            }
    }
}

template <int T, int B>
void run_blocks(const TbArgs& a, int chunks) {
    using S = TbShape<T, B>;
    const int strips = (a.L.ny + S::H - 1) / S::H;
    std::vector<double> ring((size_t)S::RING_DOUBLES + 1);
    for (int chunk = 0; chunk < chunks; ++chunk)
        for (int strip = 0; strip < strips; ++strip) {
            std::barrier<> bar(B);
            std::vector<std::thread> th;
            for (int tid = 0; tid < B; ++tid)
                th.emplace_back([&, tid] {
                    g_barrier = &bar;
                    // forced: the instantiation launch_forced (lbm_tb.cu) runs whatever the march settings
                    if (g_force[0] != 0.0 || g_force[1] != 0.0) tb_thread<T, B, true>(a, ring.data(), tid, strip, chunk);
                    else if (g_skew && g_fused) tb_thread<T, B, false, true, true>(a, ring.data(), tid, strip, chunk);
                    else if (g_skew) tb_thread<T, B, false, true>(a, ring.data(), tid, strip, chunk);
                    else tb_thread<T, B, false, false>(a, ring.data(), tid, strip, chunk);
                });
            for (auto& t : th) t.join();
        }
}

template <int B>
void run_pass_b(int depth, const TbArgs& a, int chunks) {
    if (depth == 1) run_blocks<1, B>(a, chunks);
    if (depth == 2) run_blocks<2, B>(a, chunks);
    if (depth == 3) run_blocks<3, B>(a, chunks);
}

// B = 16 and 32 keep the emulated lattices small; 64 and 128 are block heights the device runs (128 the default).
void run_pass(int depth, int B, const TbArgs& a, int chunks) {
    if (B == 16) run_pass_b<16>(depth, a, chunks);
    else if (B == 64) run_pass_b<64>(depth, a, chunks);
    else if (B == 128) run_pass_b<128>(depth, a, chunks);
    else run_pass_b<32>(depth, a, chunks);
}

// One slab of the global state in the device Layout, both buffers, the mask with its deep flag (see tb_emulate for
// the conventions: NaN wherever the kernel must never read).
void init_slab(Slab& s, int r, int world, const double* state, const unsigned char* solid, int nx, int ny, const BcArgs& bc0,
               bool per_x, bool per_y, int halo_w, int first_is_current) {
    const int lnx = nx / world;
    auto g_at = [&](int gx, int gy) { return ((size_t)gy * (nx + 2) + gx) * Q; };
    const double nan = std::numeric_limits<double>::quiet_NaN();
        s.L = Layout::make(lnx, ny, nx, r * lnx);
        for (int b = 0; b < 2; ++b) s.f[b].assign((size_t)s.L.plane * Q, nan);
        s.mask.assign((size_t)s.L.cells_padded(), 0);
        for (int gx = -Layout::XO; gx < lnx + 2 + Layout::XO; ++gx)
            for (int y = -1; y <= ny; ++y) {
                int X = r * lnx + gx;  // global padded column
                int Y = y + 1;
                if (per_x) X = tb_wrap(X - 1, nx) + 1;
                if (per_y) Y = tb_wrap(Y - 1, ny) + 1;
                const bool inside = X >= 0 && X < nx + 2;
                s.mask[s.L.at(gx, y)] = inside ? solid[(size_t)Y * (nx + 2) + X] : 0;
                const bool ghost = gx < 1 || gx > lnx || y < 0 || y >= ny;
                const bool iface_w = gx <= 0 && (r > 0 || (per_x && world > 1));
                const bool iface_e = gx >= lnx + 1 && (r < world - 1 || (per_x && world > 1));
                for (int i = 0; i < Q; ++i) {
                    double v0 = nan, v1 = nan;  // NaN = "the kernel must never read this"
                    if (!ghost) {
                        v0 = state[g_at(X, Y) + i];
                    } else if ((y < 0 || y >= ny) && !per_y) {
                        v0 = v1 = bc0.e[i];  // S/N ghost rows and corners keep the initial equilibrium (F4)
                    } else if ((iface_w || iface_e) && y >= 0 && y < ny) {
                        // ghost columns at a slab interface: only the populations the neighbour stores are defined
                        const int d = iface_w ? -gx : gx - (lnx + 1);  // 0 .. XO
                        const bool inward = iface_w ? (i == 1 || i == 5 || i == 8) : (i == 3 || i == 6 || i == 7);
                        const bool still = (i == 0 || i == 2 || i == 4), outward = !inward && !still;
                        if (!first_is_current && d < halo_w && (inward || (still && d <= halo_w - 2) || (outward && d <= halo_w - 3)))
                            v0 = state[g_at(X, Y) + i];
                    } else if (!per_x && (gx < 1 || gx > lnx) && y >= 0 && y < ny) {
                        v0 = v1 = 0.0;  // W/E ghost columns at the physical inlet / outlet (F4)
                    }
                    s.f[0][i * s.L.plane + s.L.at(gx, y)] = v0;
                    s.f[1][i * s.L.plane + s.L.at(gx, y)] = v1;
                }
            }
        // deep flag: solid with eight solid neighbours
        std::vector<unsigned char> m2 = s.mask;
        for (int gx = -Layout::XO + 1; gx < lnx + 1 + Layout::XO; ++gx)
            for (int y = 0; y < ny; ++y) {
                if (!s.mask[s.L.at(gx, y)]) continue;
                bool deep = true;
                for (int i = 1; i < Q; ++i) deep = deep && s.mask[s.L.at(gx - cxi(i), y - cyi(i))];
                if (deep) m2[s.L.at(gx, y)] = 2;
            }
        s.mask = m2;
        // solid cells of the idle buffer hold w (both buffers do, from the first iteration on)
        for (int gx = 1; gx <= lnx; ++gx)
            for (int y = 0; y < ny; ++y)
                if (s.mask[s.L.at(gx, y)])
                    for (int i = 0; i < Q; ++i) s.f[1][i * s.L.plane + s.L.at(gx, y)] = bc0.w[i];
}

}  // namespace

extern "C" {

// 0: the one-column-lag march; 1: the skewed march, every step on the general / lean step; 2: the skewed march with
// its fast lane (what the device runs by default); 3: ... and the stages T..2 fused
void tb_set_skew(int on) { g_skew = on != 0; g_fast = on >= 2; g_fused = on == 3; }
// A body force (Fx, Fy) for the next tb_emulate calls: runs k_tb<T, B, FORCED = true> (0, 0: the plain program).
void tb_set_force(double fx, double fy) {
    g_force[0] = fx;
    g_force[1] = fy;
}
// Where the LAST pass of the next tb_emulate call (world = 1) emits the moments its last stage's collisions read:
// three arrays of nx*ny doubles in the slab's native order [x*ny + y] (TbArgs::m_rho / m_ux / m_uy); nullptr: off.
void tb_set_macro_sink(double* rho, double* ux, double* uy) {
    g_sink[0] = rho;
    g_sink[1] = ux;
    g_sink[2] = uy;
}
// march steps (per block) taken on the fast lane / on the general step since the last call; resets the counters
void tb_step_counts(long long* fast, long long* general) {
    *fast = lbm::g_steps[0];
    *general = lbm::g_steps[1];
    lbm::g_steps[0] = lbm::g_steps[1] = 0;
}

// state:  global padded AoS [(gy*(nx+2)+gx)*9+i] (reference include/LBMGrid.h:105-107): a post-collision f_next
//         (first_is_current = 0) or an f_current (first_is_current = 1: the first pass must have depth 1 and
//         collides it in place).  Overwritten with f_next after the passes (interior cells; ghost ring untouched).
// solid:  global padded mask [gy*(nx+2)+gx].
// depths: the passes to run, n_pass of them.  world slabs of nx/world columns each exchange the wide halo the
//         way the GPUs do (stores into the neighbour's ghost columns by the last stage).
// flags:  1 periodic x, 2 periodic y.
// Returns the smallest flagged timestep (bad_iter numbering starts at iter0 - 1) or INT_MAX.
int tb_emulate(double* state, const unsigned char* solid, int nx, int ny, double tau, double u_in, int world, int flags,
               const int* depths, int n_pass, int B, int xc, int edge_cols, int halo_w, int first_is_current, int iter0) {
    const bool per_x = flags & 1, per_y = flags & 2;
    const int lnx = nx / world;
    std::vector<Slab> slabs(world);
    BcArgs bc0{};
    bc0.u_in = u_in;
    equilibrium_init(1.0, 0.0, 0.0, bc0.w);
    equilibrium_init(1.0, u_in, 0.0, bc0.e);
    auto g_at = [&](int gx, int gy) { return ((size_t)gy * (nx + 2) + gx) * Q; };
    const double nan = std::numeric_limits<double>::quiet_NaN();
    for (int r = 0; r < world; ++r) init_slab(slabs[r], r, world, state, solid, nx, ny, bc0, per_x, per_y, halo_w, first_is_current);
    for (auto& s : slabs) wrap_ghosts(s, per_x && world == 1, per_y);
    int first_bad = 0x7fffffff;
    int iter = iter0;
    for (int p = 0; p < n_pass; ++p) {
        const int depth = depths[p];
        for (int r = 0; r < world; ++r) {
            Slab& s = slabs[r];
            TbArgs a{};
            a.src = s.f[s.cur].data();
            a.dst = s.f[s.cur ^ 1].data();
            a.L = s.L;
            a.tau_inv = 1.0 / tau;
            a.Fx = g_force[0];
            a.Fy = g_force[1];
            a.first_bad = &first_bad;
            a.bad_iter = iter - 1;
            a.bc = bc0;
            a.bc.inlet = (!per_x && r == 0) ? 1 : 0;
            a.bc.outlet = (!per_x && r == world - 1) ? 1 : 0;
            a.bc.walls = per_y ? 0 : 1;
            a.mask = s.mask.data();
            mask_range(s, a);
            const bool has_w = r > 0 || (per_x && world > 1), has_e = r < world - 1 || (per_x && world > 1);
            a.west = has_w ? TB_EDGE_HALO : (per_x ? TB_EDGE_WRAP : TB_EDGE_CONST);
            a.east = has_e ? TB_EDGE_HALO : (per_x ? TB_EDGE_WRAP : TB_EDGE_CONST);
            a.periodic_y = per_y ? 1 : 0;
            a.pull = (p == 0 && first_is_current) ? 0 : 1;
            a.write = 1;
            a.halo_w = halo_w;
            int chunks;
            if (world > 1) {
                a.edge_cols = edge_cols;
                a.x_begin = edge_cols;
                a.x_end = lnx - edge_cols;
                a.xc = xc;
                chunks = 2 + (a.x_end > a.x_begin ? (a.x_end - a.x_begin + xc - 1) / xc : 0);
                const int wr = has_w ? tb_wrap(r - 1, world) : -1, er = has_e ? tb_wrap(r + 1, world) : -1;
                a.px.peer_dst_west = wr >= 0 ? slabs[wr].f[slabs[wr].cur ^ 1].data() : nullptr;
                a.px.peer_dst_east = er >= 0 ? slabs[er].f[slabs[er].cur ^ 1].data() : nullptr;
            } else {
                a.edge_cols = 0;
                a.x_begin = 0;
                a.x_end = lnx;
                a.xc = xc;
                chunks = (lnx + xc - 1) / xc;
            }
            tb_fill_offsets(a);
            a.pf_dist = 1;
            a.fast_lane = g_fast;
            if (world == 1 && p == n_pass - 1 && g_sink[0]) {
                a.m_rho = g_sink[0];
                a.m_ux = g_sink[1];
                a.m_uy = g_sink[2];
            }
            run_pass(depth, B, a, chunks);
            if (!a.pull) {
                // the engine's one-off launch after the first iteration: the buffer just read (an uploaded f_current may
                // hold anything in its solid cells) is the next destination, and solid cells are never stored
                for (int gx = 1; gx <= lnx; ++gx)
                    for (int y = 0; y < ny; ++y)
                        if (s.mask[s.L.at(gx, y)])
                            for (int i = 0; i < Q; ++i) s.f[s.cur][i * s.L.plane + s.L.at(gx, y)] = bc0.w[i];
            }
        }
        for (auto& s : slabs) s.cur ^= 1;
        for (auto& s : slabs) wrap_ghosts(s, per_x && world == 1, per_y);  // the engine's k_wrap launches
        iter += depth;
    }
    for (int r = 0; r < world; ++r) {
        Slab& s = slabs[r];
        for (int gx = 1; gx <= lnx; ++gx)
            for (int y = 0; y < ny; ++y)
                for (int i = 0; i < Q; ++i) state[g_at(r * lnx + gx, y + 1) + i] = s.f[s.cur][i * s.L.plane + s.L.at(gx, y)];
    }
    return first_bad;
}


// ---- one slab per PROCESS (tests/test_slab_gloo.py, world_size 2 and 4 over gloo): the last stage's peer stores go into
// out-boxes laid out like the neighbour's buffer; the test ships the halo region over gloo and puts it into the
// receiver's ghost columns -- what NVLink does on the GPUs.
struct SlabProc {
    Slab s;
    std::vector<double> out_w, out_e;
    BcArgs bc0{};
    int rank = 0, world = 1, halo_w = 2, lnx = 0, ny = 0;
    double tau = 0.6;
    int first_bad = 0x7fffffff;
    bool first_is_current = false;
    int passes = 0;
};

void* tbs_create(const double* state, const unsigned char* solid, int nx, int ny, double tau, double u_in, int rank, int world,
                 int halo_w, int first_is_current) {
    SlabProc* p = new SlabProc();
    p->rank = rank; p->world = world; p->halo_w = halo_w; p->lnx = nx / world; p->ny = ny; p->tau = tau;
    p->first_is_current = first_is_current != 0;
    p->bc0.u_in = u_in;
    equilibrium_init(1.0, 0.0, 0.0, p->bc0.w);
    equilibrium_init(1.0, u_in, 0.0, p->bc0.e);
    init_slab(p->s, rank, world, state, solid, nx, ny, p->bc0, false, false, halo_w, first_is_current);
    const double nan = std::numeric_limits<double>::quiet_NaN();
    p->out_w.assign((size_t)p->s.L.plane * Q, nan);
    p->out_e.assign((size_t)p->s.L.plane * Q, nan);
    return p;
}

void tbs_destroy(void* h) { delete static_cast<SlabProc*>(h); }

// One pass of `depth` iterations starting with iteration `iter`; returns the smallest flagged timestep so far.
int tbs_pass(void* h, int depth, int B, int xc, int edge_cols, int iter) {
    SlabProc* p = static_cast<SlabProc*>(h);
    Slab& s = p->s;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    std::fill(p->out_w.begin(), p->out_w.end(), nan);
    std::fill(p->out_e.begin(), p->out_e.end(), nan);
    TbArgs a{};
    a.src = s.f[s.cur].data();
    a.dst = s.f[s.cur ^ 1].data();
    a.L = s.L;
    a.tau_inv = 1.0 / p->tau;
    a.first_bad = &p->first_bad;
    a.bad_iter = iter - 1;
    a.bc = p->bc0;
    a.bc.inlet = p->rank == 0 ? 1 : 0;
    a.bc.outlet = p->rank == p->world - 1 ? 1 : 0;
    a.bc.walls = 1;
    a.mask = s.mask.data();
    mask_range(s, a);
    a.west = p->rank > 0 ? TB_EDGE_HALO : TB_EDGE_CONST;
    a.east = p->rank < p->world - 1 ? TB_EDGE_HALO : TB_EDGE_CONST;
    a.pull = (p->passes == 0 && p->first_is_current) ? 0 : 1;
    a.write = 1;
    a.halo_w = p->halo_w;
    a.edge_cols = edge_cols;
    a.x_begin = edge_cols;
    a.x_end = p->lnx - edge_cols;
    a.xc = xc;
    const int chunks = 2 + (a.x_end > a.x_begin ? (a.x_end - a.x_begin + xc - 1) / xc : 0);
    a.px.peer_dst_west = p->rank > 0 ? p->out_w.data() : nullptr;
    a.px.peer_dst_east = p->rank < p->world - 1 ? p->out_e.data() : nullptr;
    tb_fill_offsets(a);
    a.pf_dist = 1;
    a.fast_lane = g_fast;
    run_pass(depth, B, a, chunks);
    if (!a.pull)
        for (int gx = 1; gx <= p->lnx; ++gx)
            for (int y = 0; y < p->ny; ++y)
                if (s.mask[s.L.at(gx, y)])
                    for (int i = 0; i < Q; ++i) s.f[s.cur][i * s.L.plane + s.L.at(gx, y)] = p->bc0.w[i];
    s.cur ^= 1;
    p->passes += 1;
    return p->first_bad;
}

// What this slab's last pass stored for its neighbour: [halo_w][9][ny] (NaN where it stored nothing).
void tbs_get_outbox(void* h, int east, double* buf) {
    SlabProc* p = static_cast<SlabProc*>(h);
    const Layout& L = p->s.L;
    const std::vector<double>& box = east ? p->out_e : p->out_w;
    for (int d = 0; d < p->halo_w; ++d)
        for (int i = 0; i < Q; ++i)
            for (int y = 0; y < p->ny; ++y)
                buf[((size_t)d * Q + i) * p->ny + y] = box[i * L.plane + L.at(east ? -d : p->lnx + 1 + d, y)];
}

// ... lands in the receiver's newest buffer: from_east = it came from the east neighbour (its west out-box).
void tbs_put_inbox(void* h, int from_east, const double* buf) {
    SlabProc* p = static_cast<SlabProc*>(h);
    Slab& s = p->s;
    for (int d = 0; d < p->halo_w; ++d)
        for (int i = 0; i < Q; ++i)
            for (int y = 0; y < p->ny; ++y)
                s.f[s.cur][i * s.L.plane + s.L.at(from_east ? p->lnx + 1 + d : -d, y)] = buf[((size_t)d * Q + i) * p->ny + y];
}

// interior populations of the newest buffer, [ny][lnx][9]
void tbs_get_interior(void* h, double* out) {
    SlabProc* p = static_cast<SlabProc*>(h);
    const Slab& s = p->s;
    for (int y = 0; y < p->ny; ++y)
        for (int gx = 1; gx <= p->lnx; ++gx)
            for (int i = 0; i < Q; ++i) out[((size_t)y * p->lnx + gx - 1) * Q + i] = s.f[s.cur][i * s.L.plane + s.L.at(gx, y)];
}

}  // extern "C"
