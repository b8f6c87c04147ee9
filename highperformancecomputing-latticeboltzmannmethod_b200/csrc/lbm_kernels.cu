// lbm_kernels.cu -- sm_100a kernels of the D2Q9 collide-stream path, A-B double buffer (the in-place
// AA variant lives in lbm_aa.cu).  Compiled with -fmad=false: see lbm_cell.cuh.
//
// Per iteration t >= 1 the engine launches, on one stream:
//   k_bulk_*   every interior cell: new(c) = collide(pull(old))          branch-free, HBM-bound
//   k_fixup    O(nx + ny + solids) cells: redo ring cells with the boundary rules between pull
//              and collide; reset solid cells to w                        list-driven
//   k_forces   output steps only: link-list momentum-exchange reduction
// which together equal collision_step + exchange_ghost_cells + streaming_step +
// apply_boundary_conditions + check_stability of the reference (include/LBMSolver.h:48-64) with
// the state kept as post-collision populations (SURVEY.md Appendix A).
#include <cstdint>

#include "lbm_cell.cuh"
#include "lbm_device.cuh"
#include "lbm_kernels.cuh"
#include "lbm_launch.cuh"

namespace lbm {

namespace {

// ------------------------------------------------------------------------------------------
// Bulk kernel, variant 0: one cell per thread.  Correct for any ny; the baseline the other
// variants are measured against.
template <bool PULL, bool FORCED>
__global__ void __launch_bounds__(256) k_bulk_scalar(StepArgs a, int x_begin, int x_end) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= L.ny) return;
    bool bad = false;
    for (int x = x_begin + blockIdx.y; x < x_end; x += gridDim.y) {
        const int4 iv = column_run(a, x);
        if (y >= iv.z && y < iv.w) continue;  // deep inside the obstacle: stays w
        double f[Q];
        load_cell<PULL>(a.src, L, x + 1, y, f);
        if (PULL) bad |= any_unstable(f);
        collide_cell<FORCED>(f, a.tau_inv, a.Fx, a.Fy);
        if (a.write && !(y >= iv.x && y < iv.y)) store_cell(a.dst, L, x + 1, y, f);
    }
    if (bad) atomicMin(a.first_bad, a.bad_iter);
}

// Bulk kernel, variant 1: two y-adjacent cells per thread.  The three populations that do not
// move in y (0, 1, 3) and all nine stores are 128-bit accesses; the six y-shifted pulls are
// misaligned by one element and use two 64-bit loads each (the second one hits the lines the
// first one brought into L1).  Requires even ny.
template <bool PULL, bool FORCED>
__device__ __forceinline__ bool bulk_vec2_column(const StepArgs& a, int x, int y) {
    const Layout& L = a.L;
    const int gx = x + 1;
    const int4 iv = column_run(a, x);
    if (y >= iv.z && y + 1 < iv.w) return false;  // both cells deep inside the obstacle: they stay w
    const bool sa = (y >= iv.x && y < iv.y), sb = (y + 1 >= iv.x && y + 1 < iv.y);  // solid: never stored
    double fa[Q], fb[Q];
#pragma unroll
    for (int i = 0; i < Q; ++i) {
        const int dx = PULL ? cxi(i) : 0, dy = PULL ? cyi(i) : 0;
        const double* p = a.src + i * L.plane + L.at(gx - dx, y - dy);
        if (dy == 0) {
            const double2 v = __ldg(reinterpret_cast<const double2*>(p));
            fa[i] = v.x;
            fb[i] = v.y;
        } else {
            fa[i] = __ldg(p);
            fb[i] = __ldg(p + 1);
        }
    }
    const bool bad = PULL ? (any_unstable(fa) | any_unstable(fb)) : false;
    collide_cell<FORCED>(fa, a.tau_inv, a.Fx, a.Fy);
    collide_cell<FORCED>(fb, a.tau_inv, a.Fx, a.Fy);
    if (a.write) {
        if (!sa && !sb) {
#pragma unroll
            for (int i = 0; i < Q; ++i)
                *reinterpret_cast<double2*>(a.dst + i * L.plane + L.at(gx, y)) = make_double2(fa[i], fb[i]);
        } else {
#pragma unroll
            for (int i = 0; i < Q; ++i) {
                if (!sa) a.dst[i * L.plane + L.at(gx, y)] = fa[i];
                if (!sb) a.dst[i * L.plane + L.at(gx, y + 1)] = fb[i];
            }
        }
    }
    return bad;
}

template <bool PULL, bool FORCED>
__global__ void __launch_bounds__(128) k_bulk_vec2(StepArgs a, int x_begin, int x_end) {
    pdl_wait();
    pdl_release();
    const int y = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (y >= a.L.ny) return;
    bool bad = false;
    for (int x = x_begin + blockIdx.y; x < x_end; x += gridDim.y) bad |= bulk_vec2_column<PULL, FORCED>(a, x, y);
    if (bad) atomicMin(a.first_bad, a.bad_iter);
}

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_fixup(StepArgs a, BcArgs b, int pull, const int2* __restrict__ ring,
                                               int n_ring, const int2* __restrict__ solids, int n_solid) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < n_ring) {
        const int2 c = ring[idx];
        double f[Q];
        load_cell<true>(a.src, L, c.x + 1, c.y, f);
        double rho_bc, u_out;
        apply_bc(f, c.x, c.y, L, b, rho_bc, u_out);
        if (any_unstable(f)) atomicMin(a.first_bad, a.bad_iter);
        if (a.forced)
            collide_cell<true>(f, a.tau_inv, a.Fx, a.Fy);
        else
            collide_cell<false>(f, a.tau_inv, 0.0, 0.0);
        if (a.write) store_cell(a.dst, L, c.x + 1, c.y, f);
    } else if (idx - n_ring < n_solid) {
        // Solid cells never collide (include/LBMSolver.h:92): f_next keeps eq(1,0,0) for ever and
        // the fluid neighbours simply pull those constants (SURVEY.md F3).
        const int2 c = solids[idx - n_ring];
        if (a.write) store_cell(a.dst, L, c.x + 1, c.y, b.w);
    }
    (void)pull;
}

// ------------------------------------------------------------------------------------------
// The two slab-edge columns (x = 0 and x = lnx-1) of a multi-slab job, every rule in one launch:
// solid cells keep w, fluid cells are pulled, get the wall / inlet / outlet rule that applies to
// them, are checked, collided and stored.  Runs on the communication stream ahead of the halo
// exchange while the bulk kernel works on the interior columns (lbm_engine.cu: step_one).
__global__ void __launch_bounds__(128) k_edge(StepArgs a, BcArgs b, const unsigned char* __restrict__ mask, int pull) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= L.ny) return;
    const int x = blockIdx.y == 0 ? 0 : L.lnx - 1;
    if (mask[L.at(x + 1, y)]) {
        if (a.write) store_cell(a.dst, L, x + 1, y, b.w);
        return;
    }
    double f[Q];
    if (pull) {
        load_cell<true>(a.src, L, x + 1, y, f);
        double rho_bc, u_out;
        apply_bc(f, x, y, L, b, rho_bc, u_out);
        if (any_unstable(f)) atomicMin(a.first_bad, a.bad_iter);
    } else {
        load_cell<false>(a.src, L, x + 1, y, f);
    }
    if (a.forced)
        collide_cell<true>(f, a.tau_inv, a.Fx, a.Fy);
    else
        collide_cell<false>(f, a.tau_inv, 0.0, 0.0);
    if (a.write) store_cell(a.dst, L, x + 1, y, f);
}

// ------------------------------------------------------------------------------------------
// Edge columns + halo exchange in ONE kernel (P2pArgs in the header).  Protocol, per launch `seq`:
//   1. wait until both neighbours have delivered exchange seq-1 (their counters in MY memory).  That
//      also means they have finished reading the ghost columns this launch is about to overwrite in
//      THEIR memory (the A-B pair alternates, so the ghost written now was read by their launch seq-1);
//   2. compute the edge cells, store them locally and push the face-crossing populations into the
//      neighbours' ghost columns (plain stores to peer memory: NVLink);
//   3. __threadfence_system(), and the last block to finish publishes `seq` in the neighbours' memory.
// No rank can run more than one exchange ahead of a neighbour, there is no cycle in the waits (launch
// seq of one GPU only waits for launch seq-1 of another), and a spinning block never keeps another
// GPU from making progress.
// Step 2 for one cell of edge column `col`.
__device__ __forceinline__ void p2p_edge_cell(const StepArgs& a, const BcArgs& b, const unsigned char* __restrict__ mask, int pull,
                                              const P2pArgs& x, int col, int y) {
    const Layout& L = a.L;
    double f[Q];
    if (mask[L.at(col + 1, y)]) {
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = b.w[i];
    } else {
        if (pull) {
            // the ghost column was stored by the neighbouring GPU while this kernel may already have been
            // resident: coherent loads (lbm_device.cuh)
            load_cell<true, true>(a.src, L, col + 1, y, f);
            double rho_bc, u_out;
            apply_bc(f, col, y, L, b, rho_bc, u_out);
            if (any_unstable(f)) atomicMin(a.first_bad, a.bad_iter);
        } else {
            load_cell<false, true>(a.src, L, col + 1, y, f);
        }
        if (a.forced)
            collide_cell<true>(f, a.tau_inv, a.Fx, a.Fy);
        else
            collide_cell<false>(f, a.tau_inv, 0.0, 0.0);
    }
    store_cell(a.dst, L, col + 1, y, f);
    // interior column lnx-1 -> the east neighbour's W ghost (1,5,8 move in +x); column 0 -> the west
    // neighbour's E ghost (3,6,7).  With lnx == 1 the single column feeds both.
    if (x.peer_dst_east && col == L.lnx - 1) {
        x.peer_dst_east[1 * L.plane + L.at(0, y)] = f[1];
        x.peer_dst_east[5 * L.plane + L.at(0, y)] = f[5];
        x.peer_dst_east[8 * L.plane + L.at(0, y)] = f[8];
    }
    if (x.peer_dst_west && col == 0) {
        x.peer_dst_west[3 * L.plane + L.at(L.lnx + 1, y)] = f[3];
        x.peer_dst_west[6 * L.plane + L.at(L.lnx + 1, y)] = f[6];
        x.peer_dst_west[7 * L.plane + L.at(L.lnx + 1, y)] = f[7];
    }
}

// The edge work as the FIRST blocks of the bulk launch itself: blockIdx.y 0 and 1 are the two edge
// columns (256 rows per block, two per thread), blockIdx.y >= 2 the interior columns.  The peer
// stores and the flag hand-shake then cost nothing: they run under the 0.7 ms interior kernel.
template <bool PULL, bool FORCED>
__global__ void __launch_bounds__(128) k_bulk_vec2_p2p(StepArgs a, int x_begin, int x_end, BcArgs b,
                                                       const unsigned char* __restrict__ mask, P2pArgs px) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    if (blockIdx.y < 2) {
        p2p_block_begin(px);
        const int col = blockIdx.y == 0 ? 0 : L.lnx - 1;
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
            const int y = blockIdx.x * 256 + r * 128 + threadIdx.x;
            if (y < L.ny) p2p_edge_cell(a, b, mask, PULL ? 1 : 0, px, col, y);
        }
        p2p_block_end(px, gridDim.x * 2);
        return;
    }
    const int y = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (y >= L.ny) return;
    bool bad = false;
    for (int x = x_begin + (blockIdx.y - 2); x < x_end; x += gridDim.y - 2) bad |= bulk_vec2_column<PULL, FORCED>(a, x, y);
    if (bad) atomicMin(a.first_bad, a.bad_iter);
}

// Fallback for odd ny / the scalar variant.  Boundary fix-up of a slab with neighbours: the list-driven ring / solid work of k_fixup plus,
// in the FIRST blocks of the grid, every cell of the two slab-edge columns with the halo exchange
// fused in (steps 1-3 above).  The bulk kernel has already run over all columns; what it wrote into
// the edge columns (computed from ghost columns that may not have been refreshed yet) is simply
// overwritten here, exactly as for ring cells.
__global__ void __launch_bounds__(128) k_fixup_p2p(StepArgs a, BcArgs b, int pull, const int2* __restrict__ ring, int n_ring,
                                                   const int2* __restrict__ solids, int n_solid,
                                                   const unsigned char* __restrict__ mask, P2pArgs px, int edge_blocks) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    if ((int)blockIdx.x < edge_blocks) {
        p2p_block_begin(px);
        const int per_col = edge_blocks / (L.lnx > 1 ? 2 : 1);
        const int col = (int)blockIdx.x < per_col ? 0 : L.lnx - 1;
        const int y = ((int)blockIdx.x % per_col) * blockDim.x + threadIdx.x;
        if (y < L.ny) p2p_edge_cell(a, b, mask, pull, px, col, y);
        p2p_block_end(px, (unsigned int)edge_blocks);
        return;
    }
    const int idx = (blockIdx.x - edge_blocks) * blockDim.x + threadIdx.x;
    if (idx < n_ring) {
        if (!pull) return;  // the first iteration collides f_current as it is
        const int2 c = ring[idx];
        double f[Q];
        load_cell<true>(a.src, L, c.x + 1, c.y, f);
        double rho_bc, u_out;
        apply_bc(f, c.x, c.y, L, b, rho_bc, u_out);
        if (any_unstable(f)) atomicMin(a.first_bad, a.bad_iter);
        if (a.forced)
            collide_cell<true>(f, a.tau_inv, a.Fx, a.Fy);
        else
            collide_cell<false>(f, a.tau_inv, 0.0, 0.0);
        store_cell(a.dst, L, c.x + 1, c.y, f);
    } else if (idx - n_ring < n_solid) {
        const int2 c = solids[idx - n_ring];
        store_cell(a.dst, L, c.x + 1, c.y, b.w);
    }
}

__global__ void k_wait_halo(P2pArgs x) {
    if (x.peer_dst_west) spin_until(x.my_flags + 0, x.seq, x);
    if (x.peer_dst_east) spin_until(x.my_flags + 1, x.seq, x);
    __threadfence_system();
}

// ------------------------------------------------------------------------------------------
// Momentum exchange: F = sum over links 2 c_i f_next(fluid, i)  (include/LBMIO.h:123-160).
// The reference accumulates ONE running sum per component in (y, x, i) order over the solid
// cells; the link list is built in that order, so adding the terms one after the other gives the
// reference's bits (and with them forces.csv byte for byte, down to the sign of a lift that
// cancels to +-1e-16).  The gather is parallel (256 threads stage a chunk of link terms in shared
// memory); the additions are serial, one thread per component.  ~10 cycles per link, once every
// output_frequency steps: 7 904 links (32768 x 8192) cost ~40 us per 140 steps.
constexpr int FORCE_CHUNK = 2048;

__global__ void __launch_bounds__(256) k_forces(const double* __restrict__ f, const Link* __restrict__ links,
                                                int n_links, double* __restrict__ out) {
    pdl_wait();
    pdl_release();
    __shared__ double tx[FORCE_CHUNK], ty[FORCE_CHUNK];
    double acc = 0.0;  // thread 0: Fx, thread 32: Fy
    for (int base = 0; base < n_links; base += FORCE_CHUNK) {
        const int n = min(FORCE_CHUNK, n_links - base);
        for (int k = threadIdx.x; k < n; k += blockDim.x) {
            const Link l = links[base + k];
            const double v = f[l.off];
            tx[k] = (double)l.cx2 * v;  // 2.0 * c_ix * f_i, exact
            ty[k] = (double)l.cy2 * v;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int k = 0; k < n; ++k) acc += tx[k];
        } else if (threadIdx.x == 32) {
            for (int k = 0; k < n; ++k) acc += ty[k];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = acc;
    if (threadIdx.x == 32) out[1] = acc;
}

// The same sum as a fixed TREE (LBM_FORCES_TREE): every thread adds its links k = tid, tid + 1024, ... in that order,
// then warp shuffles and one shared-memory stage combine the 1024 partial sums in a fixed pattern -- deterministic
// from launch to launch, ~3 us whatever the link count, equal to the ordered sum to rounding (a few 1e-16 relative;
// not bit-identical: floating-point addition is not associative).  This is the mode for dense force sampling.
__global__ void __launch_bounds__(1024) k_forces_tree(const double* __restrict__ f, const Link* __restrict__ links,
                                                      int n_links, double* __restrict__ out) {
    pdl_wait();
    pdl_release();
    __shared__ double sx[32], sy[32];
    double ax = 0.0, ay = 0.0;
    for (int k = threadIdx.x; k < n_links; k += blockDim.x) {
        const Link l = links[k];
        const double v = f[l.off];
        ax += (double)l.cx2 * v;
        ay += (double)l.cy2 * v;
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        ax += __shfl_down_sync(0xffffffffu, ax, s);
        ay += __shfl_down_sync(0xffffffffu, ay, s);
    }
    if ((threadIdx.x & 31) == 0) {
        sx[threadIdx.x >> 5] = ax;
        sy[threadIdx.x >> 5] = ay;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        ax = sx[threadIdx.x];
        ay = sy[threadIdx.x];
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            ax += __shfl_down_sync(0xffffffffu, ax, s);
            ay += __shfl_down_sync(0xffffffffu, ay, s);
        }
        if (threadIdx.x == 0) {
            out[0] = ax;
            out[1] = ay;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Periodic extensions: copy the opposite interior edge into the ghost ring.
__global__ void k_wrap(double* __restrict__ f, Layout L, int wrap_x, int wrap_y) {
    pdl_wait();
    pdl_release();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    double* p = f + i * L.plane;
    if (wrap_x && t < L.ny) {
        p[L.at(0, t)] = p[L.at(L.lnx, t)];
        p[L.at(L.lnx + 1, t)] = p[L.at(1, t)];
    }
    if (wrap_y && t < L.lnx + 2) {
        // columns incl. ghost columns: after the x wrap above has been made visible by a
        // previous launch (the engine launches x then y) the corners come out right.
        p[L.at(t, -1)] = p[L.at(t, L.ny - 1)];
        p[L.at(t, L.ny)] = p[L.at(t, 0)];
    }
}

// ------------------------------------------------------------------------------------------
// Initial state.  Every padded cell of both buffers = eq(1, u_in, 0) (include/LBMGrid.h:191-212),
// solids = eq(1,0,0) (:229-242).  The W/E ghost columns at physical domain edges are set to the
// value the reference's exchange gives them from the first iteration on: 0.0 (SURVEY.md F4).
__global__ void k_init(double* __restrict__ f0, double* __restrict__ f1, Layout L,
                       const unsigned char* __restrict__ mask, BcArgs b, int west_zero, int east_zero,
                       int shear_wave, double u0) {
    const int y = (int)(blockIdx.x * blockDim.x + threadIdx.x) - 1;  // -1 .. ny
    if (y > L.ny) return;
    const bool ghost_row = (y < 0 || y >= L.ny);
    // every column of the padded slab, the XO extra ghost columns of a temporally blocked halo included
    for (int g = blockIdx.y; g < L.lnx + 2 + 2 * Layout::XO; g += gridDim.y) {
    const int gx = g - Layout::XO;
    const bool interior = !ghost_row && gx >= 1 && gx <= L.lnx;
    double v[Q];
    if (interior && mask[L.at(gx, y)]) {
#pragma unroll
        for (int i = 0; i < Q; ++i) v[i] = b.w[i];
    } else if (!ghost_row && ((gx <= 0 && west_zero) || (gx >= L.lnx + 1 && east_zero))) {
#pragma unroll
        for (int i = 0; i < Q; ++i) v[i] = 0.0;
    } else if (shear_wave) {
        int yy = y < 0 ? y + L.ny : (y >= L.ny ? y - L.ny : y);
        const double ux = u0 * sin(2.0 * 3.14159265358979323846 * (double)yy / (double)L.ny);
        equilibrium_init(1.0, ux, 0.0, v);
    } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) v[i] = b.e[i];
    }
    store_cell(f0, L, gx, y, v);
    store_cell(f1, L, gx, y, v);
    }
}

__global__ void k_reset_ghosts(double* __restrict__ f, Layout L, BcArgs b, int west_zero, int east_zero) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    double z[Q] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (t < L.ny) {
        for (int d = 0; d <= Layout::XO; ++d) {
            store_cell(f, L, -d, t, west_zero ? z : b.e);
            store_cell(f, L, L.lnx + 1 + d, t, east_zero ? z : b.e);
        }
    }
    if (t < L.lnx + 2 + 2 * Layout::XO) {
        store_cell(f, L, t - Layout::XO, -1, b.e);
        store_cell(f, L, t - Layout::XO, L.ny, b.e);
    }
}

// ------------------------------------------------------------------------------------------
// rho, ux, uy as the reference's arrays hold them (see ObserveArgs in the header).
__device__ __forceinline__ void macros_cell(const ObserveArgs& o, int x, int y, double& rho, double& ux,
                                            double& uy) {
    const Layout& L = o.L;
    const bool solid = o.mask[L.at(x + 1, y)] != 0;
    if (o.fresh) {  // include/LBMGrid.h:216-228
        rho = 1.0;
        uy = 0.0;
        if (solid)
            ux = 0.0;
        else if (o.shear_wave)
            ux = o.u0 * sin(2.0 * 3.14159265358979323846 * (double)y / (double)L.ny);
        else
            ux = o.u0;  // the velocity Grid::initialise(inlet_u) was given, not the params' inlet velocity
        return;
    }
    if (solid) {  // rho stays 1.0 from the constructor; include/LBMSolver.h:260-261
        rho = 1.0;
        ux = 0.0;
        uy = 0.0;
        return;
    }
    double f[Q], rb = 0.0, uo = 0.0;
    if (!o.cur_is_next) {
        // no iteration since an upload: moments of the uploaded f_current
        load_cell<false>(o.cur, L, x + 1, y, f);
        const Moments m = moments(f);
        rho = m.rho; ux = m.ux; uy = m.uy;
        return;
    }
    // moments stored by the last collision (include/LBMSolver.h:112-114): those of the f_current
    // that collision read, i.e. of the PREVIOUS buffer's streamed + boundary-treated state
    if (o.prev_is_next)
        current_from_next(o.prev, L, o.mask, o.bc, x, y, f, rb, uo);
    else
        load_cell<false>(o.prev, L, x + 1, y, f);
    const Moments m = moments(f);
    rho = m.rho; ux = m.ux; uy = m.uy;
    // ... then overwritten on the inlet / outlet columns by the boundary pass that built the
    // newest f_current (include/LBMSolver.h:203-205, 232-234)
    const bool on_in = o.bc.inlet && x == 0, on_out = o.bc.outlet && x == L.lnx - 1;
    if (on_in || on_out) {
        current_from_next(o.cur, L, o.mask, o.bc, x, y, f, rb, uo);
        if (on_in) { rho = rb; ux = o.bc.u_in; uy = 0.0; }
        if (on_out) { rho = 1.0; ux = uo; uy = 0.0; }
    }
}

// 32 x 32 tile transpose: reads follow the SoA (y fastest), writes follow the reference's
// interior row-major order (x fastest).
__global__ void __launch_bounds__(256) k_macros(ObserveArgs o, double* __restrict__ rho, double* __restrict__ ux,
                                                double* __restrict__ uy) {
    __shared__ double t[3][32][33];
    const Layout& L = o.L;
    const int x0 = blockIdx.y * 32, y0 = blockIdx.x * 32;
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int x = x0 + k, y = y0 + threadIdx.x;
        if (x < L.lnx && y < L.ny) {
            double r, u, v;
            macros_cell(o, x, y, r, u, v);
            t[0][k][threadIdx.x] = r;
            t[1][k][threadIdx.x] = u;
            t[2][k][threadIdx.x] = v;
        }
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int x = x0 + threadIdx.x, y = y0 + k;
        if (x < L.lnx && y < L.ny) {
            const long long g = (long long)y * L.lnx + x;
            rho[g] = t[0][threadIdx.x][k];
            ux[g] = t[1][threadIdx.x][k];
            uy[g] = t[2][threadIdx.x][k];
        }
    }
}

__global__ void __launch_bounds__(256) k_maxvel(const double* __restrict__ ux, const double* __restrict__ uy,
                                                long long n, unsigned long long* out_bits) {
    double m = 0.0;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const double v = ux[k] * ux[k] + uy[k] * uy[k];
        m = v > m ? v : m;  // include/LBMGrid.h:330-331 (max of non-negative values; NaN never wins, as _mm256_max_pd)
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const double other = __shfl_down_sync(0xffffffffu, m, s);
        m = other > m ? other : m;
    }
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits, (unsigned long long)__double_as_longlong(m));
}

// Export in the reference's padded AoS order, tile = 16 columns x 32 rows x 9 populations.
constexpr int EX_TX = 16, EX_TY = 32;

// Padded rows [row0, row0 + rows) only, `aos` pointing at the first of them: the host copy runs in chunks that
// overlap the kernel (lbm_engine.cu).
__global__ void __launch_bounds__(256) k_export_f(ObserveArgs o, int which, double* __restrict__ aos, int row0, int rows) {
    __shared__ double t[Q][EX_TX][EX_TY + 1];
    const Layout& L = o.L;
    const int tnx = L.lnx + 2, tny = min(L.ny + 2, row0 + rows);
    const int gx0 = blockIdx.y * EX_TX, gy0 = row0 + blockIdx.x * EX_TY;  // padded coordinates
    for (int c = threadIdx.x; c < EX_TX * EX_TY; c += blockDim.x) {
        const int xl = c / EX_TY, yl = c % EX_TY;
        const int gx = gx0 + xl, gy = gy0 + yl;
        if (gx >= tnx || gy >= tny) continue;
        const int x = gx - 1, y = gy - 1;
        const bool ghost = (x < 0 || x >= L.lnx || y < 0 || y >= L.ny);
        double f[Q];
        // f_next before the first iteration equals f_current (include/LBMGrid.h:209-211)
        const bool want_current = (which == 0) || !o.cur_is_next;
        if (want_current) {
            if (ghost) {  // never written after initialise (SURVEY.md Appendix A, step 6)
#pragma unroll
                for (int i = 0; i < Q; ++i) f[i] = o.bc.e[i];
            } else if (o.cur_is_next) {
                double rb, uo;
                current_from_next(o.cur, L, o.mask, o.bc, x, y, f, rb, uo);
            } else {
                load_cell<false>(o.cur, L, gx, y, f);
            }
        } else {
            load_cell<false>(o.cur, L, gx, y, f);
        }
#pragma unroll
        for (int i = 0; i < Q; ++i) t[i][xl][yl] = f[i];
    }
    __syncthreads();
    const int nxl = min(EX_TX, tnx - gx0);
    for (int k = threadIdx.x; k < EX_TY * nxl * Q; k += blockDim.x) {
        const int yl = k / (nxl * Q), e = k % (nxl * Q);
        const int gy = gy0 + yl;
        if (gy >= tny) break;
        aos[((long long)(gy - row0) * tnx + gx0) * Q + e] = t[e % Q][e / Q][yl];
    }
}

// The interior cells of padded rows [row0, row0 + rows), `aos` pointing at the first of those rows.
__global__ void __launch_bounds__(256) k_import_f(const double* __restrict__ aos, double* __restrict__ f, Layout L, int row0,
                                                  int rows) {
    __shared__ double t[Q][EX_TX][EX_TY + 1];
    const int tnx = L.lnx + 2;
    const int x0 = blockIdx.y * EX_TX, gy0 = row0 + blockIdx.x * EX_TY;
    const int gy_end = min(L.ny + 1, row0 + rows);  // one past the last interior padded row of the chunk
    const int nxl = min(EX_TX, L.lnx - x0);
    for (int k = threadIdx.x; k < EX_TY * nxl * Q; k += blockDim.x) {
        const int yl = k / (nxl * Q), e = k % (nxl * Q);
        const int gy = gy0 + yl;
        if (gy >= gy_end) break;
        if (gy >= 1) t[e % Q][e / Q][yl] = aos[((long long)(gy - row0) * tnx + (x0 + 1)) * Q + e];
    }
    __syncthreads();
    for (int k = threadIdx.x; k < Q * EX_TX * EX_TY; k += blockDim.x) {
        const int i = k / (EX_TX * EX_TY), xl = (k / EX_TY) % EX_TX, yl = k % EX_TY;
        const int x = x0 + xl, gy = gy0 + yl;
        if (x < L.lnx && gy >= 1 && gy < gy_end) f[i * L.plane + L.at(x + 1, gy - 1)] = t[i][xl][yl];
    }
}

// Caller-written f_next values of solid cells / ghost rows (lbm_upload_f_next): a compact (offset, value) list into
// both population buffers.
__global__ void __launch_bounds__(256) k_scatter(const long long* __restrict__ off, const double* __restrict__ val, int n,
                                                 double* __restrict__ f0, double* __restrict__ f1) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    f0[off[k]] = val[k];
    if (f1) f1[off[k]] = val[k];
}

// Self-test of div_pair (lbm_cell.cuh) against the compiler's IEEE division, bit for bit, on pseudo-random operands:
// densities near 1 and all over the exponent range (negative, zero, denormal, infinite, NaN included), numerators
// from exactly zero (both signs) and denormals to beyond the stability limit.
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

__device__ __forceinline__ double test_operand(unsigned long long h, int kind) {
    const unsigned long long mant = h & 0x000FFFFFFFFFFFFFULL, sign = (h >> 63) << 63;
    unsigned long long e;
    switch (kind) {
        case 0: e = 1022 + ((h >> 52) & 1); break;                  // [0.5, 2)
        case 1: e = 1023 - 30 + ((h >> 52) % 48); break;            // 2^-30 .. 2^17
        case 2: e = (h >> 52) & 0x7ff; break;                       // anything: denormals, inf, NaN
        case 3: return __longlong_as_double((long long)sign);       // +-0
        default: e = ((h >> 52) & 1) ? 1023 - 510 + ((h >> 53) % 20) : 1023 + 490 + ((h >> 53) % 20); break;  // the window's edges
    }
    return __longlong_as_double((long long)(sign | (e << 52) | mant));
}

__global__ void k_selftest_div(unsigned long long seed, long long n, unsigned long long* mismatches) {
    unsigned long long bad = 0;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const unsigned long long h0 = mix64(seed + 3 * (unsigned long long)k), h1 = mix64(h0), h2 = mix64(h1);
        const int mode = (int)(h0 % 10);
        double den = test_operand(h0 >> 1, mode < 6 ? 0 : (mode < 8 ? 1 : (mode == 8 ? 2 : 4)));
        if (mode < 7) den = fabs(den);
        const double a = test_operand(h1, (int)((h1 >> 3) % 5)), b = test_operand(h2, (int)((h2 >> 3) % 5));
        double qa, qb;
        div_pair(a, b, den, qa, qb);
        const double ra = a / den, rb = b / den;
        const bool same_a = __double_as_longlong(qa) == __double_as_longlong(ra) || (qa != qa && ra != ra);
        const bool same_b = __double_as_longlong(qb) == __double_as_longlong(rb) || (qb != qb && rb != rb);
        bad += (same_a ? 0 : 1) + (same_b ? 0 : 1);
    }
    if (bad) atomicAdd(mismatches, bad);
}

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

}  // namespace

cudaError_t launch_selftest_div(unsigned long long seed, long long n, unsigned long long* mismatches, cudaStream_t s) {
    k_selftest_div<<<148 * 8, 256, 0, s>>>(seed, n, mismatches);
    return cudaGetLastError();
}

cudaError_t launch_scatter(const long long* off, const double* val, int n, double* f0, double* f1, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    k_scatter<<<cdiv(n, 256), 256, 0, s>>>(off, val, n, f0, f1);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
cudaError_t launch_bulk(int variant, bool pull, const StepArgs& a, cudaStream_t s, int x_begin, int x_end) {
    if (x_end < 0) x_end = a.L.lnx;
    const int ncols = x_end - x_begin;
    if (ncols <= 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (variant != BULK_SCALAR && (a.L.ny % 2 == 0)) {
        dim3 grid(cdiv(a.L.ny / 2, 128), ncols < 65535 ? ncols : 65535);
        if (pull) {
            if (a.forced) e = launch_chain(k_bulk_vec2<true, true>, grid, dim3(128), s, a, x_begin, x_end);
            else e = launch_chain(k_bulk_vec2<true, false>, grid, dim3(128), s, a, x_begin, x_end);
        } else {
            if (a.forced) e = launch_chain(k_bulk_vec2<false, true>, grid, dim3(128), s, a, x_begin, x_end);
            else e = launch_chain(k_bulk_vec2<false, false>, grid, dim3(128), s, a, x_begin, x_end);
        }
    } else {
        dim3 grid(cdiv(a.L.ny, 256), ncols < 65535 ? ncols : 65535);
        if (pull) {
            if (a.forced) e = launch_chain(k_bulk_scalar<true, true>, grid, dim3(256), s, a, x_begin, x_end);
            else e = launch_chain(k_bulk_scalar<true, false>, grid, dim3(256), s, a, x_begin, x_end);
        } else {
            if (a.forced) e = launch_chain(k_bulk_scalar<false, true>, grid, dim3(256), s, a, x_begin, x_end);
            else e = launch_chain(k_bulk_scalar<false, false>, grid, dim3(256), s, a, x_begin, x_end);
        }
    }
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_fixup(bool pull, const StepArgs& a, const BcArgs& b, const int2* ring, int n_ring,
                         const int2* solids, int n_solid, cudaStream_t s) {
    if (!pull) n_ring = 0;  // the first iteration collides f_current as it is: no boundary pass before it
    const long long n = (long long)n_ring + n_solid;
    if (n == 0) return cudaSuccess;
    return launch_chain(k_fixup, dim3(cdiv(n, 128)), dim3(128), s, a, b, pull ? 1 : 0, ring, n_ring, solids, n_solid);
}

cudaError_t launch_edge(bool pull, const StepArgs& a, const BcArgs& b, const unsigned char* mask, cudaStream_t s) {
    dim3 grid(cdiv(a.L.ny, 128), a.L.lnx > 1 ? 2 : 1);
    return launch_chain(k_edge, grid, dim3(128), s, a, b, mask, pull ? 1 : 0);
}

bool bulk_p2p_supported(int variant, const StepArgs& a) { return variant != BULK_SCALAR && a.L.ny % 2 == 0 && a.L.lnx >= 4; }

cudaError_t launch_bulk_p2p(bool pull, const StepArgs& a, const BcArgs& b, const unsigned char* mask, const P2pArgs& x,
                            cudaStream_t s) {
    const int x_begin = 1, x_end = a.L.lnx - 1, ncols = x_end - x_begin;
    dim3 grid(cdiv(a.L.ny / 2, 128), (ncols < 65533 ? ncols : 65533) + 2);
    if (pull)
        return a.forced ? launch_chain(k_bulk_vec2_p2p<true, true>, grid, dim3(128), s, a, x_begin, x_end, b, mask, x)
                        : launch_chain(k_bulk_vec2_p2p<true, false>, grid, dim3(128), s, a, x_begin, x_end, b, mask, x);
    return a.forced ? launch_chain(k_bulk_vec2_p2p<false, true>, grid, dim3(128), s, a, x_begin, x_end, b, mask, x)
                    : launch_chain(k_bulk_vec2_p2p<false, false>, grid, dim3(128), s, a, x_begin, x_end, b, mask, x);
}

cudaError_t launch_fixup_p2p(bool pull, const StepArgs& a, const BcArgs& b, const int2* ring, int n_ring, const int2* solids,
                             int n_solid, const unsigned char* mask, const P2pArgs& x, cudaStream_t s) {
    const int edge_blocks = cdiv(a.L.ny, 128) * (a.L.lnx > 1 ? 2 : 1);
    const long long n = (long long)n_ring + n_solid;
    return launch_chain(k_fixup_p2p, dim3(edge_blocks + cdiv(n, 128)), dim3(128), s, a, b, pull ? 1 : 0, ring, n_ring, solids,
                        n_solid, mask, x, edge_blocks);
}

cudaError_t launch_wait_halo(const P2pArgs& x, cudaStream_t s) {
    k_wait_halo<<<1, 1, 0, s>>>(x);
    return cudaGetLastError();
}

cudaError_t launch_forces(const double* f_next, const Link* links, int n_links, double* out, cudaStream_t s, int tree) {
    if (tree) return launch_chain(k_forces_tree, dim3(1), dim3(1024), s, f_next, links, n_links, out);
    return launch_chain(k_forces, dim3(1), dim3(256), s, f_next, links, n_links, out);
}

cudaError_t launch_wrap(double* f, const Layout& L, int wrap_x, int wrap_y, cudaStream_t s) {
    cudaError_t e = cudaSuccess;
    if (wrap_x) {
        e = launch_chain(k_wrap, dim3(cdiv(L.ny, 256), Q), dim3(256), s, f, L, 1, 0);
    }
    if (wrap_y) {
        e = launch_chain(k_wrap, dim3(cdiv(L.lnx + 2, 256), Q), dim3(256), s, f, L, 0, 1);
    }
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_init(double* f0, double* f1, const Layout& L, const unsigned char* mask, const BcArgs& b,
                        int west_zero, int east_zero, int shear_wave, double u0, cudaStream_t s) {
    const int ncol = L.lnx + 2 + 2 * Layout::XO;
    dim3 grid(cdiv(L.ny + 2, 256), ncol < 65535 ? ncol : 65535);
    k_init<<<grid, 256, 0, s>>>(f0, f1, L, mask, b, west_zero, east_zero, shear_wave, u0);
    return cudaGetLastError();
}

cudaError_t launch_reset_ghosts(double* f, const Layout& L, const BcArgs& b, int west_zero, int east_zero,
                                cudaStream_t s) {
    const int n = (L.ny > L.lnx + 2 + 2 * Layout::XO) ? L.ny : L.lnx + 2 + 2 * Layout::XO;
    k_reset_ghosts<<<cdiv(n, 256), 256, 0, s>>>(f, L, b, west_zero, east_zero);
    return cudaGetLastError();
}

cudaError_t launch_macros(const ObserveArgs& o, double* rho, double* ux, double* uy, cudaStream_t s) {
    dim3 grid(cdiv(o.L.ny, 32), cdiv(o.L.lnx, 32));
    k_macros<<<grid, dim3(32, 8), 0, s>>>(o, rho, ux, uy);
    return cudaGetLastError();
}

cudaError_t launch_maxvel(const double* ux, const double* uy, long long n, unsigned long long* out_bits,
                          cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(out_bits, 0, sizeof(unsigned long long), s);
    if (e != cudaSuccess) return e;
    int blocks = cdiv(n, 256 * 8);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    k_maxvel<<<blocks, 256, 0, s>>>(ux, uy, n, out_bits);
    return cudaGetLastError();
}

cudaError_t launch_export_f(const ObserveArgs& o, int which, double* aos, int row0, int rows, cudaStream_t s) {
    dim3 grid(cdiv(rows, EX_TY), cdiv(o.L.lnx + 2, EX_TX));
    k_export_f<<<grid, 256, 0, s>>>(o, which, aos, row0, rows);
    return cudaGetLastError();
}

cudaError_t launch_import_f(const double* aos, double* f, const Layout& L, int row0, int rows, cudaStream_t s) {
    dim3 grid(cdiv(rows, EX_TY), cdiv(L.lnx, EX_TX));
    k_import_f<<<grid, 256, 0, s>>>(aos, f, L, row0, rows);
    return cudaGetLastError();
}

}  // namespace lbm
