// lbm_aa.cu -- in-place "AA pattern" variant of the collide-stream path: ONE population buffer.
//
// Same arithmetic per cell as the A-B kernels (lbm_cell.cuh), different addressing (Bailey et al.
// 2009).  Reference iterations alternate between two kinds of step on the single buffer A:
//
//   E-step (even):  f_i <- A[x][i]                 -> boundary rule -> collide -> A[x][opp(i)] <- f*_i
//   O-step (odd):   f_i <- A[x - c_i][opp(i)]      -> boundary rule -> collide -> A[x + c_i][i] <- f*_i
//
// After an E-step the buffer is in the REVERSED layout (A[x][opp(i)] = f_next_i(x)); after an
// O-step it is back in the NATURAL layout (A[x][i] = f_next_i(x - c_i), i.e. the streamed,
// not yet boundary-treated f_current_i(x)).  Every thread reads and writes the same nine slots,
// so no second buffer and no synchronisation are needed: the only writer of slot [n][s] is the
// cell n - c_s, which is also its only reader.
//
// How the reference's quirks (SURVEY.md F3/F4) survive:
//   * solid cells are reset to w after every E-step (fix-up kernel), so the O-step's pulls see w;
//   * ghost cells of non-periodic edges permanently hold the REVERSED constants
//     (slot opp(i) = value of population i: 0 in the W/E ghost columns, eq(1,u_in,0) in the S/N
//     rows) and are never written: ring cells are excluded from the bulk kernels and the
//     ring fix-up does not push out of the domain;
//   * after every O-step a list-driven fill writes the constant a fluid cell would have pulled
//     from a solid or ghost neighbour into its slot [x][i] (nobody pushes there);
//   * the populations a ring cell sends out of the domain have no slot: the O-step fix-up keeps
//     all nine post-collision values of every ring cell in a small side array for the observers.
// Periodic directions use the forward ghost wrap after E-steps and a reverse wrap (ghost -> the
// interior image) after O-steps.
#include <cstdint>

#include "lbm_cell.cuh"
#include "lbm_device.cuh"
#include "lbm_kernels.cuh"
#include "lbm_launch.cuh"

namespace lbm {

namespace {

__device__ __forceinline__ bool any_bad(const double f[Q]) {
    bool bad = false;
#pragma unroll
    for (int i = 0; i < Q; ++i) bad |= unstable_value(f[i]);
    return bad;
}

__device__ __forceinline__ void collide(double f[Q], const AaArgs& a) {
    const Moments m = moments(f);
    if (a.forced)
        bgk_forced(f, m, a.tau_inv, a.Fx, a.Fy, f);
    else
        bgk(f, m, a.tau_inv, f);
}

__device__ __forceinline__ void bc_rules(double f[Q], int x, int y, const Layout& L, const BcArgs& b, double& rho_bc,
                                         double& u_out) {
    // the reference's serial order: bottom, top, inlet, outlet (include/LBMSolver.h:153-236)
    if (b.walls && y == 0) wall_bottom(f);
    if (b.walls && y == L.ny - 1) wall_top(f);
    if (b.inlet && x == 0) rho_bc = zou_he_inlet(f, b.u_in);
    if (b.outlet && x == L.lnx - 1) u_out = zou_he_outlet(f);
}

__device__ __forceinline__ bool is_ring(int x, int y, const Layout& L, const BcArgs& b) {
    return (b.walls && (y == 0 || y == L.ny - 1)) || (b.inlet && x == 0) || (b.outlet && x == L.lnx - 1);
}

__device__ __forceinline__ int ring_slot(int x, int y, const Layout& L) {
    if (x == 0) return y;
    if (x == L.lnx - 1) return L.ny + y;
    if (y == 0) return 2 * L.ny + x;
    return 2 * L.ny + L.lnx + x;
}

// ------------------------------------------------------------------------------------------
// Bulk kernels: every interior cell that is not a ring cell.  Two y-adjacent cells per thread.
// A pair is "plain" when neither cell lies on a wall row or in the obstacle: those take the
// unpredicated path; the few other pairs write cell by cell.  Solid cells are checked (the
// reference's stability check sees what the fluid pushed into them) but never written or pushed
// from; pairs deep inside the obstacle are skipped.
template <bool FORCED>
__device__ __forceinline__ void collide_pair(double fa[Q], double fb[Q], const AaArgs& a) {
    const Moments ma = moments(fa), mb = moments(fb);
    if (FORCED) {
        bgk_forced(fa, ma, a.tau_inv, a.Fx, a.Fy, fa);
        bgk_forced(fb, mb, a.tau_inv, a.Fx, a.Fy, fb);
    } else {
        bgk(fa, ma, a.tau_inv, fa);
        bgk(fb, mb, a.tau_inv, fb);
    }
}

template <bool FIRST, bool FORCED>
__global__ void __launch_bounds__(128, 6) k_aa_even_vec2(AaArgs a) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int y = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (y >= L.ny) return;
    const bool wall_a = a.skip_rows && y == 0, wall_b = a.skip_rows && y + 1 == L.ny - 1;
    bool bad = false;
    for (int x = a.x_begin + blockIdx.y; x < a.x_end; x += gridDim.y) {
        const int4 iv = column_run(a, x);
        if (y >= iv.z && y + 1 < iv.w) continue;
        double* p = a.f + L.at(x + 1, y);
        double fa[Q], fb[Q];
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            const double2 v = *reinterpret_cast<const double2*>(p + i * L.plane);
            fa[i] = v.x;
            fb[i] = v.y;
        }
        if (!FIRST) bad |= (!wall_a && any_bad(fa)) | (!wall_b && any_bad(fb));
        collide_pair<FORCED>(fa, fb, a);
        const bool wa = !wall_a && !(y >= iv.x && y < iv.y), wb = !wall_b && !(y + 1 >= iv.x && y + 1 < iv.y);
        if (wa && wb) {
#pragma unroll
            for (int i = 0; i < Q; ++i) *reinterpret_cast<double2*>(p + oppi(i) * L.plane) = make_double2(fa[i], fb[i]);
        } else {
#pragma unroll
            for (int i = 0; i < Q; ++i) {
                if (wa) p[oppi(i) * L.plane] = fa[i];
                if (wb) p[oppi(i) * L.plane + 1] = fb[i];
            }
        }
    }
    if (bad) atomicMin(a.first_bad, a.bad_iter);
}

template <bool FORCED>
__global__ void __launch_bounds__(128, 6) k_aa_odd_vec2(AaArgs a) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int y = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (y >= L.ny) return;
    const bool wall_a = a.skip_rows && y == 0, wall_b = a.skip_rows && y + 1 == L.ny - 1;
    bool bad = false;
    for (int x = a.x_begin + blockIdx.y; x < a.x_end; x += gridDim.y) {
        const int gx = x + 1;
        const int4 iv = column_run(a, x);
        if (y >= iv.z && y + 1 < iv.w) continue;
        double fa[Q], fb[Q];
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            const double* p = a.f + oppi(i) * L.plane + L.at(gx - cxi(i), y - cyi(i));
            if (cyi(i) == 0) {
                const double2 v = *reinterpret_cast<const double2*>(p);
                fa[i] = v.x;
                fb[i] = v.y;
            } else {
                fa[i] = p[0];
                fb[i] = p[1];
            }
        }
        bad |= (!wall_a && any_bad(fa)) | (!wall_b && any_bad(fb));
        collide_pair<FORCED>(fa, fb, a);
        const bool wa = !wall_a && !(y >= iv.x && y < iv.y), wb = !wall_b && !(y + 1 >= iv.x && y + 1 < iv.y);
        if (wa && wb) {
#pragma unroll
            for (int i = 0; i < Q; ++i) {
                double* p = a.f + i * L.plane + L.at(gx + cxi(i), y + cyi(i));
                if (cyi(i) == 0) {
                    *reinterpret_cast<double2*>(p) = make_double2(fa[i], fb[i]);
                } else {
                    p[0] = fa[i];
                    p[1] = fb[i];
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < Q; ++i) {
                double* p = a.f + i * L.plane + L.at(gx + cxi(i), y + cyi(i));
                if (wa) p[0] = fa[i];
                if (wb) p[1] = fb[i];
            }
        }
    }
    if (bad) atomicMin(a.first_bad, a.bad_iter);
}

// One cell per thread: any ny.
template <bool ODD, bool FIRST>
__global__ void __launch_bounds__(256) k_aa_scalar(AaArgs a) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= L.ny) return;
    if (a.skip_rows && (y == 0 || y == L.ny - 1)) return;
    bool bad = false;
    for (int x = a.x_begin + blockIdx.y; x < a.x_end; x += gridDim.y) {
        const int gx = x + 1;
        const int4 iv = column_run(a, x);
        if (y >= iv.z && y < iv.w) continue;
        const bool solid = (y >= iv.x && y < iv.y);
        double f[Q];
#pragma unroll
        for (int i = 0; i < Q; ++i)
            f[i] = ODD ? a.f[oppi(i) * L.plane + L.at(gx - cxi(i), y - cyi(i))] : a.f[i * L.plane + L.at(gx, y)];
        if (!FIRST) bad |= any_bad(f);
        if (solid) continue;
        collide(f, a);
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            if (ODD)
                a.f[i * L.plane + L.at(gx + cxi(i), y + cyi(i))] = f[i];
            else
                a.f[oppi(i) * L.plane + L.at(gx, y)] = f[i];
        }
    }
    if (bad) atomicMin(a.first_bad, a.bad_iter);
}

// ------------------------------------------------------------------------------------------
// Fix-up after the E-step bulk launch: ring cells (in place, from their untouched inputs) and the
// reset of every solid cell to w.
__global__ void __launch_bounds__(128) k_aa_fix_even(AaArgs a, BcArgs b, const int2* __restrict__ ring, int n_ring,
                                                     const int2* __restrict__ solids, int n_solid) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < n_ring) {
        const int2 c = ring[idx];
        double* p = a.f + L.at(c.x + 1, c.y);
        double f[Q];
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = p[i * L.plane];
        if (!a.first) {
            double rb, uo;
            bc_rules(f, c.x, c.y, L, b, rb, uo);
            if (any_bad(f)) atomicMin(a.first_bad, a.bad_iter);
        }
        collide(f, a);
#pragma unroll
        for (int i = 0; i < Q; ++i) p[oppi(i) * L.plane] = f[i];
    } else if (idx - n_ring < n_solid) {
        const int2 c = solids[idx - n_ring];
        double* p = a.f + L.at(c.x + 1, c.y);
#pragma unroll
        for (int i = 0; i < Q; ++i) p[i * L.plane] = b.w[i];
    }
}

// Fix-up after the O-step bulk launch: ring cells (pull, rule, collide, push inside the domain
// only, keep all nine values in ring_out) and the constant fill of the slots nobody pushes to.
__global__ void __launch_bounds__(128) k_aa_fix_odd(AaArgs a, BcArgs b, const int2* __restrict__ ring, int n_ring,
                                                    const AaFill* __restrict__ fills, int n_fill,
                                                    double* __restrict__ ring_out, int open_x, int open_y) {
    pdl_wait();
    pdl_release();
    const Layout& L = a.L;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < n_ring) {
        const int2 c = ring[idx];
        const int gx = c.x + 1, y = c.y;
        double f[Q];
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = a.f[oppi(i) * L.plane + L.at(gx - cxi(i), y - cyi(i))];
        double rb, uo;
        bc_rules(f, c.x, y, L, b, rb, uo);
        if (any_bad(f)) atomicMin(a.first_bad, a.bad_iter);
        collide(f, a);
        double* out = ring_out + (long long)ring_slot(c.x, y, L) * Q;
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            out[i] = f[i];
            const int tx = c.x + cxi(i), ty = y + cyi(i);
            // open_x: bit 0 = the west edge is open (periodic, or a neighbouring slab takes what is pushed across it), bit 1 = east
            const bool ok_x = tx < 0 ? (open_x & 1) != 0 : (tx >= L.lnx ? (open_x & 2) != 0 : true);
            const bool ok = ok_x && (open_y || (ty >= 0 && ty < L.ny));
            if (ok) a.f[i * L.plane + L.at(tx + 1, ty)] = f[i];
        }
    } else if (idx - n_ring < n_fill) {
        const AaFill e = fills[idx - n_ring];
        a.f[e.off] = e.kind == 0 ? b.w[e.i] : (e.kind == 1 ? 0.0 : b.e[e.i]);
    }
}

// Reverse wrap after an O-step in a periodic direction: what was pushed into a ghost line belongs
// to the interior line at the opposite edge.
__global__ void k_aa_unwrap(double* __restrict__ f, Layout L, int do_x, int do_y, int rows_open) {
    pdl_wait();
    pdl_release();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (do_x) {
        const int y = t - 1;  // -1 .. ny when the rows are open (periodic y), else 0 .. ny-1
        const bool in = rows_open ? (y <= L.ny) : (y >= 0 && y < L.ny);
        if (in) {
            const int east[3] = {1, 5, 8}, west[3] = {3, 6, 7};
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                f[east[k] * L.plane + L.at(1, y)] = f[east[k] * L.plane + L.at(L.lnx + 1, y)];
                f[west[k] * L.plane + L.at(L.lnx, y)] = f[west[k] * L.plane + L.at(0, y)];
            }
        }
    }
    if (do_y && t >= 1 && t <= L.lnx) {  // interior columns (the x stage ran in an earlier launch)
        const int north[3] = {2, 5, 6}, south[3] = {4, 7, 8};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            f[north[k] * L.plane + L.at(t, 0)] = f[north[k] * L.plane + L.at(t, L.ny)];
            f[south[k] * L.plane + L.at(t, L.ny - 1)] = f[south[k] * L.plane + L.at(t, -1)];
        }
    }
}

// x-slabs: the two wraps of the periodic case go ACROSS GPUs, as plain stores into the neighbour's memory (CUDA IPC peer
// memory over NVLink) followed by the step-counter hand-shake of lbm_device.cuh.
//   forward (after an E-step): my edge columns, all nine reversed slots, into the neighbours' ghost columns -- what
//                              their O-step pulls across the face;
//   reverse (after an O-step): what my cells pushed into MY ghost columns belongs to the neighbours' edge columns
//                              (slots 1,5,8 eastwards, 3,6,7 westwards); their O-step touches none of those slots.
__global__ void __launch_bounds__(256) k_aa_halo(const double* __restrict__ f, Layout L, int reverse, int rows_open, P2pArgs px) {
    pdl_wait();
    pdl_release();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = rows_open ? t - 1 : t;
    const bool in = rows_open ? (y <= L.ny) : (y < L.ny);
    if (in) {
        if (!reverse) {
#pragma unroll
            for (int i = 0; i < Q; ++i) {
                if (px.peer_dst_east) px.peer_dst_east[i * L.plane + L.at(0, y)] = f[i * L.plane + L.at(L.lnx, y)];
                if (px.peer_dst_west) px.peer_dst_west[i * L.plane + L.at(L.lnx + 1, y)] = f[i * L.plane + L.at(1, y)];
            }
        } else {
            const int east[3] = {1, 5, 8}, west[3] = {3, 6, 7};
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                if (px.peer_dst_east) px.peer_dst_east[east[k] * L.plane + L.at(1, y)] = f[east[k] * L.plane + L.at(L.lnx + 1, y)];
                if (px.peer_dst_west) px.peer_dst_west[west[k] * L.plane + L.at(L.lnx, y)] = f[west[k] * L.plane + L.at(0, y)];
            }
        }
    }
    p2p_block_end(px, gridDim.x);
}

// Ghost ring of the single buffer: reversed constants on non-periodic edges.
__global__ void k_aa_ghosts(double* __restrict__ f, Layout L, BcArgs b, int west_zero, int east_zero) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < L.ny) {
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            f[oppi(i) * L.plane + L.at(0, t)] = west_zero ? 0.0 : b.e[i];
            f[oppi(i) * L.plane + L.at(L.lnx + 1, t)] = east_zero ? 0.0 : b.e[i];
        }
    }
    if (t < L.lnx + 2) {
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            f[oppi(i) * L.plane + L.at(t, -1)] = b.e[i];
            f[oppi(i) * L.plane + L.at(t, L.ny)] = b.e[i];
        }
    }
}

// ------------------------------------------------------------------------------------------
// Observers.
__device__ __forceinline__ bool solid_at(const AaObserve& o, int x, int y) { return o.mask[o.L.at(x + 1, y)] != 0; }

// post-collision populations of the last iteration (the reference's f_next) of an interior cell
__device__ __forceinline__ void aa_next(const AaObserve& o, int x, int y, double f[Q]) {
    const Layout& L = o.L;
    if (solid_at(o, x, y)) {
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = o.bc.w[i];
        return;
    }
    if (o.phase == 1) {
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = o.f[oppi(i) * L.plane + L.at(x + 1, y)];
    } else if (is_ring(x, y, L, o.bc)) {
        const double* r = o.ring_out + (long long)ring_slot(x, y, L) * Q;
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = r[i];
    } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = o.f[i * L.plane + L.at(x + 1 + cxi(i), y + cyi(i))];
    }
}

// the reference's f_current (streamed + boundary-treated) of an interior cell
__device__ __forceinline__ void aa_current(const AaObserve& o, int x, int y, double f[Q], double& rho_bc, double& u_out) {
    const Layout& L = o.L;
    const bool solid = solid_at(o, x, y);
    if (!o.cur_is_next) {  // straight after initialise / upload: the buffer IS f_current
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = o.f[i * L.plane + L.at(x + 1, y)];
        return;
    }
    if (o.phase == 1) {
#pragma unroll
        for (int i = 0; i < Q; ++i) f[i] = o.f[oppi(i) * L.plane + L.at(x + 1 - cxi(i), y - cyi(i))];
    } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            double v = o.f[i * L.plane + L.at(x + 1, y)];
            if (solid && i == 0) v = o.bc.w[0];  // its own rest population never left w
            if (solid && i > 0) {  // nobody filled the slots of a solid cell: rebuild what it would have pulled
                const int nx_ = x - cxi(i), ny_ = y - cyi(i);
                const bool out_x = (nx_ < 0 && !o.open_w) || (nx_ >= L.lnx && !o.open_e);
                const bool out_y = !o.periodic_y && (ny_ < 0 || ny_ >= L.ny);
                if (out_x || out_y)
                    v = out_y ? o.bc.e[i] : 0.0;  // S/N ghost rows and corners: eq(1,u_in,0); W/E columns: 0 (F4)
                else if (o.mask[L.at(nx_ + 1, ny_)])
                    v = o.bc.w[i];
            }
            f[i] = v;
        }
    }
    if (solid)
        reverse(f);
    else
        bc_rules(f, x, y, L, o.bc, rho_bc, u_out);
}

__device__ __forceinline__ void aa_macros_cell(const AaObserve& o, int x, int y, double& rho, double& ux, double& uy) {
    const Layout& L = o.L;
    const bool solid = solid_at(o, x, y);
    if (o.fresh) {
        rho = 1.0;
        uy = 0.0;
        ux = solid ? 0.0 : (o.shear_wave ? o.u0 * sin(2.0 * 3.14159265358979323846 * (double)y / (double)L.ny) : o.u0);  // Grid::initialise(inlet_u)
        return;
    }
    if (solid) {
        rho = 1.0;
        ux = 0.0;
        uy = 0.0;
        return;
    }
    double f[Q], rb = 0.0, uo = 0.0;
    if (!o.cur_is_next) {
        aa_current(o, x, y, f, rb, uo);
        const Moments m = moments(f);
        rho = m.rho; ux = m.ux; uy = m.uy;
        return;
    }
    // The last collision stored the moments of the state it read; density and momentum are
    // collision invariants (the body-force term adds F/tau of momentum), so they are recovered
    // from its output.  Equal to the reference's arrays to rounding (<= 1e-15), not bit for bit:
    // the one observable the single-buffer variant cannot keep exactly.
    aa_next(o, x, y, f);
    double r = 0.0, jx = 0.0, jy = 0.0;
#pragma unroll
    for (int i = 0; i < Q; ++i) {
        r += f[i];
        jx += cxi(i) * f[i];
        jy += cyi(i) * f[i];
    }
    rho = r;
    ux = (jx - o.Fx * o.tau_inv) / r;
    uy = (jy - o.Fy * o.tau_inv) / r;
    const bool on_in = o.bc.inlet && x == 0, on_out = o.bc.outlet && x == L.lnx - 1;
    if (on_in || on_out) {
        aa_current(o, x, y, f, rb, uo);
        if (on_in) { rho = rb; ux = o.bc.u_in; uy = 0.0; }
        if (on_out) { rho = 1.0; ux = uo; uy = 0.0; }
    }
}

__global__ void __launch_bounds__(256) k_aa_macros(AaObserve o, double* __restrict__ rho, double* __restrict__ ux,
                                                   double* __restrict__ uy) {
    __shared__ double t[3][32][33];
    const Layout& L = o.L;
    const int x0 = blockIdx.y * 32, y0 = blockIdx.x * 32;
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int x = x0 + k, y = y0 + threadIdx.x;
        if (x < L.lnx && y < L.ny) {
            double r, u, v;
            aa_macros_cell(o, x, y, r, u, v);
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

constexpr int EX_TX = 16, EX_TY = 32;

__global__ void __launch_bounds__(256) k_aa_export(AaObserve o, int which, double* __restrict__ aos, int row0, int rows) {
    __shared__ double t[Q][EX_TX][EX_TY + 1];
    const Layout& L = o.L;
    const int tnx = L.lnx + 2, tny = min(L.ny + 2, row0 + rows);
    const int gx0 = blockIdx.y * EX_TX, gy0 = row0 + blockIdx.x * EX_TY;
    for (int c = threadIdx.x; c < EX_TX * EX_TY; c += blockDim.x) {
        const int xl = c / EX_TY, yl = c % EX_TY;
        const int gx = gx0 + xl, gy = gy0 + yl;
        if (gx >= tnx || gy >= tny) continue;
        const int x = gx - 1, y = gy - 1;
        const bool ghost = (x < 0 || x >= L.lnx || y < 0 || y >= L.ny);
        const bool want_current = (which == 0) || !o.cur_is_next;
        double f[Q];
        if (ghost) {
            // f_current ghosts: never written after initialise.  f_next ghosts: the F4 convention
            // (periodic extensions: the wrapped image is not exported, the constants are).
            const bool col = (y >= 0 && y < L.ny);
            const bool zero = !want_current && col && ((x < 0 && o.west_zero) || (x >= L.lnx && o.east_zero));
#pragma unroll
            for (int i = 0; i < Q; ++i) f[i] = zero ? 0.0 : o.bc.e[i];
        } else if (want_current) {
            double rb, uo;
            aa_current(o, x, y, f, rb, uo);
        } else {
            aa_next(o, x, y, f);
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

// Grid::check_stability of the current f_current (what the next step would load), store-less.
__global__ void __launch_bounds__(256) k_aa_check(AaObserve o, int* first_bad, int bad_iter) {
    const Layout& L = o.L;
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= L.ny) return;
    bool bad = false;
    for (int x = blockIdx.y; x < L.lnx; x += gridDim.y) {
        double f[Q], rb, uo;
        aa_current(o, x, y, f, rb, uo);
        bad |= any_bad(f);
    }
    if (bad) atomicMin(first_bad, bad_iter);
}

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

}  // namespace

// ------------------------------------------------------------------------------------------
cudaError_t launch_aa_bulk(bool odd, const AaArgs& a, cudaStream_t s) {
    const int ncols = a.x_end - a.x_begin;
    if (ncols <= 0) return cudaSuccess;
    const int gy = ncols < 65535 ? ncols : 65535;
    cudaError_t e = cudaSuccess;
    if (a.L.ny % 2 == 0 && a.variant != BULK_SCALAR) {
        dim3 grid(cdiv(a.L.ny / 2, 128), gy);
        if (odd) e = a.forced ? launch_chain(k_aa_odd_vec2<true>, grid, dim3(128), s, a) : launch_chain(k_aa_odd_vec2<false>, grid, dim3(128), s, a);
        else if (a.first) e = a.forced ? launch_chain(k_aa_even_vec2<true, true>, grid, dim3(128), s, a) : launch_chain(k_aa_even_vec2<true, false>, grid, dim3(128), s, a);
        else e = a.forced ? launch_chain(k_aa_even_vec2<false, true>, grid, dim3(128), s, a) : launch_chain(k_aa_even_vec2<false, false>, grid, dim3(128), s, a);
    } else {
        dim3 grid(cdiv(a.L.ny, 256), gy);
        if (odd) e = launch_chain(k_aa_scalar<true, false>, grid, dim3(256), s, a);
        else if (a.first) e = launch_chain(k_aa_scalar<false, true>, grid, dim3(256), s, a);
        else e = launch_chain(k_aa_scalar<false, false>, grid, dim3(256), s, a);
    }
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_aa_fix_even(const AaArgs& a, const BcArgs& b, const int2* ring, int n_ring, const int2* solids,
                               int n_solid, cudaStream_t s) {
    const long long n = (long long)n_ring + n_solid;
    if (n == 0) return cudaSuccess;
    return launch_chain(k_aa_fix_even, dim3(cdiv(n, 128)), dim3(128), s, a, b, ring, n_ring, solids, n_solid);
}

cudaError_t launch_aa_fix_odd(const AaArgs& a, const BcArgs& b, const int2* ring, int n_ring, const AaFill* fills,
                              int n_fill, double* ring_out, int open_x, int open_y, cudaStream_t s) {
    const long long n = (long long)n_ring + n_fill;
    if (n == 0) return cudaSuccess;
    return launch_chain(k_aa_fix_odd, dim3(cdiv(n, 128)), dim3(128), s, a, b, ring, n_ring, fills, n_fill, ring_out, open_x, open_y);
}

cudaError_t launch_aa_unwrap(double* f, const Layout& L, int do_x, int do_y, cudaStream_t s) {
    cudaError_t e = cudaSuccess;
    if (do_x) e = launch_chain(k_aa_unwrap, dim3(cdiv(L.ny + 2, 256)), dim3(256), s, f, L, 1, 0, do_y);
    if (do_y && e == cudaSuccess) e = launch_chain(k_aa_unwrap, dim3(cdiv(L.lnx + 2, 256)), dim3(256), s, f, L, 0, 1, 0);
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_aa_halo(const double* f, const Layout& L, int reverse, int rows_open, const P2pArgs& px, cudaStream_t s) {
    return launch_chain(k_aa_halo, dim3(cdiv(L.ny + 2, 256)), dim3(256), s, f, L, reverse, rows_open, px);
}

cudaError_t launch_aa_ghosts(double* f, const Layout& L, const BcArgs& b, int west_zero, int east_zero, cudaStream_t s) {
    const int n = (L.ny > L.lnx + 2) ? L.ny : L.lnx + 2;
    k_aa_ghosts<<<cdiv(n, 256), 256, 0, s>>>(f, L, b, west_zero, east_zero);
    return cudaGetLastError();
}

cudaError_t launch_aa_macros(const AaObserve& o, double* rho, double* ux, double* uy, cudaStream_t s) {
    dim3 grid(cdiv(o.L.ny, 32), cdiv(o.L.lnx, 32));
    k_aa_macros<<<grid, dim3(32, 8), 0, s>>>(o, rho, ux, uy);
    return cudaGetLastError();
}

cudaError_t launch_aa_export(const AaObserve& o, int which, double* aos, int row0, int rows, cudaStream_t s) {
    dim3 grid(cdiv(rows, EX_TY), cdiv(o.L.lnx + 2, EX_TX));
    k_aa_export<<<grid, 256, 0, s>>>(o, which, aos, row0, rows);
    return cudaGetLastError();
}

cudaError_t launch_aa_check(const AaObserve& o, int* first_bad, int bad_iter, cudaStream_t s) {
    dim3 grid(cdiv(o.L.ny, 256), o.L.lnx < 65535 ? o.L.lnx : 65535);
    k_aa_check<<<grid, 256, 0, s>>>(o, first_bad, bad_iter);
    return cudaGetLastError();
}

}  // namespace lbm
