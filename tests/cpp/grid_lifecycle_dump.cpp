// tests/cpp/grid_lifecycle_dump.cpp -- call sequences of the C++ drop-in API that do not start at iteration 0, dumped
// for a comparison with the CPU oracle (tests/test_gpu_lifecycle.py).  Lattice 48 x 20, output frequency 5,
// cylinder radius 0.15, as tests/cpp/grid_api_dump.cpp.
//   grid_lifecycle_dump edit    <flags> <variant> <depth> <outdir>
//       7 iterations, then writes through Grid::f_current and (A-B buffers only) Grid::f_next -- a fluid cell, a solid
//       cell, an S ghost row entry and an N corner -- and 9 more iterations; both edits reach the engine in one flush.
//   grid_lifecycle_dump restart <flags> <variant> <depth> <outdir>
//       Solver::run to iteration 13 (not an output step), save_checkpoint, then a second Solver loads it and runs to 31.
// Writes f_current.bin, f_next.bin, rho.bin, ux.bin, uy.bin (and forces.csv in the working directory).
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "LBMConfig.h"
#include "LBMIO.h"
#include "LBMSolver.h"

static void write_doubles(const std::string& path, const std::vector<double>& v) {
    std::FILE* f = std::fopen(path.c_str(), "wb");
    std::fwrite(v.data(), sizeof(double), v.size(), f);
    std::fclose(f);
}

static void configure(LBM::Solver& solver, int variant, int depth) {
    lbm_handle h = solver.get_grid().handle();
    if (lbm_set_kernel_variant(h, variant) != LBM_OK || lbm_set_pass_depth(h, depth) != LBM_OK)
        throw std::runtime_error(lbm_last_error(h));
}

static void dump(const LBM::Grid& c, const std::string& out) {
    std::vector<double> fc((size_t)c.total_nx() * c.total_ny() * LBM::Q), fn(fc.size());
    size_t k = 0;
    for (int gy = 0; gy < c.total_ny(); ++gy)
        for (int gx = 0; gx < c.total_nx(); ++gx)
            for (int i = 0; i < LBM::Q; ++i, ++k) {
                fc[k] = c.f_current(gx, gy, i);
                fn[k] = c.f_next(gx, gy, i);
            }
    std::vector<double> rho((size_t)c.local_nx() * c.local_ny()), ux(rho.size()), uy(rho.size());
    k = 0;
    for (int y = 0; y < c.local_ny(); ++y)
        for (int x = 0; x < c.local_nx(); ++x, ++k) {
            rho[k] = c.rho(x, y);
            ux[k] = c.ux(x, y);
            uy[k] = c.uy(x, y);
        }
    write_doubles(out + "/f_current.bin", fc);
    write_doubles(out + "/f_next.bin", fn);
    write_doubles(out + "/rho.bin", rho);
    write_doubles(out + "/ux.bin", ux);
    write_doubles(out + "/uy.bin", uy);
}

int main(int argc, char** argv) {
    if (argc < 6) return 2;
    const std::string mode = argv[1];
    LBM::SimulationParams p;
    p.nx = 48;
    p.ny = 20;
    p.output_frequency = 5;
    p.cylinder_radius = 0.15;
    p.flags = std::atoi(argv[2]);
    const int variant = std::atoi(argv[3]), depth = std::atoi(argv[4]);
    const std::string out = argv[5];
    const bool ab = (p.flags & LBM_FLAG_AA) == 0;
    try {
        if (mode == "edit") {
            p.num_timesteps = 16;
            LBM::Solver solver(p, false);
            configure(solver, variant, depth);
            solver.initialise();
            LBM::Grid& g = const_cast<LBM::Grid&>(solver.get_grid());
            double rows[8][5];
            int n_rows = 0;
            if (g.advance(7, &rows[0][0], 8, &n_rows) >= 0) return 1;
            g.f_current(3, 4, 1) *= 1.25;                 // fluid
            g.f_current(p.nx, p.ny, 8) *= 0.5;            // fluid, next to the outlet-top corner
            if (ab) {
                const int cx = p.get_cylinder_x(), cy = p.get_cylinder_y();
                g.f_next(cx + 1, cy + 1, 5) *= 1.5;       // the solid cell at the cylinder's centre
                g.f_next(10, 0, 2) += 0.001;              // S ghost row
                g.f_next(p.nx + 1, p.ny + 1, 7) *= 0.75;  // N-E corner
            }
            if (g.advance(9, &rows[0][0], 8, &n_rows) >= 0) return 1;
            dump(solver.get_grid(), out);
        } else if (mode == "restart") {
            {
                p.num_timesteps = 13;
                LBM::Solver first(p, false);
                configure(first, variant, depth);
                LBM::IOManager io;
                first.initialise();
                if (!first.run(io)) return 1;
                first.save_checkpoint(out + "/state.ckpt");
            }
            p.num_timesteps = 31;
            LBM::Solver second(p, false);
            configure(second, variant, depth);
            LBM::IOManager io;
            second.initialise();
            second.load_checkpoint(out + "/state.ckpt");
            if (!second.run(io)) return 1;
            dump(second.get_grid(), out);
        } else {
            return 2;
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "exception: %s\n", e.what());
        return 3;
    }
    return 0;
}
