// lbm_tb.cu -- the temporally blocked collide-stream kernels (lbm_tb.cuh has the thread program and the
// design notes) and the macro finishing kernel.  Compiled with -fmad=false like every other kernel.
#include <cstdlib>

#include "lbm_device.cuh"
#include "lbm_launch.cuh"
#include "lbm_tb.cuh"

namespace lbm {

namespace {

#ifndef TB_SKEW_THREADS
#define TB_SKEW_THREADS 512
#endif

// One block = B threads on B consecutive rows, marching through its chunk of columns.  In a multi-slab
// job the blocks of chunks 0 and 1 (the slab-edge columns) run the peer-memory hand-shake around their
// march: they are the first blocks of the grid, so the neighbours get their halo while the interior
// chunks are still being worked on.
template <int T, int B, bool FORCED, bool SKEW, bool FUSED>
__device__ __forceinline__ void tb_kernel_body(const TbArgs& a, int p2p) {
    extern __shared__ double ring[];
    pdl_wait();
    pdl_release();
    const bool edge_block = p2p && blockIdx.y < 2;
    if (edge_block) p2p_block_begin(a.px);
    tb_thread<T, B, FORCED, SKEW, FUSED>(a, ring, threadIdx.x, blockIdx.x, blockIdx.y);
    if (edge_block) p2p_block_end(a.px, gridDim.x * 2);
}

// Occupancy.  The skewed depth-2 march keeps two cells in registers (stage 1's loads in flight, the later stage being
// computed): 128 registers, 512 threads = 16 warps per SM -- measured: ANY spill costs more than the warps it buys (96
// registers / 20 warps: 42 800 MLUPS, 112 / 18: 53 300, 128 / 16: 65 800; the L1 left beside 148 KB of rings is
// tiny).  The one-column-lag march fits 80 registers (768 threads).  Depth 3: 512 threads too, 128 registers without a
// spill, and four blocks of 55 KB rings (lbm_tb.cuh) fit the 228 KB of an SM; the fused later stages (168 registers) 384.
template <int T, int B, bool FORCED, bool SKEW = true, bool FUSED = false>
__global__ void __launch_bounds__(B, (T == 3 ? (FUSED ? 384 : TB_SKEW_THREADS) : ((SKEW && T == 2) || T == 1 ? TB_SKEW_THREADS : 768)) / B)
    k_tb(const __grid_constant__ TbArgs a, int p2p) {
    tb_kernel_body<T, B, FORCED, SKEW, FUSED>(a, p2p);
}

// native [x*ny + y] -> interior row-major [y*lnx + x], 32 x 32 tiles through shared memory, with the
// overrides the reference's boundary pass applies AFTER the collision that stored the moments
// (include/LBMSolver.h:203-205 inlet, :232-234 outlet): functions of the newest buffer alone.
__global__ void __launch_bounds__(256) k_macros_finish(ObserveArgs o, const double* __restrict__ m_rho,
                                                       const double* __restrict__ m_ux, const double* __restrict__ m_uy,
                                                       double* __restrict__ rho, double* __restrict__ ux,
                                                       double* __restrict__ uy) {
    __shared__ double t[3][32][33];
    const Layout& L = o.L;
    const int x0 = blockIdx.y * 32, y0 = blockIdx.x * 32;
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int x = x0 + k, y = y0 + threadIdx.x;
        if (x < L.lnx && y < L.ny) {
            const long long g = (long long)x * L.ny + y;
            double r = m_rho[g], u = m_ux[g], v = m_uy[g];
            const bool on_in = o.bc.inlet && x == 0, on_out = o.bc.outlet && x == L.lnx - 1;
            if ((on_in || on_out) && !o.mask[L.at(x + 1, y)]) {
                double f[Q], rb = 0.0, uo = 0.0;
                current_from_next(o.cur, L, o.mask, o.bc, x, y, f, rb, uo);
                if (on_in) { r = rb; u = o.bc.u_in; v = 0.0; }
                if (on_out) { r = 1.0; u = uo; v = 0.0; }
            }
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

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

int env_int(const char* name, int dflt) {
    const char* v = std::getenv(name);
    return v ? std::atoi(v) : dflt;
}

template <int T, int B, bool FORCED, bool SKEW = true, bool FUSED = false>
cudaError_t launch_one(TbArgs a, bool p2p, cudaStream_t s) {
    using S = TbShape<T, B>;
    auto kern = k_tb<T, B, FORCED, SKEW, FUSED>;
    const size_t smem = (size_t)S::RING_DOUBLES * sizeof(double);
    static int slots = 0;  // resident blocks on the whole device, per instantiation
    if (!slots) {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        int per_sm = 0, dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, B, smem);
        if (e != cudaSuccess) return e;
        slots = (per_sm > 0 ? per_sm : 1) * (sms > 0 ? sms : 1);
    }
    const int lnx = a.L.lnx;
    const int strips = cdiv(a.L.ny, S::H);
    // ---- chunking --------------------------------------------------------------------------------
    a.edge_cols = 0;
    a.x_begin = 0;
    a.x_end = lnx;
    if (p2p) {  // multi-slab: the slab-edge columns are chunks 0 and 1
        a.edge_cols = lnx / 2 < 8 ? lnx / 2 : 8;
        a.x_begin = a.edge_cols;
        a.x_end = lnx - a.edge_cols;
    }
    const int ncols = a.x_end - a.x_begin;
    int chunks = 0;
    if (ncols > 0) {
        int xc = env_int("LBM_B200_TB_XC", 0);
        if (xc <= 0) {
            // 64 columns per chunk (3 % redundant columns at depth 2; measured best on a 4096 x 8192 slab: shorter
            // chunks keep the strips of a column in step and the tail of the grid short), fewer where that
            // leaves the device with less than two waves of resident blocks
            xc = 64;
            while (xc > 16 && (long long)strips * cdiv(ncols, xc) < 2LL * slots) xc /= 2;
        }
        a.xc = xc;
        chunks = cdiv(ncols, xc);
    } else {
        a.xc = 1;
    }
    dim3 grid(strips, chunks + (p2p ? 2 : 0));
    if (grid.y == 0) return cudaSuccess;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(B);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, a, p2p ? 1 : 0);
}

template <int T, int B>
cudaError_t launch_forced(const TbArgs& a, bool p2p, cudaStream_t s) {
    const bool forced = (a.Fx != 0.0 || a.Fy != 0.0);
    static const bool skew = env_int("LBM_B200_TB_SKEW", 1) != 0;
    if (T == 2 && !forced && !skew) return launch_one<T, B, false, false>(a, p2p, s);  // (the one-column-lag march, for A/B runs)
    static const bool fused = env_int("LBM_B200_TB_FUSED", 0) != 0;
    if (T == 3 && B == 128 && !forced && fused) return launch_one<T, B, false, true, true>(a, p2p, s);  // (experimental)
    return forced ? launch_one<T, B, true>(a, p2p, s) : launch_one<T, B, false>(a, p2p, s);
}

int block_threads() {
    static const int b = [] {
        const int v = env_int("LBM_B200_TB_B", 128);
        return v == 256 ? 256 : (v == 64 ? 64 : 128);
    }();
    return b;
}

}  // namespace

cudaError_t launch_tb(int depth, TbArgs a, bool p2p, cudaStream_t s) {
    const int b = block_threads();
    tb_fill_offsets(a);
    static const int pf = env_int("LBM_B200_TB_PF", 1), fast = env_int("LBM_B200_TB_FAST", 1);
    a.pf_dist = pf;
    a.fast_lane = fast;
    switch (depth) {
        case 1: return b == 128 ? launch_forced<1, 128>(a, p2p, s) : (b == 64 ? launch_forced<1, 64>(a, p2p, s) : launch_forced<1, 256>(a, p2p, s));
        case 2: return b == 128 ? launch_forced<2, 128>(a, p2p, s) : (b == 64 ? launch_forced<2, 64>(a, p2p, s) : launch_forced<2, 256>(a, p2p, s));
        case 3: return b == 128 ? launch_forced<3, 128>(a, p2p, s) : (b == 64 ? launch_forced<3, 64>(a, p2p, s) : launch_forced<3, 256>(a, p2p, s));
        default: return cudaErrorInvalidValue;
    }
}

// Whether a slab of this shape gives the marching blocks enough parallelism to beat the one-iteration kernels:
// at least two waves of resident blocks with 64-column chunks.  Small lattices (the reference's default 2048 x 512
// lives in L2 anyway) stay on the bulk kernels.
bool tb_worthwhile(const Layout& L) {
    const int b = block_threads();
    const long long blocks = (long long)cdiv(L.ny, b - 4) * cdiv(L.lnx, 64);
    return blocks >= 2LL * 148 * (TB_SKEW_THREADS / b);
}

int tb_rows_per_block(int depth) {
    const int b = block_threads();
    return depth == 1 ? b : b - 4;
}

size_t tb_shared_bytes(int depth) {
    const int b = block_threads();
    return (size_t)(depth - 1) * TB_RING_PLANES * b * sizeof(double);
}

cudaError_t launch_macros_finish(const ObserveArgs& o, const double* m_rho, const double* m_ux, const double* m_uy,
                                 double* rho, double* ux, double* uy, cudaStream_t s) {
    dim3 grid(cdiv(o.L.ny, 32), cdiv(o.L.lnx, 32));
    k_macros_finish<<<grid, dim3(32, 8), 0, s>>>(o, m_rho, m_ux, m_uy, rho, ux, uy);
    return cudaGetLastError();
}

}  // namespace lbm
