// tools/tb_occupancy.cu -- resident blocks per SM of the temporally blocked kernels, as launch_one sees them
// (cudaOccupancyMaxActiveBlocksPerMultiprocessor with the ring as dynamic shared memory).  Built with the library's
// flags so that the kernels have the library's registers:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -fmad=false -Xcompiler -ffp-contract=off \
//        tools/tb_occupancy.cu -o build/tb_occupancy && build/tb_occupancy
#include <cstdio>

#include "../highperformancecomputing-latticeboltzmannmethod_b200/csrc/lbm_tb.cu"

namespace {

template <int T, int B, bool FORCED, bool SKEW, bool FUSED>
bool report(const char* name) {
    auto kern = lbm::k_tb<T, B, FORCED, SKEW, FUSED>;
    const int smem = lbm::TbShape<T, B>::RING_DOUBLES * (int)sizeof(double);
    cudaFuncAttributes fa{};
    int per_sm = 0;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess ||
        cudaFuncGetAttributes(&fa, kern) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, B, smem) != cudaSuccess) {
        std::printf("%s: %s\n", name, cudaGetErrorString(cudaGetLastError()));
        return false;
    }
    std::printf("{\"kernel\": \"%s\", \"registers\": %d, \"local_bytes\": %zu, \"ring_bytes\": %d, \"blocks_per_sm\": %d, "
                "\"warps_per_sm\": %d}\n", name, fa.numRegs, fa.localSizeBytes, smem, per_sm, per_sm * B / 32);
    return true;
}

}  // namespace

int main() {
    cudaDeviceProp p{};
    cudaGetDeviceProperties(&p, 0);
    std::printf("{\"device\": \"%s\", \"sms\": %d, \"smem_per_sm\": %zu, \"smem_reserved_per_block\": %zu}\n", p.name,
                p.multiProcessorCount, p.sharedMemPerMultiprocessor, p.reservedSharedMemPerBlock);
    bool ok = report<3, 128, false, true, false>("k_tb<3,128,0,1,0>");
    ok = report<3, 128, true, true, false>("k_tb<3,128,1,1,0>") && ok;
    ok = report<3, 128, false, true, true>("k_tb<3,128,0,1,1>") && ok;
    ok = report<2, 128, false, true, false>("k_tb<2,128,0,1,0>") && ok;
    return ok ? 0 : 1;
}
