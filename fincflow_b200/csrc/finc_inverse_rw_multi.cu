// the multi-level register-window inverse (finc_inverse_rw.cuh: inverse_rw_multi_kernel), in its own translation
// unit so that it compiles next to the per-level instantiations
#include "finc_inverse_rw.cuh"

namespace finc {
namespace rw {

namespace {
auto multi_kernel() { return inverse_rw_multi_kernel<RwKind0, RwKind1, RwKind2>; }
}  // namespace

int multi_ctas_per_sm(size_t smem) {
    auto kern = multi_kernel();
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, kRwMultiWarps * 32, smem) != cudaSuccess) return 0;
    return n;
}

int launch_multi(const RwMultiArgs& m, int n_ctas, size_t smem, cudaStream_t st) {
    auto kern = multi_kernel();
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    return launch_kernel(kern, dim3((unsigned)n_ctas, 1, 1), kRwMultiWarps * 32, smem, st, m);
}

}  // namespace rw
}  // namespace finc
