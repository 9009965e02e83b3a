// explicit instantiation of the register-window adjoint solve (finc_inverse_adjoint_f32) for C = 1, 3x3 kernels
#include "finc_inverse_rw.cuh"
namespace finc {
namespace rw {
template int dispatch_ck<1, 3, true>(int, const RwArgs&, dim3, int, size_t, cudaStream_t);
}
}
