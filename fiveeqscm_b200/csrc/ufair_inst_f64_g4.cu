// the fused integrator's launchers and kernels for double, 4 gas(es): every alpha mode, loop and instantiated form,
// with FP64 and with float32 outputs
#include "ufair_kernel.cuh"
namespace ufair {
UFAIR_INSTANTIATE(double, 4)
UFAIR_INSTANTIATE_OUT(double, float, 4)  // float32 outputs (UFAIR_OUTTYPE_F32)
}  // namespace ufair
