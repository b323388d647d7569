// the fused integrator's launchers and kernels for double, 3 gas(es): every alpha mode, loop and instantiated form,
// with FP64 and with float32 outputs
#include "ufair_kernel.cuh"
namespace ufair {
UFAIR_INSTANTIATE(double, 3)
UFAIR_INSTANTIATE_OUT(double, float, 3)  // float32 outputs (UFAIR_OUTTYPE_F32)
}  // namespace ufair
