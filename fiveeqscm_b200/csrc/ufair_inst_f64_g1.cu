// the fused integrator's launchers and kernels for double, 1 gas(es): every alpha mode, loop and instantiated form
#include "ufair_kernel.cuh"
namespace ufair {
UFAIR_INSTANTIATE(double, 1)
}  // namespace ufair
