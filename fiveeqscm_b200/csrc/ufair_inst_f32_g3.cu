// the fused integrator's launchers and kernels for float, 3 gas(es): every alpha mode, loop and instantiated form
#include "ufair_kernel.cuh"
namespace ufair {
UFAIR_INSTANTIATE(float, 3)
}  // namespace ufair
