// cloth_inst.cu - the step kernel for one scalar type (CLOTH_T), one compile-time grid width (CLOTH_INSTANTIATE_WC:
// 25, 64, or 0 = any width at run time) and the batch's or per-environment material (CLOTH_INSTANTIATE_PHYS 0 / 1).
// build.py compiles this file twelve times, in parallel.
#include <cstring>
#include "cloth_kernels.cuh"
