// usv_dense_g8.cu — the one-plane, 8-disparities-per-thread variant of the sliding-window SAD kernel (usv_dense.cu).
#include "usv_dense_kernel.cuh"

namespace usv {

template DenseKernel dense_kernel<1, 8>(int, int, bool);

}  // namespace usv
