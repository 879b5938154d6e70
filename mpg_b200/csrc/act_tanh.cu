// tanh instantiations of the MLP kernels (mlp_kernels.cuh)
#include "mlp_kernels.cuh"

namespace mpg {
static constexpr MlpKernels tanh64 = MlpLaunch<64, MPG_ACT_TANH>::table(), tanh128 = MlpLaunch<128, MPG_ACT_TANH>::table(),
                            tanh256 = MlpLaunch<256, MPG_ACT_TANH>::table();
const MlpKernels& tanh_kernels(int hidden) { return hidden == 64 ? tanh64 : hidden == 128 ? tanh128 : tanh256; }
}  // namespace mpg
