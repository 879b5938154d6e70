// relu instantiations of the MLP kernels (mlp_kernels.cuh)
#include "mlp_kernels.cuh"

namespace mpg {
static constexpr MlpKernels relu64 = MlpLaunch<64, MPG_ACT_RELU>::table(), relu128 = MlpLaunch<128, MPG_ACT_RELU>::table(),
                            relu256 = MlpLaunch<256, MPG_ACT_RELU>::table();
const MlpKernels& relu_kernels(int hidden) { return hidden == 64 ? relu64 : hidden == 128 ? relu128 : relu256; }
}  // namespace mpg
