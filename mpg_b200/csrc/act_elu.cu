// elu instantiations of the MLP kernels (mlp_kernels.cuh)
#include "mlp_kernels.cuh"

namespace mpg {
static constexpr MlpKernels elu64 = MlpLaunch<64, MPG_ACT_ELU>::table(), elu128 = MlpLaunch<128, MPG_ACT_ELU>::table(),
                            elu256 = MlpLaunch<256, MPG_ACT_ELU>::table();
const MlpKernels& elu_kernels(int hidden) { return hidden == 64 ? elu64 : hidden == 128 ? elu128 : elu256; }
}  // namespace mpg
