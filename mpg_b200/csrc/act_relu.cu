// relu instantiations of the MLP kernels (see act_instances.cuh)
#define MPG_ACT_UNIT
#include "act_instances.cuh"

namespace mpg {
MPG_ACT_INSTANCES(, MPG_ACT_RELU)
bool wait_dbg_attach_relu(unsigned long long* dev_ptr) {
  return cudaMemcpyToSymbol(tc::g_wait_dbg, &dev_ptr, sizeof(dev_ptr)) == cudaSuccess;
}
}  // namespace mpg
