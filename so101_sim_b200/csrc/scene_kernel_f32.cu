// Explicit instantiation of the scene pipeline kernels for float arithmetic (separate translation units build in parallel).
#include "scene_kernel.inl"
namespace so101 {
template int launch_scene_step<float>(const ArmSetT<float> &, const ArmSetT<double> &, const SceneModel<float> &, const StepCfg &, const EnvState<float> &, const PipeBuf<float> *, TierExec *, int, const float *, const so101_step_out &, cudaStream_t, KernelTimer *);
template void launch_scene_reset<float>(const StepCfg &, const EnvState<float> &, const uint8_t *, const so101_step_out &, cudaStream_t);
template size_t scene_smem_bytes<float>();
template void launch_settle_enter<float>(const EnvState<float> &, unsigned, cudaStream_t);
template void launch_settle_leave<float>(const EnvState<float> &, cudaStream_t);
template void launch_debug_overlap<float>(const double *, int, uint8_t *, cudaStream_t);
template void scene_dropcat<float>(int *);
}  // namespace so101
