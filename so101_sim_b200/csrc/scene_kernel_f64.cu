// Explicit instantiation of the scene pipeline kernels for double arithmetic (separate translation units build in parallel).
#include "scene_kernel.inl"
namespace so101 {
template int launch_scene_step<double>(const ArmSetT<double> &, const ArmSetT<double> &, const SceneModel<double> &, const StepCfg &, const EnvState<double> &, const PipeBuf<double> *, TierExec *, int, const float *, const so101_step_out &, cudaStream_t, KernelTimer *);
template void launch_scene_reset<double>(const StepCfg &, const EnvState<double> &, const uint8_t *, const so101_step_out &, cudaStream_t);
template size_t scene_smem_bytes<double>();
template void launch_settle_enter<double>(const EnvState<double> &, unsigned, cudaStream_t);
template void launch_settle_leave<double>(const EnvState<double> &, cudaStream_t);
template void launch_debug_overlap<double>(const double *, int, uint8_t *, cudaStream_t);
template void scene_dropcat<double>(int *);
}  // namespace so101
