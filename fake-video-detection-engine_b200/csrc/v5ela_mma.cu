// v5ela_mma.cu — second build of the fused kernel's device code, with the tensor-core block stage (v5ela_dctmma.cuh): everything of
// v5ela_device.cuh / v5ela_workitem.cuh / v5ela_launch.cuh again, in namespace v5m with V5_MMA_BLOCKS = 1. v5ela.cu holds the C ABI and
// the other build; v5ela_set_block_stage (include/v5ela.h) chooses between them per handle.
#define V5_NS v5m
#define V5_MMA_BLOCKS 1
#include "v5ela_launch.cuh"
