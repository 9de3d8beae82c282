// v5ela_launch.cuh — the fused kernel's __global__ entry and its launcher, written once and compiled twice: by v5ela.cu
// (namespace v5: the 4-threads-per-block shared-memory-transpose block stage) and by v5ela_mma.cu (namespace v5m, V5_MMA_BLOCKS=1: the
// tensor-core block stage). The C ABI (v5ela.cu) plans the launch (v5ela_host.h) and picks the build per handle, see
// v5ela_set_block_stage in v5ela.h.
#pragma once
#include <cuda_runtime.h>

#include "v5ela.h"
#include "v5ela_host.h"
#include "v5ela_workitem.cuh"

namespace V5_NS {

static_assert(sizeof(KParams) <= 4096, "kernel parameters must fit the 4 KB parameter bank");
static_assert(sizeof(Smem) <= (227 * 1024) / MIN_CTAS - 1024, "MIN_CTAS CTAs per SM must fit in shared memory");

template <bool FAST, bool TEXHIST, bool RAGGED = false>
__global__ void __launch_bounds__(NT, MIN_CTAS) ela_fused_kernel(const __grid_constant__ KParams p, int total_work)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    Smem &S = *reinterpret_cast<Smem *>(smem_raw);
    ThreadAcc acc_store[1];
    acc_store[0].phase = 0;
    if (threadIdx.x == 0) {
        mbar_init(reinterpret_cast<uint64_t *>(&S.full_bar[0]), 1);
        mbar_init(reinterpret_cast<uint64_t *>(&S.full_bar[1]), 1);
        mbar_init(reinterpret_cast<uint64_t *>(&S.done_bar), NT);
        mbar_init_fence();
    }
    __syncthreads();
    // Work items are drawn from a global ticket counter: no tail of idle CTAs whatever the batch size / CTA count ratio.
    for (;;) {
        if (threadIdx.x == 0) S.next_work = atomicAdd(p.ticket, 1u);
        __syncthreads();
        const int work = (int)S.next_work;
        if (work >= total_work) break;
        process_work_item<FAST, TEXHIST, RAGGED>(S, p, work, acc_store);         // ends with a CTA barrier: next_work may be rewritten
    }
}

// A sweep (v5ela_analyze_sweep): the ragged instantiation over its n x nq entries, each with its own quantisation tables and
// optional JPEG-ghost map. A kernel of its own, so that ela_fused_kernel's instantiations are left exactly as they are.
__global__ void __launch_bounds__(NT, MIN_CTAS) ela_sweep_kernel(const __grid_constant__ KParams p, int total_work)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    Smem &S = *reinterpret_cast<Smem *>(smem_raw);
    ThreadAcc acc_store[1];
    acc_store[0].phase = 0;
    if (threadIdx.x == 0) {
        mbar_init(reinterpret_cast<uint64_t *>(&S.full_bar[0]), 1);
        mbar_init(reinterpret_cast<uint64_t *>(&S.full_bar[1]), 1);
        mbar_init(reinterpret_cast<uint64_t *>(&S.done_bar), NT);
        mbar_init_fence();
    }
    __syncthreads();
    for (;;) {
        if (threadIdx.x == 0) S.next_work = atomicAdd(p.ticket, 1u);
        __syncthreads();
        const int work = (int)S.next_work;
        if (work >= total_work) break;
        process_work_item<false, false, true, true>(S, p, work, acc_store);
    }
}

// once per device: opt in to the dynamic shared memory the kernels need
cudaError_t prepare()
{
    cudaError_t e = cudaFuncSetAttribute(ela_fused_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ela_fused_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ela_fused_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ela_fused_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ela_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
    return e;
}

// Launches instantiation `inst` (v5plan::choose_instantiation) over the `total` work items of the plan p, on at most max_ctas
// persistent CTAs; p.ticket must be zeroed before on the same stream, and a ragged plan's frame table uploaded. ev_start / ev_stop
// (optional) are recorded right around the kernel. Returns 0 or a positive cudaError_t.
int launch(const KParams &p, int inst, long long total, int max_ctas, cudaStream_t st, cudaEvent_t ev_start, cudaEvent_t ev_stop)
{
    const int grid = total < max_ctas ? (int)total : max_ctas;
    if (ev_start) cudaEventRecord(ev_start, st);
    if (inst == v5plan::INST_SWEEP) ela_sweep_kernel<<<grid, NT, sizeof(Smem), st>>>(p, (int)total);
    else if (inst == v5plan::INST_RAGGED) ela_fused_kernel<false, false, true><<<grid, NT, sizeof(Smem), st>>>(p, (int)total);
    else if (inst == V5ELA_INST_TEXHIST) ela_fused_kernel<false, true><<<grid, NT, sizeof(Smem), st>>>(p, (int)total);
    else if (inst == V5ELA_INST_FAST) ela_fused_kernel<true, false><<<grid, NT, sizeof(Smem), st>>>(p, (int)total);
    else ela_fused_kernel<false, false><<<grid, NT, sizeof(Smem), st>>>(p, (int)total);
    const cudaError_t e = cudaGetLastError();
    if (ev_stop) cudaEventRecord(ev_stop, st);
    return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace V5_NS
