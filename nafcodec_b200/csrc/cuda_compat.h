// cuda_compat.h -- the one place that decides between the real CUDA toolchain (product build: nvcc, sm_100a)
// and the CPU SIMT emulator used by the test tier (tests/emul, -DNAFGPU_EMULATE; never shipped).
#pragma once
#if defined(NAFGPU_EMULATE)
#include "cuda_emul.h"
#define NAF_LAUNCH(kernel, grid, block, smem, stream, ...) \
    emul::launch(dim3(grid), dim3(block), (smem), [=]() { kernel(__VA_ARGS__); })
#define NAF_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(emul::g_dyn_smem)
#define NAF_SET_MAX_SMEM(kernel, bytes) ((void)0)
// cooperative (grid-synchronising) kernels run as ONE CTA under the emulator, so a grid barrier is a CTA barrier
#define NAF_LAUNCH_COOP(kernel, grid, block, stream, arg) emul::launch(dim3(1), dim3(block), 0, [=]() { kernel(arg); })
#define NAF_GRID_SYNC() __syncthreads()
#else
#include <cuda_runtime.h>
#if defined(__CUDACC__)
#include <cooperative_groups.h>
#define NAF_GRID_SYNC() cooperative_groups::this_grid().sync()
#endif
// one by-value argument; all CTAs must be co-resident (grid <= occupancy x SMs)
#define NAF_LAUNCH_COOP(kernel, grid, block, stream, arg) \
    do { void* _args[] = {(void*)&(arg)}; cudaLaunchCooperativeKernel((const void*)kernel, dim3(grid), dim3(block), _args, 0, (stream)); } while (0)
#define NAF_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
// The attribute belongs to the function (per device), not to the launch: contexts on several host threads (pipeline lanes) launch
// the same kernels with job-dependent sizes, and a lane that LOWERED the limit between another lane's call here and its launch
// made that launch fail with "invalid argument".  The limit only ever grows.
#include <mutex>
#define NAF_SET_MAX_SMEM(kernel, bytes) do { \
    static std::mutex _m; static int _cur[64]; \
    int _d = 0; cudaGetDevice(&_d); \
    std::lock_guard<std::mutex> _g(_m); \
    if ((int)(bytes) > _cur[_d & 63]) { cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)); _cur[_d & 63] = (int)(bytes); } \
} while (0)
#define NAF_DYN_SMEM(type, name) extern __shared__ __align__(16) unsigned char _naf_dyn_smem[]; type* name = reinterpret_cast<type*>(_naf_dyn_smem)
#endif

// Optional per-stage CUDA events (nafgpu_job_run_profiled): mark() after the kernels of a stage.
struct StageEvents {
    cudaEvent_t* ev = nullptr;
    int n = 0, cap = 0;
    cudaStream_t st = 0;
    void mark() { if (ev && n < cap) cudaEventRecord(ev[n++], st); }
    // one extra interval around the dominant kernel alone (k_huf_decode_block, with its scout k_huf_scout), for the roofline figure
    cudaEvent_t kb = nullptr, ke = nullptr;
    bool k_used = false;
    void kernel_begin() { if (ev && kb) cudaEventRecord(kb, st); }
    void kernel_end() { if (ev && ke) { cudaEventRecord(ke, st); k_used = true; } }
};
