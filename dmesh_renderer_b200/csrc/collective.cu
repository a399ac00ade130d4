// collective.cu -- the one collective of the multi-view step (SURVEY.md 8e) as a hand-written kernel over
// NVLink 5 / NVSwitch: all-reduce(SUM) of the packed scene gradients [dL_dverts | dL_dvcolor | dL_dfopacity]
// with the reduction done INSIDE the switch (NVLS multimem instructions).
//
// The reference has no distributed code at all.  The packed gradient buffer lives in symmetric memory
// (torch.distributed._symmetric_memory: every rank maps every peer's copy and a MULTICAST address that
// aliases all copies).  Rank r owns slice r of the buffer:
//     multimem.ld_reduce.add.v4.f32  [mc + i]   -> the switch returns the sum of the 16 bytes over all ranks
//     multimem.st.v4.f32             [mc + i]   -> the switch writes the sum into every rank's copy
// so every float crosses each GPU's NVLink port once in each direction (2 x n/W x (W-1)/W ... ~n bytes per
// port in total) and no GPU ever reads W copies.  The cross-GPU barriers before (all ranks' gradients complete)
// and after (all slices broadcast) run inside the same kernel, on flags in symmetric memory (see
// nvls_allreduce_sum_fused_kernel).  Measured on 8 x B200: 15 MB in [see profiles/README.md].
#include "common.cuh"
#include "../../include/dmesh_b200.h"

namespace dmr {

__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc)
{
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
    return v;
}
__device__ __forceinline__ void multimem_st(float* mc, float4 v)
{
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Reduce + broadcast the float4 elements i, i + stride, ... < end of this rank's slice.  DMR_NVLS_UNROLL vectors are
// requested before the first one is stored back; the unrolled body is predicated (no one-at-a-time tail loop).
// The depth does not matter beyond 8: 76 MB on 8 x B200 take 228 / 234 / 241 us with 8 / 16 / 32 vectors in flight per
// thread (NCCL: 309 us), 15 MB 60 / 60 / 61 us -- the transfer is bound by the switch path (each GPU's port moves
// ~85 MB in each direction: ~375 GB/s), not by latency.
constexpr int DMR_NVLS_UNROLL = 8;
__device__ __forceinline__ void nvls_reduce_slice(float* __restrict__ mc, size_t i, size_t end, size_t stride)
{
    for (; i < end; i += DMR_NVLS_UNROLL * stride) {
        float4 v[DMR_NVLS_UNROLL];
#pragma unroll
        for (int k = 0; k < DMR_NVLS_UNROLL; k++)
            if (i + k * stride < end) v[k] = multimem_ld_reduce_add(mc + 4 * (i + k * stride));
#pragma unroll
        for (int k = 0; k < DMR_NVLS_UNROLL; k++)
            if (i + k * stride < end) multimem_st(mc + 4 * (i + k * stride), v[k]);
    }
}

// ---------------------------------------------------------------------------
// The reduction with the two cross-GPU barriers INSIDE the kernel (no extra launches): separate
// signal-pad barriers cost more than the transfer itself (15 MB on 8 GPUs: 63 us with two barrier kernels
// around a ~10 us reduction).
//   n4 = number of float4 of the whole buffer (the caller pads to a multiple of world); persistent grid (one wave).
//   peer_flags[r] -> rank r's flag array in symmetric memory (W + 2 words used: word s = last epoch value
//                    signalled by rank s); local_ctl: [0] = "go" flag, [1] = finished-CTA counter (this GPU only).
//   epoch e = 1, 2, 3, ... (host counter, identical on all ranks); flag values only grow, nothing is reset.
// All CTAs are co-resident (grid <= number of SMs, one CTA per SM), so spinning inside the grid is safe.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) { uint32_t v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

__device__ __forceinline__ void cross_gpu_barrier(uint32_t* const* peer_flags, int rank, int world, uint32_t value)
{
    // one thread per peer: tell peer t that this rank has arrived, then wait for peer t's arrival here
    const int t = threadIdx.x;
    if (t < world) {
        st_release_sys(peer_flags[t] + rank, value);
        const uint32_t* mine = peer_flags[rank] + t;
        while ((int32_t)(ld_acquire_sys(mine) - value) < 0) { }
    }
}

__global__ void __launch_bounds__(512) nvls_allreduce_sum_fused_kernel(float* __restrict__ mc, size_t n4, int rank, int world,
                                                                      uint32_t* const* __restrict__ peer_flags,
                                                                      uint32_t* __restrict__ local_ctl, uint32_t epoch)
{
    // ---- barrier 1: every rank's gradient kernels have finished (each rank's kernel starts after them in
    //      stream order); CTA 0 talks to the peers, the other CTAs wait for its "go"
    if (blockIdx.x == 0) {
        cross_gpu_barrier(peer_flags, rank, world, 2 * epoch - 1);
        __syncthreads();
        if (threadIdx.x == 0) st_release_gpu(local_ctl + 0, epoch);
    } else {
        if (threadIdx.x == 0) while ((int32_t)(ld_acquire_gpu(local_ctl + 0) - epoch) < 0) { }
        __syncthreads();
    }

    // ---- reduce + broadcast this rank's slice inside the switch
    const size_t per = n4 / (size_t)world;
    const size_t begin = per * (size_t)rank, end = begin + per;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    nvls_reduce_slice(mc, i, end, stride);

    // ---- barrier 2: all slices have been broadcast.  The last CTA of this GPU to finish (its stores fenced
    //      at system scope) signals the peers and waits for theirs; the kernel -- and with it everything behind
    //      it in the stream -- completes only then.
    __shared__ bool s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        s_last = atomicAdd(local_ctl + 1, 1u) + 1u == gridDim.x * epoch;
    }
    __syncthreads();
    if (s_last) {
        __threadfence_system();
        cross_gpu_barrier(peer_flags, rank, world, 2 * epoch);
    }
}

}  // namespace dmr

using namespace dmr;

// grid size of the fused kernel for a buffer of n_floats: fixed per buffer (the finished-CTA counter relies on it)
static unsigned nvls_fused_blocks(size_t per)
{
    size_t blocks = (per + 512 - 1) / 512;
    if (blocks > 128) blocks = 128;   // co-resident with room to spare on 148 SMs (one 512-thread CTA per SM)
    return blocks ? (unsigned)blocks : 1u;
}

extern "C" int dmr_nvls_allreduce_sum_f32_fused(void* multicast_ptr, size_t n_floats, int rank, int world,
                                                void* const* peer_flag_ptrs_dev, void* local_ctl, unsigned epoch,
                                                dmr_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!multicast_ptr || !peer_flag_ptrs_dev || !local_ctl) { set_error("null pointer"); return DMR_EINVAL; }
    if (world <= 0 || world > 64 || rank < 0 || rank >= world || epoch == 0 || epoch >= (1u << 30)) { set_error("bad rank/world/epoch"); return DMR_EINVAL; }
    if (n_floats % (4 * (size_t)world) != 0) { set_error("n_floats must be a multiple of 4*world"); return DMR_EINVAL; }
    if (((uintptr_t)multicast_ptr & 15) != 0) { set_error("multicast_ptr must be 16-byte aligned"); return DMR_EINVAL; }
    const size_t n4 = n_floats / 4, per = n4 / (size_t)world;
    count_launch(1);
    nvls_allreduce_sum_fused_kernel<<<nvls_fused_blocks(per), 512, 0, stream>>>(
        static_cast<float*>(multicast_ptr), n4, rank, world, reinterpret_cast<uint32_t* const*>(peer_flag_ptrs_dev),
        static_cast<uint32_t*>(local_ctl), epoch);
    DMR_LAUNCH_CHECK("nvls_allreduce_sum_fused_kernel");
    return DMR_OK;
}
