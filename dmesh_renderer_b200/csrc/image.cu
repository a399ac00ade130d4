// image.cu -- per-pixel outputs of the image state that both renderers share in form: the alpha (coverage) image
// and the gradient with respect to the background colour; and the conversion of the per-(view, face) visibility
// statistics (FaceWeightAcc, common.cuh) into their output format.
//
// The forward passes composite colour = C + w * bg with a per-pixel background weight w:
//   tri: w = final_T (the transmittance after the last composited face, T < 1e-4 termination included);
//   tet: w = expf(final_log_T) on active pixels, 1 on inactive ones (numerical failure, shown as bg).
// alpha = 1 - w, and dL/dbg[c] = sum over views and pixels of w * dL_dcolor[c].  Neither kernel touches the render
// kernels' state: they read the image buffer after the last phase 2 of a forward call.
#include "common.cuh"
#include <algorithm>

namespace dmr {

template <bool TET>
__device__ __forceinline__ float bg_weight(const float* __restrict__ t, const uint8_t* __restrict__ active, size_t i)
{
    if constexpr (TET) return active[i] ? expf(t[i]) : 1.0f;
    else return t[i];
}

// alpha[i] = 1 - w[i]; tet: 1 - expf(final_log_T), bit-identical to 1 - T_cur of tet_march_fwd_kernel, 0 if inactive
template <bool TET>
__global__ void __launch_bounds__(256) alpha_kernel(size_t n, const float* __restrict__ t, const uint8_t* __restrict__ active,
                                                    float* __restrict__ alpha)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        if constexpr (TET) alpha[i] = active[i] ? 1.0f - expf(t[i]) : 0.0f;
        else alpha[i] = 1.0f - t[i];
    }
}

// Background gradient, fixed-order reduction (no float atomics: the same bits in every run and in both modes).
// Grid (nbx, B), nbx a function of B, W and H only: block (x, b) sums w * dL_dcolor over the pixels
// x*256 + tid + k*nbx*256 of view b, warp butterflies and the eight warp sums in warp order give its partial [3];
// bg_grad_finish_kernel adds the partials of all blocks in a fixed order.  About BG_BLOCKS blocks in all (four per SM),
// at least 1024 pixels per block.
constexpr unsigned BG_BLOCKS = 148 * 4;

template <bool TET>
__global__ void __launch_bounds__(256) bg_grad_partial_kernel(uint32_t HW, const float* __restrict__ t,
                                                              const uint8_t* __restrict__ active,
                                                              const float* __restrict__ dL_dcolor, float* __restrict__ partial)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ float s_part[8][3];
    const uint32_t b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* g = dL_dcolor + (size_t)b * 3 * HW;
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
    for (uint32_t pix = blockIdx.x * 256 + tid; pix < HW; pix += gridDim.x * 256) {
        const float w = bg_weight<TET>(t, active, (size_t)b * HW + pix);
        s0 += w * g[pix]; s1 += w * g[HW + pix]; s2 += w * g[2 * (size_t)HW + pix];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) { s_part[warp][0] = s0; s_part[warp][1] = s1; s_part[warp][2] = s2; }
    __syncthreads();
    if (tid < 3) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; w++) s += s_part[w][tid];
        partial[((size_t)b * gridDim.x + blockIdx.x) * 3 + tid] = s;
    }
}

// One CTA of three warps: warp c sums channel c of the `nblk` partials (lane l takes every 32nd, then a butterfly).
__global__ void __launch_bounds__(96) bg_grad_finish_kernel(int nblk, const float* __restrict__ partial, float* __restrict__ out)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float s = 0.0f;
    for (int k = lane; k < nblk; k += 32) s += partial[3 * (size_t)k + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[c] = s;
}

int image_alpha(bool tet, int B, int W, int H, const float* t, const uint8_t* active, float* alpha, cudaStream_t stream)
{
    const size_t n = (size_t)B * W * H;
    if (n == 0) return 0;
    const unsigned nblk = (unsigned)std::min<size_t>((n + 255) / 256, 148 * 8);
    ProfScope prof(tet ? ST_TET_ALPHA : ST_TRI_ALPHA, stream);
    if (tet) DMR_CUDA(dmr_launch(alpha_kernel<true>, dim3(nblk), dim3(256), 0, stream, n, t, active, alpha));
    else DMR_CUDA(dmr_launch(alpha_kernel<false>, dim3(nblk), dim3(256), 0, stream, n, t, active, alpha));
    DMR_LAUNCH_CHECK("alpha_kernel");
    return 0;
}

// nbx * B <= BG_BLOCKS + B
size_t image_bg_grad_bytes(int B) { return align_up(sizeof(float) * 3 * (BG_BLOCKS + (size_t)B), 256) + 256; }

int image_bg_grad(bool tet, int B, int W, int H, const float* t, const uint8_t* active, const float* dL_dcolor, float* dL_dbg,
                  void* workspace, cudaStream_t stream)
{
    ProfScope prof(tet ? ST_TET_BG_GRAD : ST_TRI_BG_GRAD, stream);
    count_launch(1);   // two kernels under one scope
    float* partial = static_cast<float*>(workspace);
    const uint32_t HW = (uint32_t)W * (uint32_t)H;
    const unsigned nbx = std::max(1u, std::min((BG_BLOCKS + B - 1) / (unsigned)B, (HW + 1023) / 1024));
    const dim3 grid(nbx, B);
    if (tet) DMR_CUDA(dmr_launch(bg_grad_partial_kernel<true>, grid, dim3(256), 0, stream, HW, t, active, dL_dcolor, partial));
    else DMR_CUDA(dmr_launch(bg_grad_partial_kernel<false>, grid, dim3(256), 0, stream, HW, t, active, dL_dcolor, partial));
    DMR_LAUNCH_CHECK("bg_grad_partial_kernel");
    DMR_CUDA(dmr_launch(bg_grad_finish_kernel, dim3(1), dim3(96), 0, stream, (int)(nbx * B), (const float*)partial, dL_dbg));
    DMR_LAUNCH_CHECK("bg_grad_finish_kernel");
    return 0;
}

size_t face_weights_bytes(int B, int F) { return 12 * (size_t)B * F; }

FaceWeightAcc face_weights_acc(void* workspace, int B, int F)
{
    FaceWeightAcc a;
    a.weight = static_cast<unsigned long long*>(workspace);
    a.hits = reinterpret_cast<uint32_t*>(a.weight + (size_t)B * F);
    return a;
}

// fixed point (2^-32) -> fp32: one rounding (the scale is a power of two)
__global__ void __launch_bounds__(256) face_weights_convert_kernel(size_t n, FaceWeightAcc acc, float* __restrict__ face_weights,
                                                                   int* __restrict__ face_hits)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        face_weights[i] = __ull2float_rn(acc.weight[i]) * 0x1p-32f;
        face_hits[i] = (int)acc.hits[i];
    }
}

int face_weights_convert(int B, int F, const FaceWeightAcc& acc, float* face_weights, int* face_hits, cudaStream_t stream)
{
    const size_t n = (size_t)B * F;
    if (n == 0) return 0;
    const unsigned nblk = (unsigned)std::min<size_t>((n + 255) / 256, 148 * 8);
    DMR_CUDA(dmr_launch(face_weights_convert_kernel, dim3(nblk), dim3(256), 0, stream, n, acc, face_weights, face_hits));
    DMR_LAUNCH_CHECK("face_weights_convert_kernel");
    return 0;
}

}  // namespace dmr
