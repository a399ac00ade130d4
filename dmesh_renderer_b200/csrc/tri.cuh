// tri.cuh -- launch interface of the tri renderer's kernels.
#pragma once
#include "common.cuh"
#include "radix_sort.cuh"

namespace dmr {

struct TriRenderParams {
    int B, P, F, W, H;
    const uint2* ranges;            // [B*tiles]
    const uint32_t* face_list;      // sorted values [R]
    const TriRecord* records;       // [B*F]
    const float* bg;                // [3]
    const float* inv_mv;            // [B,16]
    const float* inv_proj;          // [B,16]
    float* final_T;                 // [B*W*H]
    float* prev_T;                  // [B*W*H]
    uint32_t* n_contrib;            // [B*W*H]
    float* out_color;               // [B,3,H,W]
    float* out_depth;               // [B,1,H,W]
    // backward only
    const float* dL_dcolor;
    const float* dL_ddepth;
    float* dL_dverts;
    float* dL_dvcolor;
    float* dL_dfopacity;
    float* dL_dvdepth;
    float* dL_dfintense;
    float* grad_stats;              // [B*F,24] zeroed scratch (face buffer)
    float4* grad_vacc;              // [2][P] zeroed scratch: per-vertex dL_dverts / dL_dvcolor accumulators
    // deterministic mode only (tri_render_backward_deterministic): zeroed 64-bit fixed-point accumulators
    const uint32_t* det_gmax;       // [2]: bits of max |cotangent| (written by det_gmax_kernel), overflow word
    long long* det_stats;           // [B*F,24] statistics in logical order
    long long* det_vert;            // [P,8]: dL_dverts xyz, -, dL_dvcolor rgb, -
    long long* det_vdepth;          // [B*P]
    long long* det_fopa;            // [F]
};

struct TriDetLayout {               // workspace of the deterministic backward pass
    size_t gmax, stats, vert, vdepth, fopa, hi, total;   // low words stats..fopa, their high words mirrored at hi
    __host__ __device__ static TriDetLayout make(size_t B, size_t P, size_t F)
    {
        TriDetLayout L;
        size_t o = 0;
        L.gmax = o;   o = align_up(o + 4, 256);
        L.stats = o;  o = align_up(o + 8 * 24 * B * F, 256);
        L.vert = o;   o = align_up(o + 8 * 8 * P, 256);
        L.vdepth = o; o = align_up(o + 8 * B * P, 256);
        L.fopa = o;   o = align_up(o + 8 * F, 256);
        L.hi = o;     o += o - L.stats;
        L.total = o;
        return L;
    }
    // element offset of an accumulator's high word from its low word (det.cuh)
    __host__ __device__ static ptrdiff_t hi_offset(size_t B, size_t P, size_t F)
    {
        const TriDetLayout L = make(B, P, F);
        return (ptrdiff_t)((L.hi - L.stats) / 8);
    }
};

int tri_preprocess_faces(int B, int P, int F, int W, int H, const int* faces, const float4* vimg, const float* verts,
                         const float* verts_color, const float* faces_opacity, const float* faces_intense,
                         uint32_t* tiles_touched, uint32_t* depth_key, uint2* rect, TriRecord* records,
                         const SortPre& face_sort, cudaStream_t stream);
// fw != nullptr: the face-statistics instantiation, which also adds every hit's blending weight and 1 to fw's
// (view, face) accumulators (zeroed by the caller)
int tri_render_forward(const TriRenderParams& p, cudaStream_t stream, const FaceWeightAcc* fw = nullptr);
// cam_tiles != nullptr: the camera-gradient kernels, which also store one 24-float record per (view, tile) there.
// exact: the exact vertex-position instantiations (same launches, same workspace).
// dL_dalpha != nullptr: the alpha-cotangent instantiations ([B,H,W] cotangent of alpha = 1 - final_T)
int tri_render_backward(const TriRenderParams& p, cudaStream_t stream, float* cam_tiles = nullptr, bool exact = false,
                        const float* dL_dalpha = nullptr);
int tri_render_backward_deterministic(const TriRenderParams& p, cudaStream_t stream, float* cam_tiles = nullptr,
                                      bool exact = false, const float* dL_dalpha = nullptr);
// per-tile camera records of a view -> += dL_dmv[B,16], dL_dproj[B,16]
int tri_camera_finish(int B, int W, int H, const float* cam_tiles, const float* inv_mv, const float* inv_proj, float* dL_dmv,
                      float* dL_dproj, cudaStream_t stream);

}  // namespace dmr
