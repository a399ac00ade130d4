// preprocess.cu -- per-vertex projection and per-(view,face) setup.
//
//   preprocess_points_kernel   replaces preprocessPointCUDA
//                              (cuda_rasterizer/forward.cu:17-47, identical copy
//                              cuda_renderer/forward.cu:21-52)
//   tri_preprocess_faces_kernel replaces preprocessFaceCUDA
//                              (cuda_rasterizer/forward.cu:76-149) and hoists the
//                              per-face part of in_tri (auxiliary.h:179-243) and
//                              the per-instance gathers of renderCUDA
//                              (forward.cu:358-400) into one 144-byte record.
//
// Both are HBM-bound streaming kernels: one thread per element, 128-bit
// loads/stores, records transposed through shared memory so that the global
// write of a block's 256 records is one contiguous 36 KB burst.
#include "tri.cuh"
#include "tet.cuh"
#include "radix_sort.cuh"
#include <algorithm>

namespace dmr {

// ---------------------------------------------------------------------------
// points: out[b*P+p] = { pix.x, pix.y, ndc.z, verts_depth[b,p] }  (tet: 4th lane = clip w)
// algorithmic bytes per (b,p): 4 (depth) read, 16 written; + 12 (xyz) per vertex and call.
// The reference also stores ndc.xy (never read downstream, SURVEY 8a1).
// ---------------------------------------------------------------------------
constexpr int DMR_POINTS_PER_THREAD = 4;
__global__ void __launch_bounds__(256) preprocess_points_kernel(
    int B, int P, int W, int H,
    const float* __restrict__ verts, const float* __restrict__ mv_mats, const float* __restrict__ proj_mats,
    const float* __restrict__ verts_depth,   // may be null, see depth_mode
    int depth_mode,                          // 4th lane when verts_depth is null: 0 = clip-space w (tet), 1 = NDC z
    float4* __restrict__ vimg)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    // A thread owns DMR_POINTS_PER_THREAD vertices (block-strided, so every access stays coalesced) and walks the
    // views: the positions are read once per call instead of once per view (12 of the 32 bytes per (view, vertex)),
    // and the two matrices of a view -- 28 uniform loads -- once per thread and view (with one (view, vertex) per
    // thread they were two thirds of the kernel's load instructions; the L1 data pipe, not HBM, was its busiest
    // unit: 65 % against 50 % DRAM utilisation at C5).
    float3 pos[DMR_POINTS_PER_THREAD];
    size_t idx[DMR_POINTS_PER_THREAD];
#pragma unroll
    for (int it = 0; it < DMR_POINTS_PER_THREAD; it++) {
        idx[it] = ((size_t)blockIdx.x * DMR_POINTS_PER_THREAD + it) * 256 + threadIdx.x;
        pos[it] = idx[it] < (size_t)P ? f3(verts[3 * idx[it] + 0], verts[3 * idx[it] + 1], verts[3 * idx[it] + 2]) : f3(0, 0, 0);
    }
    for (int b = 0; b < B; b++) {
        float mv[16], pj[16];
#pragma unroll
        for (int i = 0; i < 16; i++) { mv[i] = mv_mats[16 * b + i]; pj[i] = proj_mats[16 * b + i]; }
#pragma unroll
        for (int it = 0; it < DMR_POINTS_PER_THREAD; it++) {
            if (idx[it] >= (size_t)P) break;
            float3 p = pos[it];
            float3 pv = xform43(p, mv);
            float4 pp = xform44(pv, pj);
            float pw = 1.0 / clamp_w(pp.w);                 // forward.cu:38 (double literal, float result)
            float3 ndc = f3(pp.x * pw, pp.y * pw, pp.z * pw);

            float4 o;
            o.x = ndc2pix(ndc.x, W);
            o.y = ndc2pix(ndc.y, H);
            o.z = ndc.z;
            // tet path: clip-space w (bbox validity); tri path without a verts_depth tensor: the vertex's own NDC z
            o.w = verts_depth ? verts_depth[(size_t)b * P + idx[it]] : (depth_mode == 1 ? ndc.z : pp.w);
            vimg[(size_t)b * P + idx[it]] = o;
        }
    }
}

int preprocess_points(int B, int P, int W, int H, const float* verts, const float* mv, const float* proj,
                      const float* verts_depth, int depth_mode, float4* vimg, cudaStream_t stream)
{
    if (B <= 0 || P <= 0) return 0;
    dim3 grid((P + 256 * DMR_POINTS_PER_THREAD - 1) / (256 * DMR_POINTS_PER_THREAD));
    ProfScope prof(ST_POINTS, stream);
    DMR_CUDA(dmr_launch(preprocess_points_kernel, dim3(grid), dim3(256), 0, stream, B, P, W, H, verts, mv, proj, verts_depth, depth_mode, vimg));
    DMR_LAUNCH_CHECK("preprocess_points_kernel");
    return 0;
}

// ---------------------------------------------------------------------------
// Fused vertex depth (SURVEY.md 8f-1): when the caller passes no verts_depth tensor the renderer uses the NDC z
// it computes anyway.  The caller's usual upstream op  verts_depth[b,p] = ndc_z(P_b M_b p)  then has to be
// differentiated here: dL/dp += sum_b dL/dverts_depth[b,p] * d ndc_z / dp, with
//   ndc_z = z_clip / clamp_w(w_clip),  d ndc_z/dp = (dz_clip/dp - ndc_z * dw_clip/dp) / w   (w not clamped)
// One thread per vertex, loop over the views (coalesced reads of dL_dvdepth rows), no atomics.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) depth_chain_kernel(int B, int P, const float* __restrict__ verts,
                                                          const float* __restrict__ mv_mats, const float* __restrict__ proj_mats,
                                                          const float* __restrict__ dL_dvdepth, float* __restrict__ dL_dverts)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)P) return;
    const float3 p = f3(verts[3 * idx + 0], verts[3 * idx + 1], verts[3 * idx + 2]);
    float3 acc = f3(0, 0, 0);
    for (int b = 0; b < B; b++) {
        const float g = dL_dvdepth[(size_t)b * P + idx];
        if (g == 0.0f) continue;
        const float* mv = mv_mats + 16 * b;
        const float* pj = proj_mats + 16 * b;
        const float3 pv = xform43(p, mv);
        const float4 pp = xform44(pv, pj);
        const float wc = clamp_w(pp.w);
        const float pw = 1.0f / wc;
        const float ndc_z = pp.z * pw;
        const bool clamped = wc != pp.w;     // |w| < 1e-4: the reciprocal is a constant
        float az[3], aw[3];                  // rows 2 and 3 of (Proj * MV)[:, 0:3]
#pragma unroll
        for (int c = 0; c < 3; c++) {
            az[c] = pj[2] * mv[4 * c + 0] + pj[6] * mv[4 * c + 1] + pj[10] * mv[4 * c + 2];
            aw[c] = pj[3] * mv[4 * c + 0] + pj[7] * mv[4 * c + 1] + pj[11] * mv[4 * c + 2];
        }
        const float k = g * pw;
        acc.x += k * (az[0] - (clamped ? 0.0f : ndc_z * aw[0]));
        acc.y += k * (az[1] - (clamped ? 0.0f : ndc_z * aw[1]));
        acc.z += k * (az[2] - (clamped ? 0.0f : ndc_z * aw[2]));
    }
    dL_dverts[3 * idx + 0] += acc.x;
    dL_dverts[3 * idx + 1] += acc.y;
    dL_dverts[3 * idx + 2] += acc.z;
}

int depth_chain(int B, int P, const float* verts, const float* mv, const float* proj, const float* dL_dvdepth,
                float* dL_dverts, cudaStream_t stream)
{
    if (B <= 0 || P <= 0) return 0;
    count_launch(1);
    DMR_CUDA(dmr_launch(depth_chain_kernel, dim3((P + 255) / 256), dim3(256), 0, stream, B, P, verts, mv, proj, dL_dvdepth, dL_dverts));
    DMR_LAUNCH_CHECK("depth_chain_kernel");
    return 0;
}

// Camera variant (dmr_tri_depth_chain_camera): the same per-(view, vertex) terms -- pv = MV p, clip = Proj (pv, 1),
// ndc_z = z_clip / clamp_w(w_clip), no derivative through a clamped w -- reduced over the vertices into the 20 nonzero
// partials of dL/dmv[b] and dL/dproj[b]:
//   gz = g / w, gw = -g ndc_z / w  (0 if clamped),  gpv = gz Proj[2, 0:3] + gw Proj[3, 0:3]
//   [0..3]   dL/dproj[2, 0..3] = gz (pv, 1)       [4..7]   dL/dproj[3, 0..3] = gw (pv, 1)
//   [8 + 3c + i]  dL/dmv[i, c] = gpv[i] (p, 1)[c]    (i < 3, c < 4)
// Fixed grid (DMR_DEPTH_CAM_BLOCKS blocks per view at most, a function of P only), per-block partials in a fixed
// order, and one CTA per view that adds the partials in block order: reproducible, no float atomics.
#define DMR_DEPTH_CAM_TERMS 20
#define DMR_DEPTH_CAM_BLOCKS 256
static int depth_cam_blocks(int P) { return (int)std::min<long long>(DMR_DEPTH_CAM_BLOCKS, ((long long)P + 1023) / 1024); }
size_t depth_chain_camera_bytes(int B, int P)
{
    return align_up(sizeof(float) * DMR_DEPTH_CAM_TERMS * (size_t)B * depth_cam_blocks(P), 256) + 256;
}

__global__ void __launch_bounds__(256) depth_chain_camera_kernel(int P, const float* __restrict__ verts,
                                                                 const float* __restrict__ mv_mats, const float* __restrict__ proj_mats,
                                                                 const float* __restrict__ dL_dvdepth, float* __restrict__ partials)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ float s_w[8][DMR_DEPTH_CAM_TERMS];
    const int b = blockIdx.y;
    const float* mv = mv_mats + 16 * b;
    const float* pj = proj_mats + 16 * b;
    float acc[DMR_DEPTH_CAM_TERMS];
#pragma unroll
    for (int k = 0; k < DMR_DEPTH_CAM_TERMS; k++) acc[k] = 0.0f;
    for (size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x; idx < (size_t)P; idx += (size_t)gridDim.x * 256) {
        const float g = dL_dvdepth[(size_t)b * P + idx];
        if (g == 0.0f) continue;
        const float3 p = f3(verts[3 * idx + 0], verts[3 * idx + 1], verts[3 * idx + 2]);
        const float3 pv = xform43(p, mv);
        const float4 pp = xform44(pv, pj);
        const float wc = clamp_w(pp.w);
        const float pw = 1.0f / wc;
        const float ndc_z = pp.z * pw;
        const bool clamped = wc != pp.w;
        const float gz = g * pw, gw = clamped ? 0.0f : -gz * ndc_z;
        acc[0] += gz * pv.x; acc[1] += gz * pv.y; acc[2] += gz * pv.z; acc[3] += gz;
        acc[4] += gw * pv.x; acc[5] += gw * pv.y; acc[6] += gw * pv.z; acc[7] += gw;
        const float gpv[3] = { gz * pj[2] + gw * pj[3], gz * pj[6] + gw * pj[7], gz * pj[10] + gw * pj[11] };
#pragma unroll
        for (int i = 0; i < 3; i++) {
            acc[8 + i] += gpv[i] * p.x; acc[11 + i] += gpv[i] * p.y; acc[14 + i] += gpv[i] * p.z; acc[17 + i] += gpv[i];
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < DMR_DEPTH_CAM_TERMS; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < DMR_DEPTH_CAM_TERMS; k++) s_w[warp][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < DMR_DEPTH_CAM_TERMS) {
        float sum = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; w++) sum += s_w[w][threadIdx.x];
        partials[((size_t)b * gridDim.x + blockIdx.x) * DMR_DEPTH_CAM_TERMS + threadIdx.x] = sum;
    }
}

// One warp per view: the view's block partials in block order, ADDED to dL_dmv[b] / dL_dproj[b] (column-major).
__global__ void __launch_bounds__(32) depth_chain_camera_finish_kernel(int nblk, const float* __restrict__ partials,
                                                                       float* __restrict__ dL_dmv, float* __restrict__ dL_dproj)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int b = blockIdx.x, k = threadIdx.x;
    if (k >= DMR_DEPTH_CAM_TERMS) return;
    float sum = 0.0f;
    for (int j = 0; j < nblk; j++) sum += partials[((size_t)b * nblk + j) * DMR_DEPTH_CAM_TERMS + k];
    if (k < 8) dL_dproj[16 * b + 4 * (k & 3) + 2 + (k >> 2)] += sum;    // row 2 (k < 4) / row 3, column k & 3
    else dL_dmv[16 * b + 4 * ((k - 8) / 3) + (k - 8) % 3] += sum;        // row (k - 8) % 3, column (k - 8) / 3
}

int depth_chain_camera(int B, int P, const float* verts, const float* mv, const float* proj, const float* dL_dvdepth,
                       float* dL_dmv, float* dL_dproj, void* workspace, cudaStream_t stream)
{
    if (B <= 0 || P <= 0) return 0;
    const int nblk = depth_cam_blocks(P);
    float* partials = static_cast<float*>(workspace);
    {
        ProfScope prof(ST_DEPTH_CAM, stream);
        DMR_CUDA(dmr_launch(depth_chain_camera_kernel, dim3(nblk, B), dim3(256), 0, stream, P, verts, mv, proj, dL_dvdepth, partials));
        DMR_LAUNCH_CHECK("depth_chain_camera_kernel");
    }
    {
        ProfScope prof(ST_DEPTH_CAM_FINISH, stream);
        DMR_CUDA(dmr_launch(depth_chain_camera_finish_kernel, dim3(B), dim3(32), 0, stream, nblk, (const float*)partials, dL_dmv, dL_dproj));
        DMR_LAUNCH_CHECK("depth_chain_camera_finish_kernel");
    }
    return 0;
}

// ---------------------------------------------------------------------------
// Tile rectangle of a triangle: getRectFromTri (auxiliary.h:55-69).
// Float -> int is cvt.rzi (saturating, NaN -> 0) as in the reference.  A
// rectangle whose max is not above its min in either axis covers 0 tiles.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tile_rect(float2 p0, float2 p1, float2 p2, int gx, int gy, int& x0, int& y0, int& x1,
                                          int& y1)
{
    float mnx = fminf(fminf(p0.x, p1.x), p2.x), mny = fminf(fminf(p0.y, p1.y), p2.y);
    float mxx = fmaxf(fmaxf(p0.x, p1.x), p2.x), mxy = fmaxf(fmaxf(p0.y, p1.y), p2.y);
    x0 = min(gx, max(0, (int)(mnx / DMR_TILE)));
    y0 = min(gy, max(0, (int)(mny / DMR_TILE)));
    x1 = min(gx, max(0, (int)((unsigned)(int)(mxx / DMR_TILE) + 1u)));
    y1 = min(gy, max(0, (int)((unsigned)(int)(mxy / DMR_TILE) + 1u)));
}

// ---------------------------------------------------------------------------
// Edge-function setup: the per-face half of in_tri (auxiliary.h:191-240).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void edge_setup(float2 p1, float2 p2, float2 p3, int W, int H, uint32_t* ea, uint32_t* eb,
                                           uint32_t* ec, uint32_t& flags)
{
    const float subpixel = 16.0f;
    int x1 = (int)(p1.x * subpixel), y1 = (int)(p1.y * subpixel);
    int x2 = (int)(p2.x * subpixel), y2 = (int)(p2.y * subpixel);
    int x3 = (int)(p3.x * subpixel), y3 = (int)(p3.y * subpixel);
    // wrapping 32-bit arithmetic throughout (the reference's int math wraps in hardware)
    uint32_t ux1 = x1, uy1 = y1, ux2 = x2, uy2 = y2, ux3 = x3, uy3 = y3;
    int area = (int)((ux2 - ux1) * (uy3 - uy1) - (ux3 - ux1) * (uy2 - uy1));
    flags = 0;
    if (area == 0) {
        for (int k = 0; k < 3; k++) { ea[k] = 0; eb[k] = 0; ec[k] = 0; }
        flags = DMR_REC_SAFE | (DMR_REC_NB_UNBOUNDED << DMR_REC_NBX_SHIFT) | (DMR_REC_NB_UNBOUNDED << DMR_REC_NBY_SHIFT);
        return;
    }
    if (area < 0) {   // make CCW: swap vertices 2 and 3
        uint32_t t = ux2; ux2 = ux3; ux3 = t;
        t = uy2; uy2 = uy3; uy3 = t;
    }
    uint32_t vx[3] = { ux1, ux2, ux3 }, vy[3] = { uy1, uy2, uy3 };
    bool safe = true;
    // exact (64-bit) check that no intermediate of the pixel test can overflow
    {
        long long lx1 = (int)ux1, ly1 = (int)uy1, lx2 = (int)ux2, ly2 = (int)uy2, lx3 = (int)ux3, ly3 = (int)uy3;
        long long a64 = (lx2 - lx1) * (ly3 - ly1) - (lx3 - lx1) * (ly2 - ly1);
        const long long lim = 0x3fffffffLL;
        if (llabs(lx1) > lim || llabs(ly1) > lim || llabs(lx2) > lim || llabs(ly2) > lim || llabs(lx3) > lim ||
            llabs(ly3) > lim || llabs(a64) > 0x7fffffffLL)
            safe = false;
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        int kn = (k + 1) % 3;
        uint32_t cx = vx[k] - vx[kn], cy = vy[k] - vy[kn];
        int scx = (int)cx, scy = (int)cy;
        uint32_t bias = (scy > 0 || (scy == 0 && scx > 0)) ? 1u : 0u;
        ea[k] = (uint32_t)0 - 16u * cy;
        eb[k] = 16u * cx;
        ec[k] = 8u * cx - 8u * cy + cy * vx[k] - cx * vy[k] - bias;
        if (safe) {
            long long lcx = (long long)(int)vx[k] - (long long)(int)vx[kn];
            long long lcy = (long long)(int)vy[k] - (long long)(int)vy[kn];
            long long A = -16 * lcy, Bc = 16 * lcx;
            long long C = 8 * lcx - 8 * lcy + lcy * (long long)(int)vx[k] - lcx * (long long)(int)vy[k] - (long long)bias;
            // (tiles at the right / bottom border extend up to 15 pixels beyond the image; the block tests evaluate there)
            long long bound = llabs(A) * (long long)(W + 16) + llabs(Bc) * (long long)(H + 16) + llabs(C);
            if (llabs(lcx) > 0x7ffffffLL || llabs(lcy) > 0x7ffffffLL || bound > 0x7fffffffLL) safe = false;
        }
    }
    // block bbox of the pixels whose centre (16 px + 8 in 1/16-pixel units) lies inside the snapped triangle's
    // bounding rectangle (closed: conservative for the strict edge tests and the fill rule)
    uint32_t bx0 = 0, by0 = 0, nbx = DMR_REC_NB_UNBOUNDED, nby = DMR_REC_NB_UNBOUNDED;
    if (safe && W <= 4096 && H <= 4096) {
        const int mnx = min(min(x1, x2), x3), mxx = max(max(x1, x2), x3);
        const int mny = min(min(y1, y2), y3), mxy = max(max(y1, y2), y3);
        int px0 = (mnx + 7) >> 4, px1 = (mxx - 8) >> 4;      // ceil((min - 8) / 16), floor((max - 8) / 16)
        int py0 = (mny + 7) >> 4, py1 = (mxy - 8) >> 4;
        px0 = max(px0, 0); py0 = max(py0, 0);
        px1 = min(px1, W - 1); py1 = min(py1, H - 1);
        if (px1 < px0 || py1 < py0) {                          // no pixel centre inside: never covered
            for (int k = 0; k < 3; k++) { ea[k] = 0; eb[k] = 0; ec[k] = 0; }
            flags = DMR_REC_SAFE | (DMR_REC_NB_UNBOUNDED << DMR_REC_NBX_SHIFT) | (DMR_REC_NB_UNBOUNDED << DMR_REC_NBY_SHIFT);
            return;
        }
        const uint32_t cx = (uint32_t)(px1 >> 3) - (uint32_t)(px0 >> 3) + 1u, cy = (uint32_t)(py1 >> 2) - (uint32_t)(py0 >> 2) + 1u;
        if (cx < DMR_REC_NB_UNBOUNDED) { bx0 = (uint32_t)(px0 >> 3); nbx = cx; }
        if (cy < DMR_REC_NB_UNBOUNDED) { by0 = (uint32_t)(py0 >> 2); nby = cy; }
    }
    flags = (safe ? DMR_REC_SAFE : 0u) | (bx0 << DMR_REC_BX0_SHIFT) | (by0 << DMR_REC_BY0_SHIFT) |
            (nbx << DMR_REC_NBX_SHIFT) | (nby << DMR_REC_NBY_SHIFT);
}

// ---------------------------------------------------------------------------
// faces (tri): tiles_touched, tile rect, depth key, 144-byte record.
// algorithmic bytes per (b,f): read 3*16 (vimg) + 4 (intensity), write 4 + 4 + 8 + 144; per face and call: read
// 12 (idx) + 3*12 (pos) + 3*12 (colour) + 4 (opacity).
// ---------------------------------------------------------------------------
constexpr int DMR_FACES_MINB = 4;
template <bool HIST, bool MULTI>   // HIST: accumulate the face sort's histograms as a by-product (small inputs only);
                                   // MULTI = false: B == 1 (no view loop: 58 instead of 64 registers + spills)
__global__ void __launch_bounds__(256, DMR_FACES_MINB) tri_preprocess_faces_kernel(
    int B, int P, int F, int W, int H, int gx, int gy,
    const int* __restrict__ faces, const float4* __restrict__ vimg,
    const float* __restrict__ verts, const float* __restrict__ verts_color,
    const float* __restrict__ faces_opacity, const float* __restrict__ faces_intense,
    uint32_t* __restrict__ tiles_touched, uint32_t* __restrict__ depth_key, uint2* __restrict__ rect,
    TriRecord* __restrict__ records, SortPre sp)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ uint4 s_rec[256 * 9];
    __shared__ uint32_t s_hist[HIST ? 4 * 256 : 1];   // digit histograms of the depth keys for the face sort (radix_sort.cuh)
    const int tid = threadIdx.x;
    if (HIST) {
        for (int i = tid; i < 4 * 256; i += 256) s_hist[i] = 0;
        __syncthreads();
    }
    // A thread owns face f and walks the views: the face's indices, world positions, colours and opacity (88 of the
    // 300 bytes moved per (view, face)) are read once per call instead of once per view.
    const size_t f0 = (size_t)blockIdx.x * 256;
    const size_t f = f0 + tid;
    const bool valid = f < (size_t)F;
    const size_t nvalid = (f0 + 256 <= (size_t)F) ? 256 : ((size_t)F > f0 ? (size_t)F - f0 : 0);
    int i0 = 0, i1 = 0, i2 = 0;
    uint32_t pos[9], col[9], opa = 0u;
#pragma unroll
    for (int k = 0; k < 9; k++) { pos[k] = 0u; col[k] = 0u; }
    if (valid) {
        i0 = faces[3 * f + 0]; i1 = faces[3 * f + 1]; i2 = faces[3 * f + 2];
        const int vi[3] = { i0, i1, i2 };
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const float* q = verts + 3 * (size_t)vi[k];
            const float* c = verts_color + 3 * (size_t)vi[k];
            pos[3 * k] = __float_as_uint(q[0]); pos[3 * k + 1] = __float_as_uint(q[1]); pos[3 * k + 2] = __float_as_uint(q[2]);
            col[3 * k] = __float_as_uint(c[0]); col[3 * k + 1] = __float_as_uint(c[1]); col[3 * k + 2] = __float_as_uint(c[2]);
        }
        opa = __float_as_uint(faces_opacity[f]);
    }

    const int nviews = MULTI ? B : 1;
    for (int b = 0; b < nviews; b++) {
        uint32_t sort_key[1] = { 0u };
        if (valid) {
            const float4* vb = vimg + (size_t)b * P;
            float4 a0 = vb[i0], a1 = vb[i1], a2 = vb[i2];

            // forward.cu:101-121
            float max_z = a0.z, min_z = a0.z, depth = 0;
            depth += a0.z;
            max_z = fmaxf(max_z, a1.z); min_z = fminf(min_z, a1.z); depth += a1.z;
            max_z = fmaxf(max_z, a2.z); min_z = fminf(min_z, a2.z); depth += a2.z;
            depth = depth / 3.0f;

            uint32_t touched = 0;
            int x0 = 0, y0 = 0, x1 = 0, y1 = 0;
            float2 p0 = make_float2(a0.x, a0.y), p1 = make_float2(a1.x, a1.y), p2 = make_float2(a2.x, a2.y);
            if (!(max_z < -1.0f || min_z > 1.0f)) {    // forward.cu:124
                tile_rect(p0, p1, p2, gx, gy, x0, y0, x1, y1);
                if (x1 > x0 && y1 > y0) touched = (uint32_t)(y1 - y0) * (uint32_t)(x1 - x0);
            }
            // forward.cu:146-148
            float dk = (depth + 1.0f) * 0.5f;
            if (dk < 0.0f) dk = 0.0f;
            if (dk > 1.0f) dk = 1.0f;

            size_t bf = (size_t)b * F + f;
            tiles_touched[bf] = touched;
            depth_key[bf] = __float_as_uint(dk);
            sort_key[0] = __float_as_uint(dk);
            rect[bf] = make_uint2((uint32_t)x0 | ((uint32_t)x1 << 16), (uint32_t)y0 | ((uint32_t)y1 << 16));

            uint32_t ea[3], eb[3], ec[3], flags;
            edge_setup(p0, p1, p2, W, H, ea, eb, ec, flags);

            uint4* r = s_rec + tid * 9;
            r[0] = make_uint4(ea[0], eb[0], ec[0], flags);
            r[1] = make_uint4(ea[1], eb[1], ec[1], (uint32_t)i0);
            r[2] = make_uint4(ea[2], eb[2], ec[2], (uint32_t)i1);
            r[3] = make_uint4(pos[0], pos[1], pos[2], opa);
            r[4] = make_uint4(pos[3], pos[4], pos[5], __float_as_uint(faces_intense[bf]));
            r[5] = make_uint4(pos[6], pos[7], pos[8], (uint32_t)i2);
            r[6] = make_uint4(col[0], col[1], col[2], __float_as_uint(a0.w));
            r[7] = make_uint4(col[3], col[4], col[5], __float_as_uint(a1.w));
            r[8] = make_uint4(col[6], col[7], col[8], __float_as_uint(a2.w));
        }
        __syncthreads();
        // coalesced write-out of the block's records of this view
        uint4* dst = reinterpret_cast<uint4*>(records + (size_t)b * F + f0);
        for (size_t i = tid; i < nvalid * 9; i += 256) dst[i] = s_rec[i];
        // by-product: digit histograms of the depth keys
        if (HIST) {
            const bool sort_valid[1] = { valid };
            rs_pre_add<1>(s_hist, sort_key, sort_valid, sp);
        }
        if (MULTI) __syncthreads();   // the next view overwrites s_rec
    }
    if (HIST) rs_pre_finish(s_hist, sp, gridDim.x);   // (last block) the plan of the face sort
}

int tri_preprocess_faces(int B, int P, int F, int W, int H, const int* faces, const float4* vimg, const float* verts,
                         const float* verts_color, const float* faces_opacity, const float* faces_intense,
                         uint32_t* tiles_touched, uint32_t* depth_key, uint2* rect, TriRecord* records,
                         const SortPre& sp, cudaStream_t stream)
{
    if (B <= 0 || F <= 0) return 0;
    int gx = (W + DMR_TILE - 1) / DMR_TILE, gy = (H + DMR_TILE - 1) / DMR_TILE;
    dim3 grid((F + 255) / 256);
    ProfScope prof(ST_FACES, stream);
#define DMR_FACES_LAUNCH(HIST_, MULTI_)                                                                                         \
    DMR_CUDA(dmr_launch(tri_preprocess_faces_kernel<HIST_, MULTI_>, dim3(grid), dim3(256), 0, stream, B, P, F, W, H, gx, gy, faces,   \
                        vimg, verts, verts_color, faces_opacity, faces_intense, tiles_touched, depth_key, rect, records, sp))
    if (sp.npass > 0) { if (B > 1) DMR_FACES_LAUNCH(true, true); else DMR_FACES_LAUNCH(true, false); }
    else              { if (B > 1) DMR_FACES_LAUNCH(false, true); else DMR_FACES_LAUNCH(false, false); }
#undef DMR_FACES_LAUNCH
    DMR_LAUNCH_CHECK("tri_preprocess_faces_kernel");
    return 0;
}

// ---------------------------------------------------------------------------
// faces (tet): replaces TET preprocessFaceCUDA (cuda_renderer/forward.cu:178-260).
// Sort depth is the clamped MIN depth (renderer_impl.cu:325); the record carries
// the world-space triangle plus min/max depth for firstIntersect.
// algorithmic bytes per (b,f): read 12 + 3*16 + 3*12, write 4 + 4 + 8 + 64.
// ---------------------------------------------------------------------------
template <bool HIST>
__global__ void __launch_bounds__(256) tet_preprocess_faces_kernel(
    int B, int P, int F, int gx, int gy,
    const int* __restrict__ faces, const float4* __restrict__ vimg, const float* __restrict__ verts,
    uint32_t* __restrict__ tiles_touched, uint32_t* __restrict__ depth_key, uint2* __restrict__ rect,
    TetFaceRec* __restrict__ records, SortPre sp)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ uint4 s_rec[256 * 4];
    __shared__ uint32_t s_hist[HIST ? 4 * 256 : 1];   // digit histograms of the depth keys for the face sort (radix_sort.cuh)
    const int tid = threadIdx.x;
    if (HIST) {
        for (int i = tid; i < 4 * 256; i += 256) s_hist[i] = 0;
        __syncthreads();
    }
    const size_t f0 = (size_t)blockIdx.x * 256;
    const int b = blockIdx.y;
    const size_t f = f0 + tid;
    uint32_t sort_key[1] = { 0u };
    if (f < (size_t)F) {
        int i0 = faces[3 * f + 0], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
        const float4* vb = vimg + (size_t)b * P;
        float4 a0 = vb[i0], a1 = vb[i1], a2 = vb[i2];
        // conservative pixel bounds of the projected triangle (valid only if all w are safely positive)
        uint32_t bbx = 0xffff0000u, bby = 0xffff0000u;
        if (a0.w > 1e-4f && a1.w > 1e-4f && a2.w > 1e-4f) {
            float lx = fminf(fminf(a0.x, a1.x), a2.x), hx = fmaxf(fmaxf(a0.x, a1.x), a2.x);
            float ly = fminf(fminf(a0.y, a1.y), a2.y), hy = fmaxf(fmaxf(a0.y, a1.y), a2.y);
            // ray through pixel x passes at x+0.5 (or, jittered, in (x-0.5, x]); keep x when that can lie in
            // [lx-1, hx+1]  <=>  x in [ceil(lx-1.5), floor(hx+1.5)]
            int x0 = max(0, min(65535, (int)fmaxf(fminf(ceilf(lx - 1.5f), 70000.0f), -1.0f)));
            int x1 = max(-1, min(65535, (int)fmaxf(fminf(floorf(hx + 1.5f), 70000.0f), -2.0f)));
            int y0 = max(0, min(65535, (int)fmaxf(fminf(ceilf(ly - 1.5f), 70000.0f), -1.0f)));
            int y1 = max(-1, min(65535, (int)fmaxf(fminf(floorf(hy + 1.5f), 70000.0f), -2.0f)));
            if (x1 < x0 || y1 < y0) { x0 = 1; x1 = 0; y0 = 1; y1 = 0; }   // empty on screen
            if (lx == lx && hx == hx && ly == ly && hy == hy) {           // NaN coordinates keep the full range
                bbx = (uint32_t)x0 | ((uint32_t)x1 << 16);
                bby = (uint32_t)y0 | ((uint32_t)y1 << 16);
            }
        }
        float max_z = a0.z, min_z = a0.z;
        max_z = fmaxf(max_z, a1.z); min_z = fminf(min_z, a1.z);
        max_z = fmaxf(max_z, a2.z); min_z = fminf(min_z, a2.z);

        uint32_t touched = 0;
        int x0 = 0, y0 = 0, x1 = 0, y1 = 0;
        if (!(max_z < -1.0f || min_z > 1.0f)) {
            tile_rect(make_float2(a0.x, a0.y), make_float2(a1.x, a1.y), make_float2(a2.x, a2.y), gx, gy, x0, y0, x1, y1);
            if (x1 > x0 && y1 > y0) touched = (uint32_t)(y1 - y0) * (uint32_t)(x1 - x0);
        }
        float mn = (min_z + 1.0f) * 0.5f;
        if (mn < 0.0f) mn = 0.0f;
        if (mn > 1.0f) mn = 1.0f;
        float mx = (max_z + 1.0f) * 0.5f;
        if (mx < 0.0f) mx = 0.0f;
        if (mx > 1.0f) mx = 1.0f;

        size_t bf = (size_t)b * F + f;
        tiles_touched[bf] = touched;
        depth_key[bf] = __float_as_uint(mn);
        sort_key[0] = __float_as_uint(mn);
        rect[bf] = make_uint2((uint32_t)x0 | ((uint32_t)x1 << 16), (uint32_t)y0 | ((uint32_t)y1 << 16));

        const float* q0 = verts + 3 * (size_t)i0; const float* q1 = verts + 3 * (size_t)i1; const float* q2 = verts + 3 * (size_t)i2;
        uint4* r = s_rec + tid * 4;
        r[0] = make_uint4(__float_as_uint(q0[0]), __float_as_uint(q0[1]), __float_as_uint(q0[2]), __float_as_uint(q1[0]));
        r[1] = make_uint4(__float_as_uint(q1[1]), __float_as_uint(q1[2]), __float_as_uint(q2[0]), __float_as_uint(q2[1]));
        r[2] = make_uint4(__float_as_uint(q2[2]), __float_as_uint(mn), __float_as_uint(mx), bbx);
        r[3] = make_uint4(bby, 0u, 0u, 0u);
    }
    __syncthreads();
    size_t nvalid = (f0 + 256 <= (size_t)F) ? 256 : ((size_t)F > f0 ? (size_t)F - f0 : 0);
    uint4* dst = reinterpret_cast<uint4*>(records + (size_t)b * F + f0);
    for (size_t i = tid; i < nvalid * 4; i += 256) dst[i] = s_rec[i];
    if (HIST) {
        const bool sort_valid[1] = { f < (size_t)F };
        rs_pre_add<1>(s_hist, sort_key, sort_valid, sp);
        rs_pre_finish(s_hist, sp, gridDim.x * gridDim.y);
    }
}

int tet_preprocess_faces(int B, int P, int F, int W, int H, const int* faces, const float4* vimg, const float* verts,
                         uint32_t* tiles_touched, uint32_t* depth_key, uint2* rect, TetFaceRec* rec,
                         const SortPre& sp, cudaStream_t stream)
{
    if (B <= 0 || F <= 0) return 0;
    int gx = (W + DMR_TILE - 1) / DMR_TILE, gy = (H + DMR_TILE - 1) / DMR_TILE;
    dim3 grid((F + 255) / 256, B);
    ProfScope prof(ST_FACES, stream);
    if (sp.npass > 0)
        DMR_CUDA(dmr_launch(tet_preprocess_faces_kernel<true>, dim3(grid), dim3(256), 0, stream, B, P, F, gx, gy, faces, vimg, verts, tiles_touched,
                                                                   depth_key, rect, rec, sp));
    else
        DMR_CUDA(dmr_launch(tet_preprocess_faces_kernel<false>, dim3(grid), dim3(256), 0, stream, B, P, F, gx, gy, faces, vimg, verts, tiles_touched,
                                                                    depth_key, rect, rec, sp));
    DMR_LAUNCH_CHECK("tet_preprocess_faces_kernel");
    return 0;
}

}  // namespace dmr
