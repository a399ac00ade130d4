// tet.cuh -- records, workspace layouts and launch interface of the tet renderer.
#pragma once
#include "common.cuh"
#include "radix_sort.cuh"

namespace dmr {

// Per-(view,face) record staged by the first-intersection kernel
// (replaces the gathers of cuda_renderer/forward.cu:368-381): 64 bytes.
// bbox = conservative screen-space pixel bounds (projected vertices +-1 px) used to skip
// faces no pixel of a warp's block / no pixel at all can hit; 0..65535 (= no culling) when
// a vertex is not safely in front of the camera (w <= 1e-4), where the projected
// vertices do not bound the visible part of the triangle.
struct __align__(16) TetFaceRec {
    float p0[3], p1[3], p2[3];   // world positions in faces[] order
    float min_depth, max_depth;  // clamped (z+1)/2, cuda_renderer/forward.cu:253-259
    uint32_t bbox_x, bbox_y;     // lo | hi << 16, inclusive pixel bounds
    uint32_t pad[3];
};
static_assert(sizeof(TetFaceRec) == 64, "TetFaceRec must be 4 x 16 bytes");

// View-independent per-tet adjacency record used by the ray march.  The
// reference re-gathers, at every step, tet_faces -> faces -> verts (3 dependent
// levels), the tet's 4 vertices four times over and face_tets
// (cuda_renderer/forward.cu:672-768, ~670 B per step).  One 128-byte record (exactly
// one cache line) per tet turns that into a single dependent load.
//
// The march is bound by the bytes each lane pulls through L1 per step (ncu: l1tex data pipe 55-90%
// busy, DRAM < 10%), so the four sides do not carry their own copies of the vertices (the first
// version: 224 B): vert[k] is the tet vertex OPPOSITE side k, side k's triangle is made of the other
// three, and a 4-bit order code says in which order faces[] lists them -- the hit test must see
// (p0,p1,p2) in the reference's order to reproduce its (t,u,v) bits.  A tet whose sides are not made
// of its own four vertices (inconsistent input tables, or two coincident vertices) cannot be represented:
// it is flagged (code 0xF) and the march tests its sides with the vertices of the per-(view, face) records --
// the triangle the reference gathers through faces[] -- on an out-of-line path (tet_side_hit_irregular).
struct __align__(16) TetRec {
    int face[4];          // tet_faces[4*t + k]
    uint32_t next[4];     // bits 0..27: 1 + first entry of face_tets[face[k]] that is neither t nor -1 (0 = none)
                          // bits 28..31: order code a | b << 2: p0 = cyc[a], p1 = cyc[b], p2 = cyc[3-a-b] with
                          //              cyc = (vert[(k+1)&3], vert[(k+2)&3], vert[(k+3)&3]); 0xF = irregular tet
    float vert[4][3];     // vert[k] = position of the vertex opposite side k
    float nrm[4][3];      // outward unit normal of side k w.r.t. this tet
};
static_assert(sizeof(TetRec) == 128, "TetRec must be one 128-byte line");
#define DMR_TET_MAX_TETS ((1 << 28) - 2)

// View-independent per-face shading record: 64 bytes.
struct __align__(16) TetShade {
    float c0[3], c1[3], c2[3];   // vertex colours
    float opacity;
    float log1m_opacity;         // logf(1 - opacity)      -- the first 48 bytes are all the forward march reads
    int i0, i1, i2;              // vertex ids (gradient scatter)
    int t0, t1;                  // face_tets[2f], face_tets[2f+1]
};
static_assert(sizeof(TetShade) == 64, "TetShade must be 4 x 16 bytes");

// Face buffer of the tet renderer.  The view-independent adjacency records (TetRec[T]) are NOT part of it: they
// depend only on the geometry tables, so they live in a separate `tet_records` buffer the caller may keep across
// calls while the geometry stays the same (dmr_tet_records_bytes, dmr_tet_forward_bin's tet_records_valid).  With
// vertex-position gradients (dmr_tet_backward_vertex) `verts` changes in every optimisation step, and the records
// have to be rebuilt whenever it does.  The backward scratch is the caller's workspace (the state buffers of the
// forward call stay read-only).
struct TetFaceLayout {
    FaceBinLayout bin;
    size_t face_rec, shade, total;
    __host__ static TetFaceLayout make(size_t BF, size_t F)
    {
        TetFaceLayout L;
        L.bin = FaceBinLayout::make(BF);
        size_t o = L.bin.end;
        L.face_rec = o;      o = align_up(o + sizeof(TetFaceRec) * BF, 256);
        L.shade = o;         o = align_up(o + sizeof(TetShade) * F, 256);
        L.total = o + 256;
        return L;
    }
};

// Face trail: the forward march records, for every face it composites, the face id AND the hit parameters
// (t, u, v) it composited with -- one 16-byte entry, step-major (trail[k * BI + pixel], coalesced across a warp) --
// so that the backward pass walks the SAME faces in reverse with independent, prefetchable loads instead of
// re-marching through the adjacency with one dependent load chain per step (cuda_renderer/backward.cu:382-477),
// and needs neither the face's vertices (48 B per step through L1, which bounds the march) nor a second
// ray/triangle test per step: the values ARE the forward pass's bits.  Only the first `cap` steps of a ray are
// recorded; rays that composite more faces re-march the part beyond the cap exactly as before.
// cap: 512 steps while the trail stays below 2 GiB, never less than 32 (debug override for tests).
extern int g_tet_trail_cap_override;
__host__ inline size_t tet_trail_cap(size_t BI)
{
    if (g_tet_trail_cap_override > 0) return (size_t)g_tet_trail_cap_override;
    if (BI == 0) return 32;
    size_t cap = ((size_t)2048 << 20) / (16 * BI);
    return cap > 512 ? 512 : (cap < 32 ? 32 : cap);
}

struct TetImageLayout {
    size_t n_contrib, ranges, final_log_T, prev_log_T, first_face, first_tet, last_face, last_tet, active, jitter, fi_key, trail, trail_cap, total;
    __host__ static TetImageLayout make(size_t B, size_t W, size_t H)
    {
        TetImageLayout L;
        size_t BI = B * W * H;
        size_t tiles = B * ((W + DMR_TILE - 1) / DMR_TILE) * ((H + DMR_TILE - 1) / DMR_TILE);
        size_t o = 0;
        L.n_contrib = o;   o = align_up(o + 4 * BI, 256);
        L.ranges = o;      o = align_up(o + 8 * tiles, 256);
        L.final_log_T = o; o = align_up(o + 4 * BI, 256);
        L.prev_log_T = o;  o = align_up(o + 4 * BI, 256);
        L.first_face = o;  o = align_up(o + 4 * BI, 256);
        L.first_tet = o;   o = align_up(o + 4 * BI, 256);
        L.last_face = o;   o = align_up(o + 4 * BI, 256);
        L.last_tet = o;    o = align_up(o + 4 * BI, 256);
        L.active = o;      o = align_up(o + BI, 256);
        L.jitter = o;      o = align_up(o + 8 * BI, 256);   // float2 pixel coordinate, written only when seed > 0
        // first-intersect partial results: u64 (t bits << 32 | list position) per pixel, directly followed by
        // u32 max-depth bits per pixel (one memset)
        L.fi_key = o;      o = align_up(o + 12 * BI, 256);
        L.trail_cap = tet_trail_cap(BI);
        L.trail = o;       o = align_up(o + 16 * BI * L.trail_cap, 256);
        L.total = o + 256;
        return L;
    }
};

struct TetParams {
    int B, P, F, T, W, H;
    const float* mv; const float* proj; const float* inv_mv; const float* inv_proj;
    const float* faces_intense;   // [B,F]
    const float* bg;
    // records
    const TetFaceRec* face_rec;   // [B*F]
    const TetRec* tet_rec;        // [T]
    const TetShade* shade;        // [F]
    // binning
    const uint2* ranges; const uint32_t* face_list;
    // per-pixel state
    const float2* jitter;         // null when ray_random_seed <= 0
    int* first_face; int* first_tet; int* last_face; int* last_tet;
    float* final_log_T; float* prev_log_T; uint32_t* n_contrib; uint8_t* active;
    int4* trail; int trail_cap;   // [trail_cap][B*W*H] { face id | flag, t, u, v (float bits) } in march order
    unsigned long long* fi_key;   // [B*W*H] split first-intersect: per-pixel atomicMin slot
    uint32_t* fi_close;           // [B*W*H] smallest max depth (float bits) of any hit found so far
    int fi_split;                 // CTAs per tile in tet_first_intersect_kernel
    // outputs
    float* out_color; float* out_depth; float* out_active;
    // backward
    const float* dL_dcolor; const float* dL_ddepth;
    float* dL_dverts_color; float* dL_dfaces_opacity;
    float4* grad_vacc;            // [P] zeroed scratch: per-vertex colour gradient (xyz), summed over views
    // deterministic mode only (tet_march_backward_deterministic): zeroed 64-bit fixed-point accumulators (det.cuh)
    const uint32_t* det_gmax;     // [2]: bits of max |cotangent|, overflow word
    long long* det_vert;          // [P,4]: dL_dverts_color rgb, -
    long long* det_fopa;          // [F]
};

// Outputs of the vertex-position backward (dmr_tet_backward_vertex), a kernel argument of its own so that TetParams, and
// with it the parameter layout of every other kernel, stays as it is.
struct TetVertGrad {
    float* dL_dverts;             // [P,3], added to
    float4* grad_pacc;            // default mode: [P] zeroed scratch, per-vertex position gradient (xyz) summed over views
    long long* det_pos;           // deterministic mode: [P,4] zeroed fixed-point dL_dverts xyz, - (TetDetLayout::pos)
};

// Outputs of the face-intensity backward (dmr_tet_backward_intensity), a kernel argument of its own like TetVertGrad.
struct TetIntGrad {
    float* dL_dfint;              // [B,F], added to (default mode: by the march kernels directly)
    long long* det_fint;          // deterministic mode: [B,F] zeroed fixed-point low words, behind the mode's scratch
    ptrdiff_t det_hi;             // ... and the element offset of their high words (B*F: a [B,F] block outgrows
                                  // TetDetLayout::hi_offset, which is sized for P and F)
};

// Camera gradients of the backward march: one record of DMR_TET_CAM_REC floats per (view, march CTA of 8 x 8 pixels),
// written by every CTA (layout: tet_march_bwd_cam, tet_kernels.cu).
#define DMR_TET_CAM_REC 32
__host__ __device__ inline size_t tet_cam_records(size_t B, int W, int H) { return B * (size_t)((W + 7) / 8) * ((H + 7) / 8); }

struct TetDetLayout {             // workspace of the deterministic backward pass
    size_t gmax, vert, fopa, hi, total;   // low words vert..fopa, their high words mirrored at hi
    // vertex-position gradients: a [P,4] block appended behind `total`, its high words at the same element offset
    // (hi_offset) as every other accumulator's; total_pos is the workspace of that mode
    size_t pos, total_pos;
    __host__ __device__ static TetDetLayout make(size_t P, size_t F)
    {
        TetDetLayout L;
        size_t o = 0;
        L.gmax = o; o = align_up(o + 4, 256);
        L.vert = o; o = align_up(o + 8 * 4 * P, 256);
        L.fopa = o; o = align_up(o + 8 * F, 256);
        L.hi = o;   o += o - L.vert;
        L.total = o;
        L.pos = o;
        L.total_pos = align_up(o + (L.hi - L.vert) + 8 * 4 * P, 256);
        return L;
    }
    // element offset of an accumulator's high word from its low word (det.cuh)
    __host__ __device__ static ptrdiff_t hi_offset(size_t P, size_t F)
    {
        const TetDetLayout L = make(P, F);
        return (ptrdiff_t)((L.hi - L.vert) / 8);
    }
};

int preprocess_points(int B, int P, int W, int H, const float* verts, const float* mv, const float* proj,
                      const float* verts_depth, int depth_mode, float4* vimg, cudaStream_t stream);
int depth_chain(int B, int P, const float* verts, const float* mv, const float* proj, const float* dL_dvdepth,
                float* dL_dverts, cudaStream_t stream);
// camera variant of the fused-depth chain: += dL_dmv[B,16], dL_dproj[B,16]; workspace of depth_chain_camera_bytes
size_t depth_chain_camera_bytes(int B, int P);
int depth_chain_camera(int B, int P, const float* verts, const float* mv, const float* proj, const float* dL_dvdepth,
                       float* dL_dmv, float* dL_dproj, void* workspace, cudaStream_t stream);
int tet_preprocess_faces(int B, int P, int F, int W, int H, const int* faces, const float4* vimg, const float* verts,
                         uint32_t* tiles_touched, uint32_t* depth_key, uint2* rect, TetFaceRec* rec,
                         const SortPre& face_sort, cudaStream_t stream);
// tet_rec == nullptr: the adjacency records are valid already (cached by the caller), only the shading records
// (colour / opacity change every step) are rebuilt
int tet_build_records(int P, int F, int T, const float* verts, const int* faces, const float* verts_color,
                      const float* faces_opacity, const int* tets, const int* face_tets, const int* tet_faces,
                      TetRec* tet_rec, TetShade* shade, cudaStream_t stream);
// first_view: index, in the whole job, of the call's view 0; it offsets the cuRAND subsequence of every pixel
int tet_jitter(int B, int W, int H, int seed, int first_view, float2* jitter, cudaStream_t stream);
int tet_first_intersect(const TetParams& p, cudaStream_t stream);
int tet_march_forward(const TetParams& p, cudaStream_t stream);
// cam_rec != nullptr: the camera-gradient kernels, which also store one DMR_TET_CAM_REC-float record per (view, march
// CTA) there
// vert != nullptr: the vertex-position kernels, which also add dL/dverts to vert->dL_dverts
// fint != nullptr: the face-intensity kernels, which also add dL/dfaces_intense to fint->dL_dfint
// dL_dalpha != nullptr: the alpha-cotangent instantiations of the same mode ([B,H,W] cotangent of the alpha image)
int tet_march_backward(const TetParams& p, cudaStream_t stream, float* cam_rec = nullptr, const TetVertGrad* vert = nullptr,
                       const TetIntGrad* fint = nullptr, const float* dL_dalpha = nullptr);
int tet_march_backward_deterministic(const TetParams& p, cudaStream_t stream, float* cam_rec = nullptr,
                                     const TetVertGrad* vert = nullptr, const TetIntGrad* fint = nullptr,
                                     const float* dL_dalpha = nullptr);
// records of a view -> += dL_dmv[B,16], dL_dproj[B,16]
int tet_camera_finish(const TetParams& p, const float* cam_rec, float* dL_dmv, float* dL_dproj, cudaStream_t stream);

}  // namespace dmr
