// capi_tet.cu -- extern "C" entry points of the tet renderer (include/dmesh_b200.h).
// Stage sequencing of CudaRenderer::Renderer::forward / backward
// (cuda_renderer/renderer_impl.cu:193-410, 413-498) without the per-stage
// device synchronisation.
#include "tet.cuh"
#include "../../include/dmesh_b200.h"

using namespace dmr;

namespace dmr { int g_tet_trail_cap_override = 0; }
static int g_tet_first_split_override = 0;

namespace {

template <typename T>
T* at(void* base, size_t off) { return reinterpret_cast<T*>(static_cast<unsigned char*>(base) + off); }
template <typename T>
const T* at(const void* base, size_t off) { return reinterpret_cast<const T*>(static_cast<const unsigned char*>(base) + off); }

bool tet_sizes_ok(long long B, long long P, long long F, long long T, long long W, long long H)
{
    if (B < 0 || P < 0 || F < 0 || T < 0 || W <= 0 || H <= 0) { set_error("negative or zero size"); return false; }
    if (B * P >= (1LL << 31) || B * F >= (1LL << 31) || B * W * H >= (1LL << 31) || T > DMR_TET_MAX_TETS) {
        set_error("B*P, B*F and B*W*H must stay below 2^31 and T below 2^28 - 1");
        return false;
    }
    if ((W + DMR_TILE - 1) / DMR_TILE >= 65536 || (H + DMR_TILE - 1) / DMR_TILE >= 65536) {
        set_error("image too large for 16-bit tile coordinates");
        return false;
    }
    return true;
}

// scratch of the backward pass of either mode (dmr_tet_backward_workspace_bytes without its slack,
// dmr_tet_backward_deterministic_bytes); vert: with the per-vertex position accumulator (default mode: a second
// float4[P] right behind the colour one; deterministic mode: TetDetLayout::pos); fint_n: number of fixed-point
// face-intensity accumulators (deterministic mode: B*F low words, then B*F high words, behind the rest; the default
// mode needs none)
size_t tet_bwd_scratch_bytes(int P, int F, bool deterministic, bool vert = false, size_t fint_n = 0)
{
    if (deterministic) {
        const TetDetLayout L = TetDetLayout::make((size_t)P, (size_t)F);
        const size_t s = vert ? L.total_pos : L.total;
        return fint_n ? align_up(s, 256) + 2 * sizeof(long long) * fint_n : s;
    }
    return sizeof(float4) * (size_t)P * (vert ? 2 : 1);
}

// workspace of the camera-gradient backward: the mode's own scratch, then DMR_TET_CAM_REC floats per (view, march CTA)
size_t tet_cam_bytes(int B, int P, int F, int W, int H, bool deterministic, bool vert = false, size_t fint_n = 0)
{
    return align_up(tet_bwd_scratch_bytes(P, F, deterministic, vert, fint_n), 256) +
           align_up(sizeof(float) * DMR_TET_CAM_REC * tet_cam_records((size_t)B, W, H), 256) + 256;
}

// workspace of the vertex-position backward, with or without camera gradients
size_t tet_vert_bytes(int B, int P, int F, int W, int H, bool deterministic, bool cam)
{
    return cam ? tet_cam_bytes(B, P, F, W, H, deterministic, true) : tet_bwd_scratch_bytes(P, F, deterministic, true) + 256;
}

// workspace of the face-intensity backward, with or without camera and vertex-position gradients
size_t tet_int_bytes(int B, int P, int F, int W, int H, bool deterministic, bool cam, bool vert)
{
    const size_t n = (size_t)B * F;
    return cam ? tet_cam_bytes(B, P, F, W, H, deterministic, vert, n) : tet_bwd_scratch_bytes(P, F, deterministic, vert, n) + 256;
}

}  // namespace

extern "C" {

int dmr_tet_state_bytes(int B, int P, int F, int T, int W, int H, size_t out[3])
{
    if (!out) { set_error("out is null"); return DMR_EINVAL; }
    if (!tet_sizes_ok(B, P, F, T, W, H)) return DMR_ETOOLARGE;
    out[0] = align_up(sizeof(float4) * (size_t)B * P, 256) + 256;
    out[1] = TetFaceLayout::make((size_t)B * F, (size_t)F).total;
    out[2] = TetImageLayout::make(B, W, H).total;
    return DMR_OK;
}

int dmr_tet_forward_bin(int B, int P, int F, int T, int W, int H, const float* verts, const int* faces,
                        const float* verts_color, const float* faces_opacity, const float* mv_mats,
                        const float* proj_mats, const int* tets, const int* face_tets, const int* tet_faces,
                        void* point_buffer, void* face_buffer, void* tet_records, int tet_records_valid,
                        int32_t* num_rendered_host, dmr_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!tet_sizes_ok(B, P, F, T, W, H)) return DMR_ETOOLARGE;
    if (!num_rendered_host) { set_error("num_rendered_host is null"); return DMR_EINVAL; }
    if (B == 0 || P == 0 || F == 0) { *num_rendered_host = 0; return DMR_OK; }
    if (!verts || !faces || !verts_color || !faces_opacity || !mv_mats || !proj_mats || !face_tets ||
        (T > 0 && (!tets || !tet_faces || !tet_records)) || !point_buffer || !face_buffer) { set_error("null pointer"); return DMR_EINVAL; }
    const size_t BF = (size_t)B * F;
    TetFaceLayout L = TetFaceLayout::make(BF, (size_t)F);
    float4* vimg = static_cast<float4*>(point_buffer);
    int rc;
    SortPre face_sort;
    if ((rc = bin_faces_begin(BF, face_buffer, L.bin, &face_sort, stream))) return rc;
    if ((rc = preprocess_points(B, P, W, H, verts, mv_mats, proj_mats, nullptr, 0, vimg, stream))) return rc;
    if ((rc = tet_preprocess_faces(B, P, F, W, H, faces, vimg, verts, at<uint32_t>(face_buffer, L.bin.tiles_touched),
                                   at<uint32_t>(face_buffer, L.bin.depth_key), at<uint2>(face_buffer, L.bin.rect),
                                   at<TetFaceRec>(face_buffer, L.face_rec), face_sort, stream)))
        return rc;
    if ((rc = bin_faces(BF, face_buffer, L.bin, num_rendered_host, stream))) return rc;
    // view-independent march records; independent of the scan, enqueued behind it.  (Measured and rejected:
    // building them on a second stream concurrently with the binning chain -- the chain's preprocess and sort
    // kernels are HBM-bound like the record builders, they just slow each other down: C3 forward 1.78 ms both ways.)
    if ((rc = tet_build_records(P, F, T, verts, faces, verts_color, faces_opacity, tets, face_tets, tet_faces,
                                tet_records_valid ? nullptr : static_cast<TetRec*>(tet_records),
                                at<TetShade>(face_buffer, L.shade), stream)))
        return rc;
    return DMR_OK;
}

static void fill_params(TetParams& p, int B, int P, int F, int T, int W, int H, int seed, const float* bg,
                        const float* mv, const float* proj, const float* inv_mv, const float* inv_proj,
                        const float* faces_intense, const void* face_buffer, const void* tet_records,
                        const void* image_buffer)
{
    TetFaceLayout FL = TetFaceLayout::make((size_t)B * F, (size_t)F);
    TetImageLayout IL = TetImageLayout::make(B, W, H);
    p = TetParams{};
    p.B = B; p.P = P; p.F = F; p.T = T; p.W = W; p.H = H;
    p.mv = mv; p.proj = proj; p.inv_mv = inv_mv; p.inv_proj = inv_proj;
    p.faces_intense = faces_intense; p.bg = bg;
    p.face_rec = at<TetFaceRec>(face_buffer, FL.face_rec);
    p.tet_rec = static_cast<const TetRec*>(tet_records);
    p.shade = at<TetShade>(face_buffer, FL.shade);
    p.ranges = at<uint2>(image_buffer, IL.ranges);
    p.jitter = seed > 0 ? at<float2>(image_buffer, IL.jitter) : nullptr;
    void* ib = const_cast<void*>(image_buffer);
    p.first_face = at<int>(ib, IL.first_face);
    p.first_tet = at<int>(ib, IL.first_tet);
    p.last_face = at<int>(ib, IL.last_face);
    p.last_tet = at<int>(ib, IL.last_tet);
    p.final_log_T = at<float>(ib, IL.final_log_T);
    p.prev_log_T = at<float>(ib, IL.prev_log_T);
    p.n_contrib = at<uint32_t>(ib, IL.n_contrib);
    p.active = at<uint8_t>(ib, IL.active);
    p.trail = at<int4>(ib, IL.trail);
    p.trail_cap = (int)IL.trail_cap;
    p.fi_key = at<unsigned long long>(ib, IL.fi_key);
    p.fi_close = reinterpret_cast<uint32_t*>(p.fi_key + (size_t)B * W * H);
    // CTAs per tile of the first-intersection search.  Measured at C3 (1024 tiles), later parts scheduled
    // after all part-0 CTAs: 1 -> 260 us, 2 -> 189 us, 4 -> 166 us, 8 -> 168 us.  (With the parts of a tile
    // adjacent in the grid: 2 -> 200, 4 -> 275, 8 -> 433 us -- every interior tile then repeats rounds a single
    // CTA would have skipped after its first hits.)
    {
        const size_t tiles = (size_t)B * ((W + DMR_TILE - 1) / DMR_TILE) * ((H + DMR_TILE - 1) / DMR_TILE);
        p.fi_split = tiles <= 4096 ? 4 : tiles <= 16384 ? 2 : 1;
        if (g_tet_first_split_override > 0) p.fi_split = g_tet_first_split_override;
    }
}

int dmr_tet_forward_render(int B, int P, int F, int T, int W, int H, int R, int ray_random_seed,
                           const float* background, const float* mv_mats, const float* proj_mats,
                           const float* inv_mv_mats, const float* inv_proj_mats, const float* faces_intense,
                           const void* point_buffer, void* face_buffer, const void* tet_records, void* binning_buffer,
                           void* image_buffer, float* out_color, float* out_depth, float* out_active, dmr_stream_t stream)
{
    return dmr_tet_forward_render_views(B, P, F, T, W, H, R, ray_random_seed, 0, background, mv_mats, proj_mats,
                                        inv_mv_mats, inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records,
                                        binning_buffer, image_buffer, out_color, out_depth, out_active, stream);
}

int dmr_tet_forward_render_views(int B, int P, int F, int T, int W, int H, int R, int ray_random_seed, int first_view,
                                 const float* background, const float* mv_mats, const float* proj_mats,
                                 const float* inv_mv_mats, const float* inv_proj_mats, const float* faces_intense,
                                 const void* point_buffer, void* face_buffer, const void* tet_records,
                                 void* binning_buffer, void* image_buffer, float* out_color, float* out_depth,
                                 float* out_active, dmr_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (first_view < 0) { set_error("first_view must not be negative (got %d)", first_view); return DMR_EINVAL; }
    if (!tet_sizes_ok(B, P, F, T, W, H) || R < 0) return DMR_ETOOLARGE;
    if (B == 0) return DMR_OK;
    if (!background || !mv_mats || !proj_mats || !inv_mv_mats || !inv_proj_mats || !face_buffer || !image_buffer ||
        !out_color || !out_depth || !out_active || (F > 0 && !faces_intense) || (R > 0 && !binning_buffer) ||
        (T > 0 && !tet_records)) {
        set_error("null pointer");
        return DMR_EINVAL;
    }
    (void)point_buffer;
    TetFaceLayout FL = TetFaceLayout::make((size_t)B * F, (size_t)F);
    TetImageLayout IL = TetImageLayout::make(B, W, H);
    uint2* ranges = at<uint2>(image_buffer, IL.ranges);
    int rc;
    TetParams p;
    fill_params(p, B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                faces_intense, face_buffer, tet_records, image_buffer);
    if (ray_random_seed > 0)
        if ((rc = tet_jitter(B, W, H, ray_random_seed, first_view, at<float2>(image_buffer, IL.jitter), stream))) return rc;
    if ((rc = bin_instances(B, F, W, H, (size_t)R, face_buffer, FL.bin, binning_buffer, ranges, stream))) return rc;
    if (R > 0) p.face_list = at<uint32_t>(binning_buffer, BinningLayout::make((size_t)R).vals_sorted);
    p.out_color = out_color; p.out_depth = out_depth; p.out_active = out_active;
    if ((rc = tet_first_intersect(p, stream))) return rc;
    if ((rc = tet_march_forward(p, stream))) return rc;
    return DMR_OK;
}

static int tet_backward_impl(int B, int P, int F, int T, int W, int H, int ray_random_seed, const float* background,
                             const float* mv_mats, const float* proj_mats, const float* inv_mv_mats,
                             const float* inv_proj_mats, const float* faces_intense, const void* point_buffer,
                             const void* face_buffer, const void* tet_records, const void* image_buffer,
                             const float* dL_dcolor, const float* dL_ddepth, float* dL_dverts_color,
                             float* dL_dfaces_opacity, void* workspace, size_t workspace_bytes, bool deterministic,
                             dmr_stream_t stream_, float* dL_dmv = nullptr, float* dL_dproj = nullptr,
                             float* dL_dverts = nullptr, float* dL_dfaces_intense = nullptr,
                             const float* dL_dalpha = nullptr)
{
    const bool cam = dL_dmv != nullptr;
    const bool vert = dL_dverts != nullptr;
    const bool fint = dL_dfaces_intense != nullptr;
    const size_t fint_n = fint ? (size_t)B * F : 0;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!tet_sizes_ok(B, P, F, T, W, H)) return DMR_ETOOLARGE;
    if (B == 0 || F == 0 || T == 0) return DMR_OK;
    if (!background || !mv_mats || !proj_mats || !inv_mv_mats || !inv_proj_mats || !faces_intense || !face_buffer ||
        !tet_records || !image_buffer || !dL_dcolor || !dL_ddepth || !dL_dverts_color || !dL_dfaces_opacity) {
        set_error("null pointer");
        return DMR_EINVAL;
    }
    (void)point_buffer;
    if (fint) {
        const size_t need = tet_int_bytes(B, P, F, W, H, deterministic, cam, vert);
        if (!workspace || workspace_bytes < need) {
            set_error("intensity-gradient backward needs a workspace of %zu bytes (dmr_tet_backward_intensity_bytes)", need);
            return DMR_EINVAL;
        }
    }
    if (vert) {
        const size_t need = tet_vert_bytes(B, P, F, W, H, deterministic, cam);
        if (!workspace || workspace_bytes < need) {
            set_error("vertex-gradient backward needs a workspace of %zu bytes (dmr_tet_backward_vertex_bytes)", need);
            return DMR_EINVAL;
        }
    }
    // camera gradients: one record per (view, march CTA) behind the mode's own scratch, written by every CTA, so it is
    // not cleared
    float* cam_rec = nullptr;
    if (cam) {
        const size_t need = tet_cam_bytes(B, P, F, W, H, deterministic, vert, fint_n);
        if (!workspace || workspace_bytes < need) {
            set_error("camera-gradient backward needs a workspace of %zu bytes (dmr_tet_backward_camera_bytes)", need);
            return DMR_EINVAL;
        }
        cam_rec = at<float>(workspace, align_up(tet_bwd_scratch_bytes(P, F, deterministic, vert, fint_n), 256));
    }
    TetVertGrad vg{ dL_dverts, nullptr, nullptr };
    TetIntGrad ig{ dL_dfaces_intense, nullptr, (ptrdiff_t)fint_n };
    void* det_workspace = workspace;
    const size_t det_workspace_bytes = workspace_bytes;
    TetParams p;
    fill_params(p, B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                faces_intense, face_buffer, tet_records, image_buffer);
    p.dL_dcolor = dL_dcolor; p.dL_ddepth = dL_ddepth;
    p.dL_dverts_color = dL_dverts_color; p.dL_dfaces_opacity = dL_dfaces_opacity;
    p.det_gmax = nullptr; p.det_vert = nullptr; p.det_fopa = nullptr;
    if (deterministic) {
        TetDetLayout DL = TetDetLayout::make((size_t)P, (size_t)F);
        if (!det_workspace || det_workspace_bytes < DL.total) {
            set_error("deterministic backward needs a workspace of %zu bytes (dmr_tet_backward_deterministic_bytes)", DL.total);
            return DMR_EINVAL;
        }
        p.det_gmax = at<uint32_t>(det_workspace, DL.gmax);
        p.det_vert = at<long long>(det_workspace, DL.vert);
        p.det_fopa = at<long long>(det_workspace, DL.fopa);
        p.grad_vacc = nullptr;
        vg.det_pos = at<long long>(det_workspace, DL.pos);
        ig.det_fint = at<long long>(det_workspace, align_up(vert ? DL.total_pos : DL.total, 256));
        DMR_CUDA(cudaMemsetAsync(det_workspace, 0, tet_bwd_scratch_bytes(P, F, true, vert, fint_n), stream));
        int rc = tet_march_backward_deterministic(p, stream, cam_rec, vert ? &vg : nullptr, fint ? &ig : nullptr, dL_dalpha);
        if (rc || !cam) return rc;
        return tet_camera_finish(p, cam_rec, dL_dmv, dL_dproj, stream);
    }
    // backward scratch: float4 per vertex (colour gradient, 16-byte aligned for red.v4) in the caller's workspace
    if (!workspace || workspace_bytes < sizeof(float4) * (size_t)P) {
        set_error("backward needs a workspace of %zu bytes (dmr_tet_backward_workspace_bytes)", sizeof(float4) * (size_t)P);
        return DMR_EINVAL;
    }
    p.grad_vacc = static_cast<float4*>(workspace);
    vg.grad_pacc = p.grad_vacc + P;
    DMR_CUDA(cudaMemsetAsync(p.grad_vacc, 0, sizeof(float4) * (size_t)P * (vert ? 2 : 1), stream));
    int rc = tet_march_backward(p, stream, cam_rec, vert ? &vg : nullptr, fint ? &ig : nullptr, dL_dalpha);
    if (rc || !cam) return rc;
    return tet_camera_finish(p, cam_rec, dL_dmv, dL_dproj, stream);
}

int dmr_tet_backward(int B, int P, int F, int T, int W, int H, int ray_random_seed, const float* background,
                     const float* mv_mats, const float* proj_mats, const float* inv_mv_mats,
                     const float* inv_proj_mats, const float* faces_intense, const void* point_buffer,
                     const void* face_buffer, const void* tet_records, const void* image_buffer, const float* dL_dcolor,
                     const float* dL_ddepth, float* dL_dverts_color, float* dL_dfaces_opacity, void* workspace,
                     size_t workspace_bytes, dmr_stream_t stream)
{
    return tet_backward_impl(B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats,
                             inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records, image_buffer, dL_dcolor,
                             dL_ddepth, dL_dverts_color, dL_dfaces_opacity, workspace, workspace_bytes, false, stream);
}

size_t dmr_tet_backward_workspace_bytes(int P) { return P < 0 ? 0 : sizeof(float4) * (size_t)P + 256; }

int dmr_tet_build_records(int P, int F, int T, const float* verts, const int* faces, const int* tets,
                          const int* face_tets, const int* tet_faces, void* tet_records, dmr_stream_t stream)
{
    if (P < 0 || F < 0 || T < 0 || T > DMR_TET_MAX_TETS) { set_error("bad size"); return DMR_EINVAL; }
    if (T == 0) return DMR_OK;
    if (!verts || !faces || !tets || !face_tets || !tet_faces || !tet_records) { set_error("null pointer"); return DMR_EINVAL; }
    return tet_build_records(P, F, T, verts, faces, nullptr, nullptr, tets, face_tets, tet_faces,
                             static_cast<TetRec*>(tet_records), nullptr, (cudaStream_t)stream);
}

size_t dmr_tet_records_bytes(int T) { return T < 0 ? 0 : align_up(sizeof(TetRec) * (size_t)T, 256) + 256; }

size_t dmr_tet_backward_deterministic_bytes(int P, int F)
{
    if (P < 0 || F < 0) return 0;
    return TetDetLayout::make((size_t)P, (size_t)F).total;
}

int dmr_tet_backward_deterministic(int B, int P, int F, int T, int W, int H, int ray_random_seed,
                                   const float* background, const float* mv_mats, const float* proj_mats,
                                   const float* inv_mv_mats, const float* inv_proj_mats, const float* faces_intense,
                                   const void* point_buffer, const void* face_buffer, const void* tet_records,
                                   const void* image_buffer, const float* dL_dcolor, const float* dL_ddepth,
                                   float* dL_dverts_color, float* dL_dfaces_opacity, void* workspace,
                                   size_t workspace_bytes, dmr_stream_t stream)
{
    return tet_backward_impl(B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats,
                             inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records, image_buffer, dL_dcolor,
                             dL_ddepth, dL_dverts_color, dL_dfaces_opacity, workspace, workspace_bytes, true, stream);
}

size_t dmr_tet_backward_camera_bytes(int B, int P, int F, int W, int H, int deterministic)
{
    if (B < 0 || P < 0 || F < 0 || W < 0 || H < 0) return 0;
    return tet_cam_bytes(B, P, F, W, H, deterministic != 0);
}

int dmr_tet_backward_camera(int B, int P, int F, int T, int W, int H, int ray_random_seed, const float* background,
                            const float* mv_mats, const float* proj_mats, const float* inv_mv_mats,
                            const float* inv_proj_mats, const float* faces_intense, const void* point_buffer,
                            const void* face_buffer, const void* tet_records, const void* image_buffer,
                            const float* dL_dcolor, const float* dL_ddepth, float* dL_dverts_color,
                            float* dL_dfaces_opacity, int deterministic, float* dL_dmv, float* dL_dproj, void* workspace,
                            size_t workspace_bytes, dmr_stream_t stream)
{
    if (B > 0 && (!dL_dmv || !dL_dproj)) { set_error("null pointer"); return DMR_EINVAL; }
    return tet_backward_impl(B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats,
                             inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records, image_buffer, dL_dcolor,
                             dL_ddepth, dL_dverts_color, dL_dfaces_opacity, workspace, workspace_bytes, deterministic != 0,
                             stream, dL_dmv, dL_dproj);
}

size_t dmr_tet_backward_vertex_bytes(int B, int P, int F, int W, int H, int deterministic, int camera)
{
    if (B < 0 || P < 0 || F < 0 || W < 0 || H < 0) return 0;
    return tet_vert_bytes(B, P, F, W, H, deterministic != 0, camera != 0);
}

int dmr_tet_backward_vertex(int B, int P, int F, int T, int W, int H, int ray_random_seed, const float* background,
                            const float* mv_mats, const float* proj_mats, const float* inv_mv_mats,
                            const float* inv_proj_mats, const float* faces_intense, const void* point_buffer,
                            const void* face_buffer, const void* tet_records, const void* image_buffer,
                            const float* dL_dcolor, const float* dL_ddepth, float* dL_dverts_color,
                            float* dL_dfaces_opacity, int deterministic, float* dL_dmv, float* dL_dproj, float* dL_dverts,
                            void* workspace, size_t workspace_bytes, dmr_stream_t stream)
{
    if ((dL_dmv == nullptr) != (dL_dproj == nullptr)) {
        set_error("dL_dmv and dL_dproj: pass both (camera gradients) or neither");
        return DMR_EINVAL;
    }
    if (B > 0 && !dL_dverts) { set_error("null pointer: dL_dverts"); return DMR_EINVAL; }
    return tet_backward_impl(B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats,
                             inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records, image_buffer, dL_dcolor,
                             dL_ddepth, dL_dverts_color, dL_dfaces_opacity, workspace, workspace_bytes, deterministic != 0,
                             stream, dL_dmv, dL_dproj, dL_dverts);
}

size_t dmr_tet_backward_intensity_bytes(int B, int P, int F, int W, int H, int deterministic, int camera, int vertex)
{
    if (B < 0 || P < 0 || F < 0 || W < 0 || H < 0) return 0;
    return tet_int_bytes(B, P, F, W, H, deterministic != 0, camera != 0, vertex != 0);
}

int dmr_tet_backward_intensity(int B, int P, int F, int T, int W, int H, int ray_random_seed, const float* background,
                               const float* mv_mats, const float* proj_mats, const float* inv_mv_mats,
                               const float* inv_proj_mats, const float* faces_intense, const void* point_buffer,
                               const void* face_buffer, const void* tet_records, const void* image_buffer,
                               const float* dL_dcolor, const float* dL_ddepth, float* dL_dverts_color,
                               float* dL_dfaces_opacity, int deterministic, float* dL_dmv, float* dL_dproj,
                               float* dL_dverts, float* dL_dfaces_intense, void* workspace, size_t workspace_bytes,
                               dmr_stream_t stream)
{
    if ((dL_dmv == nullptr) != (dL_dproj == nullptr)) {
        set_error("dL_dmv and dL_dproj: pass both (camera gradients) or neither");
        return DMR_EINVAL;
    }
    if (B > 0 && !dL_dfaces_intense) { set_error("null pointer: dL_dfaces_intense"); return DMR_EINVAL; }
    return tet_backward_impl(B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats,
                             inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records, image_buffer, dL_dcolor,
                             dL_ddepth, dL_dverts_color, dL_dfaces_opacity, workspace, workspace_bytes, deterministic != 0,
                             stream, dL_dmv, dL_dproj, dL_dverts, dL_dfaces_intense);
}

int dmr_tet_backward_alpha(int B, int P, int F, int T, int W, int H, int ray_random_seed, const float* background,
                           const float* mv_mats, const float* proj_mats, const float* inv_mv_mats,
                           const float* inv_proj_mats, const float* faces_intense, const void* point_buffer,
                           const void* face_buffer, const void* tet_records, const void* image_buffer,
                           const float* dL_dcolor, const float* dL_ddepth, float* dL_dverts_color,
                           float* dL_dfaces_opacity, int deterministic, float* dL_dmv, float* dL_dproj,
                           float* dL_dverts, float* dL_dfaces_intense, const float* dL_dalpha, void* workspace,
                           size_t workspace_bytes, dmr_stream_t stream)
{
    if ((dL_dmv == nullptr) != (dL_dproj == nullptr)) {
        set_error("dL_dmv and dL_dproj: pass both (camera gradients) or neither");
        return DMR_EINVAL;
    }
    if (B > 0 && !dL_dalpha) { set_error("null pointer: dL_dalpha"); return DMR_EINVAL; }
    return tet_backward_impl(B, P, F, T, W, H, ray_random_seed, background, mv_mats, proj_mats, inv_mv_mats,
                             inv_proj_mats, faces_intense, point_buffer, face_buffer, tet_records, image_buffer, dL_dcolor,
                             dL_ddepth, dL_dverts_color, dL_dfaces_opacity, workspace, workspace_bytes, deterministic != 0,
                             stream, dL_dmv, dL_dproj, dL_dverts, dL_dfaces_intense, dL_dalpha);
}

int dmr_tet_alpha(int B, int W, int H, const void* image_buffer, float* out_alpha, dmr_stream_t stream)
{
    if (!tet_sizes_ok(B, 0, 0, 0, W, H)) return DMR_ETOOLARGE;
    if (B == 0) return DMR_OK;
    if (!image_buffer || !out_alpha) { set_error("null pointer"); return DMR_EINVAL; }
    const TetImageLayout IL = TetImageLayout::make(B, W, H);
    return image_alpha(true, B, W, H, at<float>(image_buffer, IL.final_log_T), at<uint8_t>(image_buffer, IL.active),
                       out_alpha, (cudaStream_t)stream);
}

size_t dmr_tet_background_grad_bytes(int B) { return B < 0 ? 0 : image_bg_grad_bytes(B); }

int dmr_tet_background_grad(int B, int W, int H, const void* image_buffer, const float* dL_dcolor, float* dL_dbg,
                            void* workspace, size_t workspace_bytes, dmr_stream_t stream)
{
    if (!tet_sizes_ok(B, 0, 0, 0, W, H)) return DMR_ETOOLARGE;
    if (!dL_dbg) { set_error("null pointer: dL_dbg"); return DMR_EINVAL; }
    if (B > 0 && (!image_buffer || !dL_dcolor)) { set_error("null pointer"); return DMR_EINVAL; }
    const size_t need = image_bg_grad_bytes(B);
    if (!workspace || workspace_bytes < need) {
        set_error("background gradient needs a workspace of %zu bytes (dmr_tet_background_grad_bytes)", need);
        return DMR_EINVAL;
    }
    if (B == 0) { DMR_CUDA(cudaMemsetAsync(dL_dbg, 0, 3 * sizeof(float), (cudaStream_t)stream)); return DMR_OK; }
    const TetImageLayout IL = TetImageLayout::make(B, W, H);
    return image_bg_grad(true, B, W, H, at<float>(image_buffer, IL.final_log_T), at<uint8_t>(image_buffer, IL.active),
                         dL_dcolor, dL_dbg, workspace, (cudaStream_t)stream);
}

int dmr_debug_set_tet_first_split(int split)
{
    g_tet_first_split_override = (split > 0 && split <= 16) ? split : 0;
    return DMR_OK;
}

int dmr_debug_set_tet_trail_cap(int cap)
{
    g_tet_trail_cap_override = cap > 0 ? cap : 0;
    return DMR_OK;
}

}  // extern "C"
